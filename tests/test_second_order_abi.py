"""C-ABI checks of the score net's double backward that need no GPU: the ctypes mirror of DmipMlpGradGrad has the
header's size, and the workspace query is 0 for nets the tcgen05 kernels do not serve (no device needed for either)."""
import ctypes as C
import os

import pytest
import torch

import test_abi


@pytest.fixture(scope="module")
def lib():
    import dmip
    if not os.path.exists(dmip.library_path()):
        dmip.build()
    lib = dmip._lib.lib()
    from dmip import nets
    lib.dmip_mlp_double_backward_workspace_bytes.restype = C.c_size_t
    lib.dmip_mlp_double_backward_workspace_bytes.argtypes = [C.POINTER(nets.DmipMlpGradGrad)]
    return lib


def test_ctypes_mirror_matches_the_header():
    from dmip import nets
    sizes = test_abi._sizeof_from_c(["DmipMlpGradGrad", "DmipMlpGrad"])
    assert C.sizeof(nets.DmipMlpGradGrad) == sizes["DmipMlpGradGrad"]
    assert C.sizeof(nets.DmipMlpGrad) == sizes["DmipMlpGrad"]


def test_entry_points_are_declared_and_exported(lib):
    syms = test_abi.declared_symbols()
    for s in ("dmip_mlp_double_backward", "dmip_mlp_double_backward_workspace_bytes"):
        assert s in syms
        getattr(lib, s)


@pytest.mark.parametrize("hidden,in_dim,out_dim,ok", [((512, 512, 512), 5, 2, True), ((256, 256, 256), 5, 2, False),
                                                     ((512, 512), 5, 2, False), ((512, 512, 512), 65, 2, False),
                                                     ((512, 512, 512), 5, 65, False)])
def test_workspace_is_zero_outside_the_tcgen05_shapes(lib, hidden, in_dim, out_dim, ok):
    from dmip import _lib, nets
    d = nets.DmipMlpGradGrad()
    dims = [in_dim] + list(hidden) + [out_dim]
    d.net.n_layers, d.net.in_dim, d.net.out_dim = len(dims) - 1, in_dim, out_dim
    for i, w in enumerate(dims[1:]):
        d.net.width[i] = w
        d.net.W[i] = d.net.b[i] = 1024      # the query reads shapes only; the pointers just have to be set
    d.n, d.x_dim, d.cond_dim = 100, in_dim - 1, 0
    assert (lib.dmip_mlp_double_backward_workspace_bytes(C.byref(d)) > 0) == ok
    d.n = -1
    assert lib.dmip_mlp_double_backward_workspace_bytes(C.byref(d)) == 0
    assert lib.dmip_mlp_double_backward_workspace_bytes(None) == 0
    assert _lib.MAX_LAYERS >= len(dims) - 1

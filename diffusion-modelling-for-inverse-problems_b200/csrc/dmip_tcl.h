// dmip_tcl.h — interface between the loss orchestration (dmip_loss.cu) and the tcgen05 loss kernels (dmip_tcl.cu).
//
// The tensor-core path of the fused score-training losses (K2 DSM, K3 PINN / Score-FPE / DSM_PDE, the two DPS passes):
// the same forward-mode jets as the fp32 FFMA kernels of dmip_loss.cu, with every GEMM on tcgen05.mma as a bf16x3 split
// product (x = hi + lo, both bf16;  acc += a_hi w_hi + a_hi w_lo + a_lo w_hi, fp32 accumulation in tensor memory:
// relative error ~4e-6 per 512-deep contraction against 2.9e-7 for fp32 and 2.8e-4 for TF32, tools/study_split_gemm.py).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "dmip_common.h"

namespace dmip {

constexpr int kTclRows = 64;        // rows (sample x stream pairs) per tile = N of every tcgen05.mma
constexpr int kTclWin = 32;         // rows per epilogue window (one tcgen05.ld of 32 columns); a sample never straddles one
constexpr int kTclStage = 16384;    // one weight stage: 128 features x 64 k, bf16, K-major, 128-byte swizzle
constexpr int kTclFwdStages = 8 + 64 + 64 + 16;   // hi/lo stages of W0 | W1 | W2 | W3 in consumption order
constexpr int kTclBwdStages = 8 + 64 + 64;        // W3^T | W2^T | W1^T
constexpr int kTclBwdStagesIn = kTclBwdStages + 16;   // ... | W0^T: the input-gradient GEMM of dmip_mlp_backward
constexpr int kTclSmallF = 64;      // feature count of the narrow stash images (layer-0 inputs, output-layer adjoints)

// stream configuration of one pass: which jets ride along with the primal P (dmip_loss.cu header)
struct TclStreams {
  int has_I, has_T, n_tan, has_Q;
  int ns() const { return 1 + has_I + has_T + n_tan + (has_Q ? n_tan * (n_tan + 1) / 2 : 0); }
  int n_adj() const { return 1 + has_I + has_T; }
  int spt_fwd() const { return 2 * (kTclWin / ns()); }       // samples per forward tile
  int spt_bwd() const { return 2 * (kTclWin / n_adj()); }    // samples per backward tile (= per 64-row stash block)
};

// the problem (dmip_common.h: LossProblem, shared with the FFMA kernels), the net, the stream set and the workspace
struct TclDev : LossProblem {
  // ---- net: [in_dim] -> 512 -> 512 -> 512 -> [out_dim]
  const uint8_t* stages_fwd;   // kTclFwdStages x 16 KB
  const uint8_t* stages_bwd;   // kTclBwdStagesIn x 16 KB (the last 16 are consumed only when grad_in is set)
  const float* W[4];           // original fp32 weights (pack kernel input)
  const float* b[4];
  int in_dim, out_dim;
  int k0steps_fwd, k0steps_bwd;   // K = 16 steps of the first GEMM: ceil(in_dim / 16), ceil(out_dim / 16)
  int has_I, has_T, n_tan, has_Q;
  float* abar;                 // [B][n_adj][out_dim] adjoints of the net outputs
  // ---- stashes, laid out as 64-row blocks in the BACKWARD tile geometry (block = one backward tile), each block an
  // MN-major 128B-swizzled bf16 image [row][feature] that k_tcl_wgrad bulk-copies as is:
  //   byte(block, row, f) = block * F * 128 + (f / 64) * 8192 + (row / 8) * 1024 + (row % 8) * 128
  //                         + (((f % 64) / 8) ^ (row % 8)) * 16 + (f % 8) * 2
  uint8_t* in_img[4][2];       // IN_l  hi/lo: inputs of layer l for the adjoint streams (l = 0: F = 64, else F = 512)
  uint8_t* adj_img[4][2];      // ADJ_l hi/lo: adjoints of layer l pre-activations (l = 3: F = 64, else F = 512)
  float* st[3];                // [B][n_adj][512] fp32 state of hidden layer l the backward epilogue needs, one slot per
                               // adjoint stream: P: phi'(z_P) | I: phi'(z_I) | T: phi''(z_P) * zd_T (the T -> P coupling)
  // ---- plain net forward / backward (dmip_mlp_forward_stash / dmip_mlp_backward): post == 4
  float* net_out;              // forward: (B, out_dim) net outputs; inputs are x (B, xdim) | y = cond (B, ydim) | t (B,) as they are
  float* grad_in;              // backward: (B, in_dim) gradient w.r.t. the concatenated inputs, or NULL
  float* grad;                 // flat gradient [W_0, b_0, W_1, b_1, ...] (bias sums are added here by the kernels)
  long long off_b[4];          // float offset of b_l inside grad
  long long n_tiles_fwd, n_tiles_bwd;
};

// which (has_I, has_T, n_tan, has_Q) combinations are compiled in
bool tcl_streams_supported(const TclStreams& s);
size_t tcl_image_bytes();                                   // packed weight images (forward + backward)
int tcl_launch_pack(const TclDev& P, cudaStream_t s);
int tcl_launch_fwd(const TclDev& P, cudaStream_t s);
int tcl_launch_bwd(const TclDev& P, cudaStream_t s);
// dW_l for all four layers: four split-K tcgen05 GEMMs over the stash images, fp32 atomics into P.grad
int tcl_launch_wgrad(const TclDev& P, cudaStream_t s);
// timing builds (-DDMIP_JOBMARKS): CTA 0 of k_tcl_fwd records (clock << 16 | code) entries; no-op otherwise
void tcl_debug_set_timeline(unsigned long long* buf, int cap);

}  // namespace dmip

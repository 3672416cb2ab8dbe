// dmip_pairs.cuh — the pair-tiling bookkeeping shared by the all-pairs metric kernels (k_mmd in dmip_mmd.cu, k_ksd in
// dmip_ksd.cu).  Both walk tiles of an n x n pair square with a persistent grid that takes a static contiguous split of
// the work units, fold per-thread fp64 sums into one workspace slot per (CTA, group) and let a finish kernel add the
// slots of each group in CTA order, so results are bit-identical from run to run on one device.
#pragma once
#include <math.h>

namespace dmip {
namespace pairs {

// row index I and column index J >= I of unit r of the upper triangle (row-major) of a t x t tiling
__device__ __forceinline__ void tri_decode(long long r, long long t, long long& I, long long& J) {
  const double b = 2.0 * static_cast<double>(t) + 1.0;
  long long i = static_cast<long long>((b - sqrt(b * b - 8.0 * static_cast<double>(r))) * 0.5);
  auto off = [t](long long k) { return k * t - k * (k - 1) / 2; };
  if (i < 0) i = 0;
  if (i > t - 1) i = t - 1;
  while (i > 0 && off(i) > r) --i;
  while (i + 1 < t && off(i + 1) <= r) ++i;
  I = i;
  J = i + (r - off(i));
}

// Reduces the per-thread fp64 sums acc[0..NB) over the block in a fixed order into slot[0..NB) and zeroes acc.  Every
// thread of the block calls it; red is shared scratch of THREADS / 32 rows.  When a CTA leaves a group it writes the
// group's slot [cta + group]: the (cta, group) pairs of a contiguous split form a staircase, so cta + group is unique.
template <int NB, int THREADS>
__device__ __forceinline__ void flush_group(double (&acc)[NB], double* slot, double (*red)[NB]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int b = 0; b < NB; ++b) {
    double v = acc[b];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp][b] = v;
    acc[b] = 0.0;
  }
  __syncthreads();
  if (threadIdx.x < NB) {
    double s = 0.0;
    for (int w = 0; w < THREADS / 32; ++w) s += red[w][threadIdx.x];
    slot[threadIdx.x] = s;
  }
  __syncthreads();
}

// Entry b of group g summed over the CTAs of a `grid`-CTA contiguous split of u_total units whose range meets the
// group's units [gb, ge), in CTA order; slots are `stride` doubles wide and CTA c wrote group g to slot c + g.
__device__ __forceinline__ double sum_group_slots(const double* __restrict__ partial, long long u_total, int grid,
                                                  long long g, long long gb, long long ge, int stride, int b) {
  double s = 0.0;
  for (int c = 0; c < grid; ++c) {
    const long long cb = static_cast<long long>(c) * u_total / grid, ce = static_cast<long long>(c + 1) * u_total / grid;
    if (cb < ge && ce > gb) s += partial[(c + g) * stride + b];
  }
  return s;
}

}  // namespace pairs
}  // namespace dmip

// Launch dispatch for one (lmax_filter, lmax_out) group of tensor-product kinds.  Each group is
// its own translation unit (conv_group_*.cu) so that the kinds compile in parallel.
#pragma once
#include "conv_kernels.cuh"

namespace s7b {

// channel pairs per lane in the l1 = 0 backward kernels (1 is 6% faster but splits a (node, l1) role over
// two CTAs, whose per-edge dY/dE/dr sums then need atomics)
constexpr int kBwdL0NV = 2;
// channel pairs per lane in the l1 = 0 forward kernels (1 was measured 4 % slower)
constexpr int kFwdL0NV = 2;

template <int LPN>
static inline dim3 conv_grid(const ConvArgs& a, const ConvRole& role, int nv) {
  const int nodes_per_block = kConvWarpsPerBlock * (32 / LPN);
  return dim3((a.n_dst - a.n_begin + nodes_per_block - 1) / nodes_per_block, role.mul / (2 * LPN * nv));
}

template <class Kind, int NV, int LPN>
static int launch_fwd_one(bool table, const ConvArgs& a, const ConvRole& role, float* out, cudaStream_t st) {
  const dim3 grid = conv_grid<LPN>(a, role, NV);
  if (table) conv_fwd_kernel<Kind, NV, LPN, true><<<grid, 32 * kConvWarpsPerBlock, 0, st>>>(a, role, out);
  else conv_fwd_kernel<Kind, NV, LPN, false><<<grid, 32 * kConvWarpsPerBlock, 0, st>>>(a, role, out);
  return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

template <class Kind, int NV, int LPN, bool TABLE, bool NEED_DX>
static void launch_bwd_split(const dim3& grid, const ConvArgs& a, const ConvRole& role, const float* gout,
                             float* dx, float* dY, float* dEdr, float* dw, cudaStream_t st) {
  const int blk = 32 * kConvWarpsPerBlock;
  // a role split over several CTAs (grid.y > 1) accumulates its per-edge sums atomically
  if (grid.y > 1) conv_bwd_kernel<Kind, NV, LPN, TABLE, NEED_DX, true><<<grid, blk, 0, st>>>(a, role, gout, dx, dY, dEdr, dw);
  else conv_bwd_kernel<Kind, NV, LPN, TABLE, NEED_DX, false><<<grid, blk, 0, st>>>(a, role, gout, dx, dY, dEdr, dw);
}

template <class Kind, int NV, int LPN, bool ALLOW_NODX>
static int launch_bwd_one(bool table, bool need_dx, const ConvArgs& a, const ConvRole& role,
                          const float* gout, float* dx, float* dY, float* dEdr, float* dw, cudaStream_t st) {
  const dim3 grid = conv_grid<LPN>(a, role, NV);
  if (!need_dx && ALLOW_NODX) {
    if (table) launch_bwd_split<Kind, NV, LPN, true, !ALLOW_NODX>(grid, a, role, gout, dx, dY, dEdr, dw, st);
    else launch_bwd_split<Kind, NV, LPN, false, !ALLOW_NODX>(grid, a, role, gout, dx, dY, dEdr, dw, st);
  } else {
    if (table) launch_bwd_split<Kind, NV, LPN, true, true>(grid, a, role, gout, dx, dY, dEdr, dw, st);
    else launch_bwd_split<Kind, NV, LPN, false, true>(grid, a, role, gout, dx, dY, dEdr, dw, st);
  }
  return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

// Lane mapping by multiplicity: 128 | mul -> a warp per node, 2 channel pairs per lane (only
// instantiated where MAXNV == 2); 64 | mul -> a warp per node, 1 pair; else half a warp per node
// (for mul = 32, 29 % faster than one channel per lane on a full warp: 0.099 vs 0.139 ms, 7net-0 l1 = 2).
template <class Kind, int MAXNV>
static int fwd_kind(bool table, const ConvArgs& a, const ConvRole& role, float* out, cudaStream_t st) {
  if (MAXNV >= 2 && role.mul % 128 == 0) return launch_fwd_one<Kind, MAXNV, 32>(table, a, role, out, st);
  if (role.mul % 64 == 0) return launch_fwd_one<Kind, 1, 32>(table, a, role, out, st);
  return launch_fwd_one<Kind, 1, 16>(table, a, role, out, st);
}

// ALLOW_NODX: only the l1 = 0 kinds are ever run without dx (first layer: x depends on species only)
template <class Kind, int MAXNV, bool ALLOW_NODX>
static int bwd_kind(bool table, bool need_dx, const ConvArgs& a, const ConvRole& role,
                    const float* gout, float* dx, float* dY, float* dEdr, float* dw, cudaStream_t st) {
  if (MAXNV >= 2 && role.mul % 128 == 0)
    return launch_bwd_one<Kind, MAXNV, 32, ALLOW_NODX>(table, need_dx, a, role, gout, dx, dY, dEdr, dw, st);
  if (role.mul % 64 == 0)
    return launch_bwd_one<Kind, 1, 32, ALLOW_NODX>(table, need_dx, a, role, gout, dx, dY, dEdr, dw, st);
  return launch_bwd_one<Kind, 1, 16, ALLOW_NODX>(table, need_dx, a, role, gout, dx, dY, dEdr, dw, st);
}

}  // namespace s7b

// Defines  launch_conv_fwd_LF_LO / launch_conv_bwd_LF_LO  for l1 = 0..LF.
#define S7B_DEFINE_CONV_GROUP(LF, LO)                                                              \
  namespace s7b {                                                                                  \
  int launch_conv_fwd_##LF##_##LO(int l1, bool table, const ConvArgs& a, const ConvRole& role,     \
                                  float* out, cudaStream_t st) {                                   \
    switch (l1) {                                                                                  \
      case 0: return fwd_kind<TPKind<0, LF, LO>, kFwdL0NV>(table, a, role, out, st);                      \
      case 1: return fwd_kind<TPKind<1, LF, LO>, 1>(table, a, role, out, st);                      \
      case 2: return fwd_kind<TPKind<2, LF, LO>, 1>(table, a, role, out, st);                      \
      case 3: return fwd_kind<TPKind<(LF >= 3 ? 3 : 2), LF, LO>, 1>(table, a, role, out, st);      \
    }                                                                                              \
    return 1;                                                                                      \
  }                                                                                                \
  int launch_conv_bwd_##LF##_##LO(int l1, bool table, bool need_dx, const ConvArgs& a,             \
                                  const ConvRole& role, const float* gout, float* dx, float* dY,   \
                                  float* dEdr, float* dw, cudaStream_t st) {                       \
    switch (l1) {                                                                                  \
      case 0: return bwd_kind<TPKind<0, LF, LO>, kBwdL0NV, true>(table, need_dx, a, role, gout, dx, dY, dEdr, dw, st);  \
      case 1: return bwd_kind<TPKind<1, LF, LO>, 1, false>(table, need_dx, a, role, gout, dx, dY, dEdr, dw, st); \
      case 2: return bwd_kind<TPKind<2, LF, LO>, 1, false>(table, need_dx, a, role, gout, dx, dY, dEdr, dw, st); \
      case 3: return bwd_kind<TPKind<(LF >= 3 ? 3 : 2), LF, LO>, 1, false>(table, need_dx, a, role, gout, dx, dY, dEdr, dw, st); \
    }                                                                                              \
    return 1;                                                                                      \
  }                                                                                                \
  }

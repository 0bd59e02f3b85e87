// Fused neighbour-gather -> Clebsch-Gordan tensor product -> scatter-to-centre kernels.
//
// Replaces, for one interaction layer, the reference's
//   x[edge_src] gather                     sevenn/nn/convolution.py:131
//   e3nn TensorProduct ('uvu', per-edge w) sevenn/nn/convolution.py:84-100,131
//   message_gather scatter_reduce_         sevenn/nn/convolution.py:17-26,133
// and their autograd backward (sevenn/nn/force_output.py:177-182) with one forward and one
// backward kernel per l1 "kind" (see csrc/gen_kernels.py).
//
// Mapping: a group of LPN lanes (32 = a warp, or 16 = half a warp for 32-channel irreps) owns one
// destination atom n and one l1 block.  Every lane carries NV channel PAIRS (channels 2*lane,
// 2*lane+1, then +2*LPN): all per-channel arithmetic is issued as Blackwell packed-FP32
// instructions (FFMA2/FMUL2, csrc/vec_ops.cuh), every global access of a group is one contiguous
// 8-byte-per-lane segment of the component-major ("cm") layout, and the node accumulators of all
// paths stay in registers over the whole CSR row -- no atomics in the forward.
// The radial weights w_p,u(r) come either from a cubic-Hermite table indexed by the edge length
// (TABLE: L2-resident, per (knot, channel pair) {a0e,a0o,a1e,a1o} fp32 + {a2e,a2o,a3e,a3o} fp16 = 24 B)
// or from a stored [E, W]
// array (!TABLE: the reference's plug-in boundary, where the radial MLP stays outside).
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"
#include "generated/tp_kinds.cuh"

namespace s7b {

constexpr int kConvWarpsPerBlock = 4;
// Register budget, as the min-resident-CTAs argument of __launch_bounds__ (128-thread CTAs: 4 -> 128
// registers, 3 -> 168, 1 -> 255).  Measured on B200 (7net-0, 12k atoms, A/B inside one box):
//  * forward: an explicit 1 lets ptxas keep more gathers in flight for the l1 = 0 kernels (96 -> 128
//    registers, -22 % time); the l1 >= 1 kernels do not change;
//  * backward: l1 = 0 is fastest at 3 (-6 %), l1 = 1 at 4 (128 registers; 168 or 220 are 3-4 % slower),
//    l1 >= 2 at 3 (what ptxas picks by itself).  The lmax = 3 kinds need > 168 registers (they spill
//    otherwise) and are left at 2.
#define S7B_FWD_BOUNDS __launch_bounds__(32 * kConvWarpsPerBlock, 1)
#define S7B_BWD_BOUNDS __launch_bounds__(32 * kConvWarpsPerBlock, (Kind::NY != 9) ? 2 : ((Kind::D1 == 3) ? 4 : 3))

// The 16-byte edge record {neighbour, table interval, frac} heads the per-edge dependency chain
// (record -> gather address / table address -> loads -> math).  Loading it per edge costs one
// dependent L2 round trip per edge; instead lane i of a group loads the record of edge e0 + i of the
// row (one coalesced 16*LPN-byte request per LPN edges, i.e. about once per row) and every iteration
// takes its record by shuffle.  Prefetching record + harmonics into registers was measured slower
// (register pressure); this costs three registers.
template <int LPN>
struct EdgeRecs {
  int cx, cy, cz;
  __device__ __forceinline__ void fill(const ConvArgs& a, int e0, int len, int it, int sl) {
    const int ei = it + sl;
    int4 r = make_int4(0, 0, 0, 0);
    if (ei < len) r = __ldg(a.rec + e0 + ei);
    cx = r.x; cy = r.y; cz = r.z;
  }
  __device__ __forceinline__ int4 get(int it) const {
    const int l = it % LPN;
    return make_int4(__shfl_sync(0xffffffffu, cx, l, LPN), __shfl_sync(0xffffffffu, cy, l, LPN),
                     __shfl_sync(0xffffffffu, cz, l, LPN), 0);
  }
};

// Sum M values (M = 8 or 16) over the LPN lanes of a group with ~M-1+log2(LPN/M) shuffles instead
// of M*log2(LPN).  On return v[0] of group-lane sl holds the total of value (sl / (LPN/M)) % M.
template <int M, int LPN>
__device__ __forceinline__ void group_reduce_multi(float (&v)[M], int sl) {
  static_assert((M == 8 || M == 16) && (LPN == 16 || LPN == 32) && M <= LPN, "unsupported reduction shape");
  int off = LPN / 2;
#pragma unroll
  for (int m = M / 2; m >= 1; m >>= 1, off >>= 1) {
    const bool up = (sl & off) != 0;
#pragma unroll
    for (int j = 0; j < m; ++j) {
      const float send = up ? v[j] : v[j + m];
      const float keep = up ? v[j + m] : v[j];
      v[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
#pragma unroll
  for (; off >= 1; off >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], off);
}

template <int LPN>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int off = LPN / 2; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

template <class Kind>
__device__ __forceinline__ void load_Y(const float* __restrict__ Yrow, float (&Y)[Kind::NY]) {
  Y[0] = 1.0f;
  constexpr int NQ = (Kind::NY - 1 + 3) / 4;
  const float4* p = reinterpret_cast<const float4*>(Yrow);
#pragma unroll
  for (int q = 0; q < NQ; ++q) {
    const float4 v = __ldg(p + q);
    if (4 * q + 1 < Kind::NY) Y[4 * q + 1] = v.x;
    if (4 * q + 2 < Kind::NY) Y[4 * q + 2] = v.y;
    if (4 * q + 3 < Kind::NY) Y[4 * q + 3] = v.z;
    if (4 * q + 4 < Kind::NY) Y[4 * q + 4] = v.w;
  }
}

__device__ __forceinline__ float2 ldg2(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }

// cubic coefficients of the channel pair starting at (even) column c of table row tk
__device__ __forceinline__ void table_coef(const ConvArgs& a, int tk, int c, V2& a0, V2& a1, V2& a2, V2& a3) {
  const size_t ti = (size_t)tk * (a.w_numel >> 1) + (c >> 1);
  const float4 c01 = __ldg(a.table + ti);
  const uint2 c23 = __ldg(a.table23 + ti);
  a0 = make_float2(c01.x, c01.y);
  a1 = make_float2(c01.z, c01.w);
  a2 = __half22float2(*reinterpret_cast<const __half2*>(&c23.x));
  a3 = __half22float2(*reinterpret_cast<const __half2*>(&c23.y));
}

// Which node / channel pair this lane works on.
template <int NV, int LPN>
struct LaneMap {
  int n, sl, uc0, e0, len, nmax;
  bool node_ok;
  __device__ __forceinline__ LaneMap(const ConvArgs& a) {
    constexpr int GPW = 32 / LPN;
    const int lane = threadIdx.x & 31;
    sl = lane % LPN;
    n = a.n_begin + (blockIdx.x * kConvWarpsPerBlock + (threadIdx.x >> 5)) * GPW + lane / LPN;
    node_ok = n < a.n_dst;
    uc0 = blockIdx.y * (2 * LPN * NV) + 2 * sl;
    e0 = 0;
    len = 0;
    if (node_ok) {
      e0 = __ldg(a.rowptr + n);
      len = __ldg(a.rowptr + n + 1) - e0;
    }
    nmax = len;
    if (GPW > 1) nmax = max(len, __shfl_xor_sync(0xffffffffu, len, 16));
  }
};

// ------------------------------------------------------------------------------------------
// forward:  out[n, path block] = sum_{e in row n} w_e * CG(x[src_e], Y_e)
// grid = (ceil(n_dst / (kConvWarpsPerBlock * 32/LPN)), mul / (2*LPN*NV)), block = 32*kConvWarpsPerBlock
// ------------------------------------------------------------------------------------------
template <class Kind, int NV, int LPN, bool TABLE>
__global__ void S7B_FWD_BOUNDS
conv_fwd_kernel(const ConvArgs a, const ConvRole role, float* __restrict__ out) {
  const LaneMap<NV, LPN> m(a);
  if (m.nmax == 0 && !m.node_ok) return;      // whole warp beyond the last node (uniform)

  V2 acc[NV][Kind::NACC];
#pragma unroll
  for (int c = 0; c < NV; ++c)
#pragma unroll
    for (int q = 0; q < Kind::NACC; ++q) acc[c][q] = splat2(0.0f);

  EdgeRecs<LPN> recs;
  for (int it = 0; it < m.nmax; ++it) {
    const bool valid = (LPN == 32) || (it < m.len);
    const int e = valid ? m.e0 + it : 0;
    if (it % LPN == 0) recs.fill(a, m.e0, m.len, it, m.sl);
    const int4 rec = recs.get(it);
    float Y[Kind::NY];
    load_Y<Kind>(a.Y + (size_t)e * a.ny_stride, Y);
    const float* __restrict__ xrow = a.x + (size_t)rec.x * a.dim_x + role.x_off;
    const float tt = __int_as_float(rec.z);
#pragma unroll
    for (int c = 0; c < NV; ++c) {
      const int u = m.uc0 + 2 * LPN * c;
      V2 x[Kind::D1], w[Kind::NPATH];
#pragma unroll
      for (int i = 0; i < Kind::D1; ++i) x[i] = ldg2(xrow + i * role.mul + u);
#pragma unroll
      for (int p = 0; p < Kind::NPATH; ++p) {
        if (TABLE) {
          V2 a0, a1, a2, a3;
          table_coef(a, rec.y, role.w_off[p] + u, a0, a1, a2, a3);
          w[p] = fma_(tt, fma_(tt, fma_(tt, a3, a2), a1), a0);
        } else {
          w[p] = ldg2(a.w + (size_t)e * a.w_numel + role.w_off[p] + u);
        }
        if (LPN != 32 && !valid) w[p] = splat2(0.0f);
      }
      Kind::fwd(x, Y, w, acc[c]);
    }
  }

  // row maxima of the mid features for the tensor-core self_interaction_2 (fixed-point row scaling): one
  // group reduction and one atomicMax per (l3, k) row this role contributes to -- saves a pass over the mid tensor
  if (a.row_max != nullptr) {
#pragma unroll
    for (int l3 = 0; l3 < kMaxL; ++l3) {
      bool present = false;
#pragma unroll
      for (int p = 0; p < Kind::NPATH; ++p) present = present || (Kind::path_l3(p) == l3);
      if (!present) continue;
#pragma unroll
      for (int k = 0; k < 2 * l3 + 1; ++k) {
        float mx = 0.0f;
#pragma unroll
        for (int c = 0; c < NV; ++c)
#pragma unroll
          for (int p = 0; p < Kind::NPATH; ++p)
            if (Kind::path_l3(p) == l3) {
              const V2 v = acc[c][Kind::acc_off(p) + k];
              mx = fmaxf(mx, fmaxf(fabsf(v.x), fabsf(v.y)));
            }
#pragma unroll
        for (int off = LPN / 2; off >= 1; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
        if (m.node_ok && m.sl == 0) atomicMax(a.row_max + (size_t)m.n * a.rows_per_node + l3 * l3 + k, __float_as_uint(mx));
      }
    }
  }
  if (!m.node_ok) return;
  float* __restrict__ orow = out + (size_t)m.n * a.dim_mid;
#pragma unroll
  for (int c = 0; c < NV; ++c) {
    const int u = m.uc0 + 2 * LPN * c;
#pragma unroll
    for (int p = 0; p < Kind::NPATH; ++p) {
#pragma unroll
      for (int k = 0; k < 2 * Kind::path_l3(p) + 1; ++k)
        *reinterpret_cast<float2*>(orow + role.out_off[p] + k * role.out_stride[p] + u) = acc[c][Kind::acc_off(p) + k];
    }
  }
}

// ------------------------------------------------------------------------------------------
// backward (centre-major): given ga = dE/d out[n, :], per edge of row n
//   TABLE : dEdr_acc[e] += sum_{p,u} (dE/dw_{p,u}) * w'_{p,u}(r_e)         (radial chain rule)
//   !TABLE: dw[e, :]     = dE/dw                                          (plug-in boundary)
//   dY_acc[e, 1..]      += sum_u dE/dY                                    (group reduction)
//   dx[src_e, :]        += dE/dx                                          (RED.ADD.F32x2, NEED_DX)
// dY_acc / dEdr_acc / dw rows are owned by exactly one group of one launch: plain read-modify-write.
// ------------------------------------------------------------------------------------------
template <class Kind, int NV, int LPN, bool TABLE, bool NEED_DX, bool SPLIT>
__global__ void S7B_BWD_BOUNDS
conv_bwd_kernel(const ConvArgs a, const ConvRole role, const float* __restrict__ gout,
                float* __restrict__ dx, float* __restrict__ dY_acc, float* __restrict__ dEdr_acc,
                float* __restrict__ dw) {
  const LaneMap<NV, LPN> m(a);
  if (m.nmax == 0) return;                    // uniform: no edges in any row of this warp

  V2 ga[NV][Kind::NACC];
  {
    const float* __restrict__ grow = gout + (size_t)(m.node_ok ? m.n : 0) * a.dim_mid;
#pragma unroll
    for (int c = 0; c < NV; ++c) {
      const int u = m.uc0 + 2 * LPN * c;
#pragma unroll
      for (int p = 0; p < Kind::NPATH; ++p)
#pragma unroll
        for (int k = 0; k < 2 * Kind::path_l3(p) + 1; ++k)
          ga[c][Kind::acc_off(p) + k] = ldg2(grow + role.out_off[p] + k * role.out_stride[p] + u);
    }
  }

  constexpr int NR = (Kind::NY <= 9) ? 8 : 16;   // values reduced with the transposing butterfly
  constexpr bool RIDE = TABLE && (Kind::NY - 1 < NR);     // a free slot of the butterfly carries dE/dr
  constexpr int PER = LPN / NR;
  const int idx = (m.sl / PER) % NR;                      // which reduced value ends up in this lane
  const bool is_dY = idx + 1 < Kind::NY;
  const bool writer = (m.sl % PER) == 0 && (is_dY || (RIDE && idx == NR - 1));
  EdgeRecs<LPN> recs;
  for (int it = 0; it < m.nmax; ++it) {
    const bool valid = (LPN == 32) || (it < m.len);
    const int e = valid ? m.e0 + it : 0;
    if (it % LPN == 0) recs.fill(a, m.e0, m.len, it, m.sl);
    const int4 rec = recs.get(it);
    float Y[Kind::NY];
    load_Y<Kind>(a.Y + (size_t)e * a.ny_stride, Y);
    const float* __restrict__ xrow = a.x + (size_t)rec.x * a.dim_x + role.x_off;
    const float tt = __int_as_float(rec.z);
    V2 dY[Kind::NY];
#pragma unroll
    for (int j = 0; j < Kind::NY; ++j) dY[j] = splat2(0.0f);
    V2 dEdr2 = splat2(0.0f);
#pragma unroll
    for (int c = 0; c < NV; ++c) {
      const int u = m.uc0 + 2 * LPN * c;
      V2 x[Kind::D1], w[Kind::NPATH], wd[Kind::NPATH], dwv[Kind::NPATH], dxv[Kind::D1];
#pragma unroll
      for (int i = 0; i < Kind::D1; ++i) x[i] = ldg2(xrow + i * role.mul + u);
#pragma unroll
      for (int p = 0; p < Kind::NPATH; ++p) {
        if (TABLE) {
          const size_t ti = (size_t)rec.y * (a.w_numel >> 1) + ((role.w_off[p] + u) >> 1);
          const float4 c01 = __ldg(a.table + ti);
          const uint2 c23 = __ldg(a.table23 + ti);
          const V2 a0 = make_float2(c01.x, c01.y), a1 = make_float2(c01.z, c01.w);
          const V2 a2 = __half22float2(*reinterpret_cast<const __half2*>(&c23.x));
          const V2 a3 = __half22float2(*reinterpret_cast<const __half2*>(&c23.y));
          w[p] = fma_(tt, fma_(tt, fma_(tt, a3, a2), a1), a0);
          wd[p] = mul_(fma_(tt, fma_(3.0f * tt, a3, mul_(a2, 2.0f)), a1), a.inv_h);
        } else {
          w[p] = ldg2(a.w + (size_t)e * a.w_numel + role.w_off[p] + u);
        }
      }
      Kind::bwd(x, Y, w, ga[c], dwv, dxv, dY);
      if (valid) {
#pragma unroll
        for (int p = 0; p < Kind::NPATH; ++p) {
          if (TABLE) dEdr2 = fma_(dwv[p], wd[p], dEdr2);
          else *reinterpret_cast<float2*>(dw + (size_t)e * a.w_numel + role.w_off[p] + u) = dwv[p];
        }
        if (NEED_DX) {
          float* __restrict__ dxrow = dx + (size_t)rec.x * a.dim_x + role.x_off;
#pragma unroll
          for (int i = 0; i < Kind::D1; ++i)
            atomicAdd(reinterpret_cast<float2*>(dxrow + i * role.mul + u), dxv[i]);
        }
      }
    }
    // cross-channel reduction of dE/dY (NY-1 values) and dE/dr (1 value) over the group
    const float dEdr = dEdr2.x + dEdr2.y;
    float red[NR];
#pragma unroll
    for (int j = 0; j < NR; ++j) red[j] = (j + 1 < Kind::NY) ? dY[j + 1].x + dY[j + 1].y : 0.0f;
    if (RIDE) red[NR - 1] = dEdr;
    group_reduce_multi<NR, LPN>(red, m.sl);
    // a (node, l1) role normally belongs to one group -> plain read-modify-write (deterministic);
    // SPLIT (launched with gridDim.y > 1: the role's channels are spread over several CTAs) adds atomically
    if (valid && writer) {
      float* dst = is_dY ? dY_acc + (size_t)e * a.ny_stride + idx : dEdr_acc + e;
      if (SPLIT) atomicAdd(dst, red[0]);
      else *dst += red[0];      // (requesting the old value at the top of the iteration was measured 1 % slower)
    }
    if (TABLE && !RIDE) {
      const float s = group_sum<LPN>(dEdr);
      if (valid && m.sl == 0) {
        if (SPLIT) atomicAdd(dEdr_acc + e, s);
        else dEdr_acc[e] += s;
      }
    }
  }
}

}  // namespace s7b

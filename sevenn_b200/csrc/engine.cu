// Host side of the C ABI (include/sevenn_b200.h): model description -> per-layer launch plans,
// device buffers, and the stage sequence of one energy/force evaluation.
//
// The stage sequence restates, with hand-written kernels and a hand-written backward, what the
// reference executes per MD step through torch modules and autograd:
//   AtomGraphSequential.forward          sevenn/nn/sequential.py:157-183
//   NequIP_interaction_block order       sevenn/nn/interaction_blocks.py:41-76
//   ForceStressOutputFromEdge            sevenn/nn/force_output.py:171-230
//   segment-wise forward / backward      sevenn/pair_e3gnn/pair_e3gnn_parallel.cpp:345-441
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <string>
#include <vector>

#include "../../include/sevenn_b200.h"
#include "common.cuh"
#include "conv_kernels.cuh"
#include "edge_kernels.cuh"
#include "neighbor.cuh"
#include "node_kernels.cuh"
#include "tc_gemm.cuh"

namespace s7b {

static thread_local std::string g_error;
static int64_t g_launches = 0;
extern int64_t g_conv_launches;

void set_error(const char* file, int line, const char* msg) {
  char buf[512];
  snprintf(buf, sizeof(buf), "%s:%d: %s", file, line, msg);
  g_error = buf;
}
static int fail(const std::string& m) {
  g_error = m;
  return 1;
}

#define S7B_LAUNCH_CHECK()                          \
  do {                                              \
    ++g_launches;                                   \
    S7B_CUDA_CHECK(cudaGetLastError());             \
  } while (0)

// ---- conv launch dispatch (defined in conv_dispatch_*.cu) ---------------------------------
int launch_conv_fwd(int l1, int lf, int lo, bool table, const ConvArgs& a, const ConvRole& role,
                    float* out, cudaStream_t st);
int launch_conv_bwd(int l1, int lf, int lo, bool table, bool need_dx, const ConvArgs& a,
                    const ConvRole& role, const float* gout, float* dx, float* dY_acc,
                    float* dEdr_acc, float* dw, cudaStream_t st);

static int64_t g_alloc_gen = 0;   // bumped by every (re)allocation: captured CUDA graphs hold raw pointers

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  int ensure(size_t need) {
    if (need <= bytes) return 0;
    ++g_alloc_gen;
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
    size_t want = need + need / 8 + 256;
    if (cudaMalloc(&p, want) != cudaSuccess) {
      cudaGetLastError();
      return 1;
    }
    bytes = want;
    return 0;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
  }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct PathCfg { int l1, l2, l3, mul, w_off, k_off; };

// Optional per-kernel timing with CUDA events on the launching stream (bench.py roofline leg).
struct Profiler {
  bool enabled = false;
  struct Rec { std::string label; cudaEvent_t a, b; };
  std::vector<Rec> recs;
  std::vector<cudaEvent_t> pool;
  std::map<std::string, std::pair<double, int64_t>> totals;   // label -> (ms, calls)
  cudaEvent_t get() {
    if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
  }
  void collect() {
    for (auto& r : recs) {
      cudaEventSynchronize(r.b);
      float ms = 0.f;
      cudaEventElapsedTime(&ms, r.a, r.b);
      auto& t = totals[r.label];
      t.first += ms;
      t.second += 1;
      pool.push_back(r.a);
      pool.push_back(r.b);
    }
    recs.clear();
  }
  void clear() { collect(); totals.clear(); }
};

struct ProfScope {
  Profiler* p;
  cudaStream_t st;
  cudaEvent_t b;
  ProfScope(Profiler& prof, cudaStream_t s, const char* what, int t = -1, int l = -1) : p(nullptr), st(s) {
    if (!prof.enabled) return;
    p = &prof;
    char buf[64];
    if (t >= 0 && l >= 0) snprintf(buf, sizeof(buf), "%s.t%d.l%d", what, t, l);
    else if (t >= 0) snprintf(buf, sizeof(buf), "%s.t%d", what, t);
    else snprintf(buf, sizeof(buf), "%s", what);
    cudaEvent_t a = prof.get();
    b = prof.get();
    cudaEventRecord(a, st);
    prof.recs.push_back({buf, a, b});
  }
  ~ProfScope() { if (p) cudaEventRecord(b, st); }
};

struct LayerCfg {
  int n_lx = 0, n_lg = 0;             // number of l's in x / gate-out irreps
  int x_muls[kMaxL] = {0}, out_muls[kMaxL] = {0}, g_muls[kMaxL] = {0};
  int x_off[kMaxL] = {0}, g_off[kMaxL] = {0}, h_off[kMaxL] = {0};
  int dim_x = 0, dim_g = 0, dim_h = 0, dim_mid = 0, W = 0;
  int mid_K[kMaxL] = {0}, mid_off[kMaxL] = {0};
  int lmax_out = 0;
  std::vector<PathCfg> paths;
  ConvRole roles[kMaxL];
  GateDesc gate;
  std::map<std::string, DevBuf> params;
  std::map<std::string, struct TcWeights*> tcw;   // tensor-core form of si1/si1T/sc/scT/si2/si2T (engine.cu: TcWeights)
};

// Row exponents of a GEMM input (tc_gemm.cuh): E[n, row_base[l] + i]
struct RowExp {
  DevBuf buf;
  int rows_per_node = 0;
  bool bits = false;      // raw |a|-maximum bits (filled by the producer kernel) instead of exponents
};

}  // namespace s7b

using namespace s7b;

struct S7bEngine {
  S7bModelDesc desc;
  std::vector<LayerCfg> layers;
  std::map<std::string, DevBuf> params;   // global parameters
  RadialDesc radial;
  bool radial_ready = false;
  int ny_stride = 8;
  int max_lx = 0;                         // largest n_lx of any layer = number of per-l1 parts of dY_acc / dEdr_acc
  // graph
  int n_nodes = 0, n_local = 0, n_interior = 0;
  int64_t n_edges = 0;
  const int* d_species = nullptr;
  const int* d_rowptr = nullptr;
  const int* d_src = nullptr;
  const float* d_edge_vec = nullptr;
  // per-step buffers
  DevBuf rec, Y, rlen, emb, dY_acc, dEdr_acc, demb_acc, fedge;
  std::vector<DevBuf> x, g, wbuf, z1, z2, h1, h2;   // per layer (wbuf.. exact-MLP mode only)
  DevBuf mid, h, dh, dg, dx, dwbuf, tmpA, tmpB;
  RowExp re_mid, re_h, re_dg, re_dx;      // row exponents of the tensor-core GEMM inputs
  DevBuf energy, atomic_energy, forces, virial, atomic_virial;
  bool want_atomic_virial = false;
  // host staging for compute_host
  DevBuf hs_species, hs_rowptr, hs_src, hs_vec, hs_centre, hs_flag;
  // device neighbour list (positions -> CSR)
  DevBuf nl_pos, nl_wrapped, nl_key, nl_key_sorted, nl_idx, nl_idx_sorted, nl_bin_start, nl_count, nl_tmp, nl_centres;
  int nl_n_centres = 0;
  int64_t nl_n_edges = 0;
  Profiler prof;
  // side streams: the per-l1 convolution kernels of one layer are independent (disjoint outputs) and
  // stress different units (l1 = 0: L1/L2 latency, l1 >= 1: FP32 pipe), so they are co-scheduled
  cudaStream_t side[kMaxL] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev_fork = nullptr, ev_join[kMaxL] = {nullptr, nullptr, nullptr, nullptr};
  bool concurrent = true;
  // Per-edge buffers are strided / gridded by a capacity E_cap >= n_edges and the edge kernels read the
  // live edge count from d_nE, so that one captured CUDA graph of the whole step can be replayed while
  // the neighbour count drifts between MD steps.
  int64_t E_cap = 0;
  DevBuf d_nE;
  cudaGraphExec_t gexec = nullptr;
  cudaStream_t gstream = nullptr;
  cudaEvent_t g_in = nullptr, g_out = nullptr;
  std::vector<int64_t> g_key;
  int64_t g_launches_per_replay = 0;
  int64_t g_captures = 0, g_replays = 0;
  // one graph per (stage, layer) for callers that drive the stages themselves (multi-GPU runner, LAMMPS front-ends)
  struct StageGraph {
    cudaGraphExec_t exec = nullptr;
    std::vector<int64_t> key;
    int64_t launches = 0, replays_since_capture = 0;
    int thrash = 0;                       // re-captures that were replayed fewer than twice
  };
  std::map<int, StageGraph> stage_graphs;
  bool capturing = false;
  int64_t sg_captures = 0, sg_replays = 0;
};

struct S7bConvPlan {
  LayerCfg cfg;
  int lmax_filter = 0;
  int ny_stride = 8;
};

namespace s7b {

static int irreps_dim(const int* muls, int n_l) {
  int d = 0;
  for (int l = 0; l < n_l; ++l) d += (2 * l + 1) * muls[l];
  return d;
}

// Restates build_layer() of sevenn_b200/spec.py (reference convolution.py:61-82 path order).
static int build_layer_cfg(LayerCfg& L, const int* x_muls, int n_lx, const int* out_muls, int n_lo,
                           int lmax_filter) {
  L.n_lx = n_lx;
  L.n_lg = n_lo;
  L.lmax_out = n_lo - 1;
  int off = 0;
  for (int l = 0; l < n_lx; ++l) {
    if (x_muls[l] % 32 != 0 || x_muls[l] <= 0) return fail("multiplicities must be positive multiples of 32");
    L.x_muls[l] = x_muls[l];
    L.x_off[l] = off;
    off += (2 * l + 1) * x_muls[l];
  }
  L.dim_x = off;
  int n_gates = 0;
  for (int l = 1; l < n_lo; ++l) n_gates += out_muls[l];
  for (int l = 0; l < n_lo; ++l) {
    if (out_muls[l] % 32 != 0 || out_muls[l] <= 0) return fail("multiplicities must be positive multiples of 32");
    L.out_muls[l] = out_muls[l];
    L.g_muls[l] = out_muls[l] + (l == 0 ? n_gates : 0);
  }
  L.dim_g = irreps_dim(L.g_muls, n_lo);
  L.dim_h = irreps_dim(L.out_muls, n_lo);
  off = 0;
  int hoff = 0;
  for (int l = 0; l < n_lo; ++l) {
    L.g_off[l] = off;
    off += (2 * l + 1) * L.g_muls[l];
    L.h_off[l] = hoff;
    hoff += (2 * l + 1) * L.out_muls[l];
  }
  // paths: creation order (l1, l2, l3 ascending), then stable sort by l3
  struct C { int l1, l2, l3, mul; };
  std::vector<C> created;
  for (int l1 = 0; l1 < n_lx; ++l1)
    for (int l2 = 0; l2 <= lmax_filter; ++l2)
      for (int l3 = abs(l1 - l2); l3 <= l1 + l2; ++l3)
        if (l3 <= L.lmax_out) created.push_back({l1, l2, l3, x_muls[l1]});
  std::vector<int> order;
  for (int l3 = 0; l3 <= L.lmax_out; ++l3)
    for (size_t c = 0; c < created.size(); ++c)
      if (created[c].l3 == l3) order.push_back((int)c);
  int w_off = 0;
  int k_run[kMaxL] = {0, 0, 0, 0};
  L.paths.clear();
  for (int c : order) {
    const C& q = created[c];
    L.paths.push_back({q.l1, q.l2, q.l3, q.mul, w_off, k_run[q.l3]});
    k_run[q.l3] += q.mul;
    w_off += q.mul;
  }
  L.W = w_off;
  off = 0;
  for (int l = 0; l <= L.lmax_out; ++l) {
    L.mid_K[l] = k_run[l];
    L.mid_off[l] = off;
    off += (2 * l + 1) * k_run[l];
  }
  L.dim_mid = off;
  // conv roles: per l1 the paths in slot order
  for (int l1 = 0; l1 < n_lx; ++l1) {
    ConvRole& r = L.roles[l1];
    memset(&r, 0, sizeof(r));
    r.x_off = L.x_off[l1];
    r.mul = x_muls[l1];
    int p = 0;
    for (const PathCfg& q : L.paths) {
      if (q.l1 != l1) continue;
      if (p >= kMaxPaths) return fail("too many paths for one l1");
      r.w_off[p] = q.w_off;
      r.out_off[p] = L.mid_off[q.l3] + q.k_off;
      r.out_stride[p] = L.mid_K[q.l3];
      ++p;
    }
  }
  // gate
  GateDesc& gd = L.gate;
  memset(&gd, 0, sizeof(gd));
  gd.n_scalars = out_muls[0];
  gd.lmax = n_lo - 1;
  gd.dim_g = L.dim_g;
  gd.dim_h = L.dim_h;
  int goff = out_muls[0];
  for (int l = 0; l < kMaxL; ++l) {
    gd.mul[l] = l < n_lo ? out_muls[l] : 0;
    gd.g_off[l] = l < n_lo ? L.g_off[l] : L.dim_g;
    gd.h_off[l] = l < n_lo ? L.h_off[l] : L.dim_h;
    gd.gate_off[l] = L.g_muls[0];
  }
  for (int l = 1; l < n_lo; ++l) {
    gd.gate_off[l] = goff;
    goff += out_muls[l];
  }
  return 0;
}

static int g_opt_atomic_virial = 0;   // engines created afterwards also produce the per-atom virial
static int g_opt_concurrent = 1;   // co-schedule the per-l1 convolution kernels of a layer on side streams
static int g_opt_gate_bwd_rows = 0; // gate backward also leaves the row maxima of dg (saves one row-exponent pass per layer; opt-in)
static int g_opt_stage_graphs = 0;  // s7b_engine_run_stage replays one captured graph per (stage, layer)
static int g_opt_cuda_graph = 1;   // s7b_engine_compute replays a captured CUDA graph of the step (table mode)
static int g_opt_tc_gemm = 1;   // 1 (default): node linears on tcgen05 (error-free bf16x3 slices, tc_gemm.cuh); 0: FP32 SIMT
static long long* g_tc_trace = nullptr;   // device buffer [1 + 4 * cap] when s7b_tc_trace_enable was called (debug)
static int g_tc_trace_cap = 0;
static int g_opt_tc_swizzle = 1;   // 128B-swizzled TMA tile for the raw A chunk (0: plain rows; A/B switch)

__global__ void set_i64_kernel(int64_t* p, int64_t v) { *p = v; }

// CSR over centres from a centre-sorted edge list, with validation (thread e handles the row starts
// between centre[e-1] and centre[e]; thread n_edges closes the tail).  flag: 1 = not sorted / centre out
// of range, 2 = neighbour out of range.
__global__ void csr_from_sorted_kernel(const int* __restrict__ centre, const int* __restrict__ neighbour,
                                       int64_t n_edges, int n_nodes, int* __restrict__ rowptr,
                                       int* __restrict__ flag) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e > n_edges) return;
  const int prev = (e == 0) ? -1 : centre[e - 1];
  const int cur = (e == n_edges) ? n_nodes : centre[e];
  if (e < n_edges) {
    if (cur < prev || cur < 0 || cur >= n_nodes) { atomicOr(flag, 1); return; }
    const int nb = neighbour[e];
    if (nb < 0 || nb >= n_nodes) atomicOr(flag, 2);
  }
  for (int c = max(prev, -1) + 1; c <= min(cur, n_nodes); ++c) rowptr[c] = (int)e;
}

// ---- tensor-core linear: host side --------------------------------------------------------------
// Pre-sliced weights of one block-diagonal linear (see tc_gemm.cuh): per block l the three bf16 slices of
// W^T in the canonical K-major UMMA layout, cut into (n tile, 32-wide K chunk) blobs that one
// cp.async.bulk moves into a pipeline stage, plus the per-column scales 2^(Eb-7).
struct TcWeights {
  DevBuf q, fb;
  int nblocks = 0;
  bool ok = false;
  struct Blk { int K, N, NT; size_t q_off, fb_off; } blk[kMaxL];
};

// The node linear `name` of layer L runs on the tensor cores: the option is on and its weights were packed.
static bool tc_ready(const LayerCfg& L, const char* name) {
  auto it = L.tcw.find(name);
  return g_opt_tc_gemm && it != L.tcw.end() && it->second && it->second->ok;
}

// column tiling of an N-wide block: as few tiles of <= 128 columns as possible, tile width a multiple of 16;
// the last tile may be padded (zero weights, masked in the epilogue)
static int tc_pick_nt(int N) {
  if (N <= 0) return 0;
  const int tiles = (N + kTcMaxNT - 1) / kTcMaxNT;
  const int w = (N + tiles - 1) / tiles;
  return (w + 15) / 16 * 16;
}
static int tc_tiles(int N, int NT) { return (N + NT - 1) / NT; }

static inline uint16_t bf16_bits_exact(float v) {   // v has <= 8 significant bits: truncation is exact
  uint32_t u;
  memcpy(&u, &v, 4);
  return (uint16_t)(u >> 16);
}

// W [K, N] row-major (fp32) -> q [(N/NT) * (K/32) * 3 * NT*32] bf16 bits, fb [N].  Host only.
static void tc_pack_block(const float* W, int K, int N, int NT, uint16_t* q, float* fb) {
  const int n_kc = K / kTcKC;
  for (int n = 0; n < N; ++n) {
    double amax = 0.0;
    for (int k = 0; k < K; ++k) amax = std::max(amax, (double)fabsf(W[(size_t)k * N + n]));
    int Eb = 0;
    const bool zero = !(amax > 1e-30);
    if (!zero) frexp(amax, &Eb);                       // amax = m * 2^Eb, m in [0.5, 1)  =>  amax < 2^Eb
    fb[n] = zero ? 0.0f : (float)ldexp(1.0, Eb - 7);
    const int nt = n / NT, r = n % NT;
    for (int k = 0; k < K; ++k) {
      double sl[3] = {0.0, 0.0, 0.0};
      if (!zero) {
        const double t = ldexp((double)W[(size_t)k * N + n], 23 - Eb);     // |t| < 2^23, exact
        const double q0 = nearbyint(t / 65536.0);
        const double r1 = t - q0 * 65536.0;
        const double q1 = nearbyint(r1 / 256.0);
        const double r2 = r1 - q1 * 256.0;
        const double q2 = nearbyint(r2);
        sl[0] = q0; sl[1] = q1 / 256.0; sl[2] = q2 / 65536.0;
      }
      const int kc = k / kTcKC, kk = k % kTcKC;
      const size_t elem = (size_t)((r & 7) * 16 + (r >> 3) * 512 + (kk >> 3) * 128 + (kk & 7) * 2) / 2;
      for (int sidx = 0; sidx < 3; ++sidx)
        q[(((size_t)nt * n_kc + kc) * 3 + sidx) * ((size_t)NT * kTcKC) + elem] = bf16_bits_exact((float)sl[sidx]);
    }
  }
}

static int tc_build_weights(TcWeights& w, const float* host, const int* Ks, const int* Ns, int n_l) {
  w.ok = false;
  w.nblocks = 0;
  size_t q_total = 0, fb_total = 0, woff = 0;
  for (int l = 0; l < n_l; ++l) {
    const int K = Ks[l], N = Ns[l];
    if (K == 0 || N == 0) continue;
    const int NT = tc_pick_nt(N);
    if (NT == 0 || K % kTcKC != 0) return 0;          // not expressible: caller keeps the SIMT kernel
    TcWeights::Blk& b = w.blk[w.nblocks++];
    b = {K, N, NT, q_total, fb_total};
    q_total += (size_t)3 * K * NT * tc_tiles(N, NT);
    fb_total += (size_t)N;
  }
  std::vector<uint16_t> q(q_total);
  std::vector<float> fb(fb_total);
  int bi = 0;
  for (int l = 0; l < n_l; ++l) {
    const int K = Ks[l], N = Ns[l];
    if (K == 0 || N == 0) continue;
    const TcWeights::Blk& b = w.blk[bi++];
    tc_pack_block(host + woff, K, N, b.NT, q.data() + b.q_off, fb.data() + b.fb_off);
    woff += (size_t)K * N;
  }
  if (w.q.ensure(q_total * sizeof(uint16_t) + 16) || w.fb.ensure(fb_total * sizeof(float) + 16)) return fail("cudaMalloc failed for tensor-core weights");
  S7B_CUDA_CHECK(cudaMemcpy(w.q.p, q.data(), q_total * sizeof(uint16_t), cudaMemcpyHostToDevice));
  S7B_CUDA_CHECK(cudaMemcpy(w.fb.p, fb.data(), fb_total * sizeof(float), cudaMemcpyHostToDevice));
  w.ok = true;
  return 0;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tensor_map_encoder() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
    else cudaGetLastError();
  }
  return fn;
}

static int launch_row_exponents(RowExp& re, const float* A, int lda, const int* a_off, const int* a_K, int n_l,
                                int n_nodes, cudaStream_t st) {
  RowExpArgs r;
  memset(&r, 0, sizeof(r));
  r.A = A;
  r.lda = lda;
  r.n_nodes = n_nodes;
  int rows = 0;
  for (int l = 0; l < n_l; ++l) {
    if (a_K[l] == 0) continue;
    if (a_K[l] % 4 != 0) return fail("row exponents need K % 4 == 0");
    const int b = r.nblocks++;
    r.d[b] = 2 * l + 1;
    r.K[b] = a_K[l];
    r.a_off[b] = a_off[l];
    r.row_base[b] = rows;
    rows += 2 * l + 1;
  }
  r.rows_per_node = rows;
  re.rows_per_node = rows;
  re.bits = false;
  if (rows == 0 || n_nodes == 0) return 0;
  if (re.buf.ensure((size_t)n_nodes * rows * sizeof(int))) return fail("cudaMalloc failed for row exponents");
  r.E = re.buf.as<int>();
  if (rows > 16) return fail("row exponents: more than 16 rows per node");
  const int blk = 256, wpb = blk / 32;
  row_exponent_kernel<<<(n_nodes + wpb - 1) / wpb, blk, 0, st>>>(r);
  S7B_LAUNCH_CHECK();
  return 0;
}

// C blocks (+)= A blocks * W blocks on the tensor cores.  A's row exponents must be current in `re`.
// Block l of the call uses row group l of `re` (both enumerate l = 0.. over non-empty blocks).
static int launch_tc_linear(const TcWeights& w, const RowExp& re, const float* A, int lda, const int* a_off,
                            const int* a_K, float* C, int ldc, const int* c_off, const int* c_N, int n_l,
                            int n_nodes, bool accumulate, cudaStream_t st) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enc) return fail("cuTensorMapEncodeTiled is unavailable (driver too old?)");
  if (ldc % 4 != 0 || (reinterpret_cast<uintptr_t>(C) & 15) != 0) return fail("tensor-core linear: C rows must be 16-byte aligned");
  for (int l = 0; l < n_l; ++l)
    if (c_N[l] != 0 && a_K[l] != 0 && (c_N[l] % 4 != 0 || c_off[l] % 4 != 0)) return fail("tensor-core linear: output blocks must be multiples of 4 floats");
  TcLinArgs t;
  TcMaps maps;
  memset(&t, 0, sizeof(t));
  memset(&maps, 0, sizeof(maps));
  t.C = C;
  t.E = re.buf.as<int>();
  t.ldc = ldc;
  t.n_nodes = n_nodes;
  t.rows_per_node = re.rows_per_node;
  t.accumulate = accumulate ? 1 : 0;
  t.swizzle = g_opt_tc_swizzle;
  t.e_bits = re.bits ? 1 : 0;
  t.trace = g_tc_trace;
  t.trace_cap = g_tc_trace_cap;
  const int n_mt = (n_nodes + kTcBM - 1) / kTcBM;
  int tiles = 0, rows = 0, bi = 0;
  for (int l = 0; l < n_l; ++l) {
    if (a_K[l] == 0 || c_N[l] == 0) { if (a_K[l] != 0) rows += 2 * l + 1; continue; }
    if (bi >= w.nblocks || w.blk[bi].K != a_K[l] || w.blk[bi].N != c_N[l]) return fail("tensor-core weights do not match the call");
    TcLinBlock& b = t.blk[t.nblocks];
    b.Wq = w.q.as<uint16_t>() + w.blk[bi].q_off;
    b.fb = w.fb.as<float>() + w.blk[bi].fb_off;
    b.d = 2 * l + 1;
    b.K = a_K[l];
    b.N = c_N[l];
    b.NT = w.blk[bi].NT;
    b.nnt = tc_tiles(b.N, b.NT);
    b.c_off = c_off[l];
    b.c_cs = c_N[l];
    b.row_base = rows;
    b.tile0 = tiles;
    tiles += n_mt * b.d * b.nnt;
    rows += 2 * l + 1;
    // A block viewed as (k, component, node): strides K*4 and lda*4 bytes
    const cuuint64_t gdim[3] = {(cuuint64_t)b.K, (cuuint64_t)b.d, (cuuint64_t)n_nodes};
    const cuuint64_t gstr[2] = {(cuuint64_t)b.K * 4, (cuuint64_t)lda * 4};
    const cuuint32_t box[3] = {(cuuint32_t)kTcKC, 1, (cuuint32_t)kTcBM};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult cr = enc(&maps.m[t.nblocks], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void*)(A + a_off[l]), gdim, gstr, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, g_opt_tc_swizzle ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled failed (" + std::to_string((int)cr) + ")");
    ++t.nblocks;
    ++bi;
  }
  if (tiles == 0) return 0;
  t.n_tiles = tiles;
  static int n_sm = 0;
  static bool configured = false;
  if (!configured) {
    int dev = 0;
    S7B_CUDA_CHECK(cudaGetDevice(&dev));
    S7B_CUDA_CHECK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
    S7B_CUDA_CHECK(cudaFuncSetAttribute(blocklin_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemBytes));
    configured = true;
  }
  blocklin_tc_kernel<<<std::min(tiles, n_sm), kTcThreads, kTcSmemBytes, st>>>(t, maps);
  S7B_LAUNCH_CHECK();
  return 0;
}

static int launch_gemm(const LinArgs& a, cudaStream_t st) {
  int max_rows = 0, max_n = 0;
  for (int b = 0; b < a.nblocks; ++b) {
    max_rows = std::max(max_rows, a.n_nodes * a.blk[b].d);
    max_n = std::max(max_n, a.blk[b].N);
  }
  if (max_rows == 0 || max_n == 0) return 0;
  dim3 grid((max_rows + kGemmBM - 1) / kGemmBM, (max_n + kGemmBN - 1) / kGemmBN, a.nblocks);
  blocklin_gemm_kernel<<<grid, kGemmThreads, 0, st>>>(a);
  S7B_LAUNCH_CHECK();
  return 0;
}

// Block-diagonal linear over irreps: for each l < n_l:  C_l (+)= A_l * W_l, W_l = [K_l, N_l]
// stored one after another in `W`.  A blocks: (a_off[l], K = a_K[l]); C blocks: (c_off[l], N = c_N[l]).
static int irreps_linear(const float* A, int lda, const int* a_off, const int* a_K, float* C, int ldc,
                         const int* c_off, const int* c_N, int n_l, const float* W, int n_nodes,
                         bool accumulate, cudaStream_t st) {
  LinArgs a;
  memset(&a, 0, sizeof(a));
  a.A = A;
  a.C = C;
  a.lda = lda;
  a.ldc = ldc;
  a.n_nodes = n_nodes;
  a.accumulate = accumulate ? 1 : 0;
  a.epilogue = kEpiNone;
  a.nblocks = 0;
  size_t woff = 0;
  for (int l = 0; l < n_l; ++l) {
    if (a_K[l] == 0 || c_N[l] == 0) continue;
    LinBlock& b = a.blk[a.nblocks++];
    b.W = W + woff;
    b.d = 2 * l + 1;
    b.K = a_K[l];
    b.N = c_N[l];
    b.a_off = a_off[l];
    b.a_cs = a_K[l];
    b.c_off = c_off[l];
    b.c_cs = c_N[l];
    woff += (size_t)a_K[l] * c_N[l];
  }
  return launch_gemm(a, st);
}

// One block-diagonal node linear of layer `L`, parameter `name`: tensor cores when the shapes allow it
// (default), else the FP32 SIMT kernel.  `re` holds the row exponents of A; `fresh_re` = compute them now
// over the n_l_A irrep blocks of A (a later call on the same A reuses them).
static int node_linear(const LayerCfg& L, const char* name, RowExp& re, bool fresh_re, int n_l_A, const float* A,
                       int lda, const int* a_off, const int* a_K, float* C, int ldc, const int* c_off,
                       const int* c_N, int n_l, const float* W, int n_nodes, bool accumulate, cudaStream_t st) {
  if (tc_ready(L, name)) {
    if (fresh_re && launch_row_exponents(re, A, lda, a_off, a_K, n_l_A, n_nodes, st)) return 1;
    return launch_tc_linear(*L.tcw.at(name), re, A, lda, a_off, a_K, C, ldc, c_off, c_N, n_l, n_nodes, accumulate, st);
  }
  return irreps_linear(A, lda, a_off, a_K, C, ldc, c_off, c_N, n_l, W, n_nodes, accumulate, st);
}

static int dense_gemm(const float* A, int K, float* C, int N, const float* W, int64_t rows, int epilogue,
                      const float* aux_in, float* aux_out, bool accumulate, cudaStream_t st) {
  // rows can exceed what a single grid.x covers comfortably; chunk to stay below 2^31 indexing
  const int64_t chunk = 1 << 22;
  for (int64_t r0 = 0; r0 < rows; r0 += chunk) {
    const int n = (int)std::min<int64_t>(chunk, rows - r0);
    LinArgs a;
    memset(&a, 0, sizeof(a));
    a.A = A + r0 * K;
    a.C = C + r0 * N;
    a.aux_in = aux_in ? aux_in + r0 * N : nullptr;
    a.aux_out = aux_out ? aux_out + r0 * N : nullptr;
    a.lda = K;
    a.ldc = N;
    a.n_nodes = n;
    a.accumulate = accumulate ? 1 : 0;
    a.epilogue = epilogue;
    a.nblocks = 1;
    a.blk[0] = LinBlock{W, 1, K, N, 0, K, 0, N};
    if (launch_gemm(a, st)) return 1;
  }
  return 0;
}

// One tensor-core linear with weights from the host (the test entry points below): packs W_host, computes
// the row exponents of A, launches, waits for `st` and frees the packed weights and exponents again.
// `unsupported` is the error when the shapes have no tensor-core form.
static int tc_linear_once(const float* W_host, const char* unsupported, const float* A, int lda, const int* a_off,
                          const int* a_K, float* C, int ldc, const int* c_off, const int* c_N, int n_l, int n_nodes,
                          bool accumulate, cudaStream_t st) {
  TcWeights w;
  RowExp re;
  int rc = tc_build_weights(w, W_host, a_K, c_N, n_l);
  if (!rc && !w.ok) rc = fail(unsupported);
  if (!rc) rc = launch_row_exponents(re, A, lda, a_off, a_K, n_l, n_nodes, st);
  if (!rc) rc = launch_tc_linear(w, re, A, lda, a_off, a_K, C, ldc, c_off, c_N, n_l, n_nodes, accumulate, st);
  cudaStreamSynchronize(st);
  w.q.release();
  w.fb.release();
  re.buf.release();
  return rc;
}

// launch(l1, stream) for every l1 block of layer L, profiled as `label`.t.l1.  With concurrent convolutions
// (and not profiling) l1 >= 1 run on the side streams, forked from `st` before the first launch and joined
// back into it after each; otherwise everything runs on `st` in order.
template <class Launch>
static int fork_join_l1(S7bEngine* e, const LayerCfg& L, cudaStream_t st, const char* label, int t, Launch launch) {
  const bool par = e->concurrent && g_opt_concurrent && !e->prof.enabled && L.n_lx > 1;
  if (par) S7B_CUDA_CHECK(cudaEventRecord(e->ev_fork, st));
  for (int l1 = 0; l1 < L.n_lx; ++l1) {
    cudaStream_t s1 = (par && l1 > 0) ? e->side[l1] : st;
    if (par && l1 > 0) S7B_CUDA_CHECK(cudaStreamWaitEvent(s1, e->ev_fork, 0));
    ProfScope ps(e->prof, s1, label, t, l1);
    if (launch(l1, s1)) return 1;
    if (par && l1 > 0) {
      S7B_CUDA_CHECK(cudaEventRecord(e->ev_join[l1], s1));
      S7B_CUDA_CHECK(cudaStreamWaitEvent(st, e->ev_join[l1], 0));
    }
  }
  return 0;
}

static int conv_forward(const LayerCfg& L, int lmax_filter, bool table, ConvArgs a, float* out,
                        cudaStream_t st) {
  for (int l1 = 0; l1 < L.n_lx; ++l1)
    if (launch_conv_fwd(l1, lmax_filter, L.lmax_out, table, a, L.roles[l1], out, st)) return 1;
  return 0;
}

}  // namespace s7b

// =========================================================================================
extern "C" {

const char* s7b_last_error(void) { return g_error.c_str(); }
int s7b_version(void) { return 1; }
int64_t s7b_launch_count(int reset) {
  const int64_t v = g_launches + g_conv_launches;
  if (reset) { g_launches = 0; g_conv_launches = 0; }
  return v;
}

int s7b_set_option(const char* name, int value) {
  if (!name) return fail("null option name");
  if (std::string(name) == "tc_gemm") { g_opt_tc_gemm = value; return 0; }
  if (std::string(name) == "tc_swizzle") { g_opt_tc_swizzle = value; return 0; }
  if (std::string(name) == "atomic_virial") { g_opt_atomic_virial = value; return 0; }
  if (std::string(name) == "concurrent_conv") { g_opt_concurrent = value; return 0; }
  if (std::string(name) == "cuda_graph") { g_opt_cuda_graph = value; return 0; }
  if (std::string(name) == "stage_graphs") { g_opt_stage_graphs = value; return 0; }
  if (std::string(name) == "gate_bwd_rows") { g_opt_gate_bwd_rows = value; return 0; }
  return fail(std::string("unknown option: ") + name);
}

int s7b_gather_rows(const float* src, int32_t ld_src, const int32_t* idx, int64_t n, int32_t width, float* out, void* stream) {
  if (n <= 0 || width <= 0) return 0;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool vec = width % 4 == 0 && ld_src % 4 == 0 && (reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(out)) % 16 == 0;
  const size_t total = (size_t)n * (vec ? width / 4 : width);
  const int grd = (int)std::min<size_t>((total + 255) / 256, 148 * 16);
  if (vec) gather_rows_idx_kernel<true><<<grd, 256, 0, st>>>(src, ld_src, idx, n, width, out);
  else gather_rows_idx_kernel<false><<<grd, 256, 0, st>>>(src, ld_src, idx, n, width, out);
  S7B_LAUNCH_CHECK();
  return 0;
}

int s7b_scatter_add_rows(float* dst, int32_t ld_dst, const int32_t* idx, int64_t n, int32_t width, const float* in, void* stream) {
  if (n <= 0 || width <= 0) return 0;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool vec = width % 4 == 0 && ld_dst % 4 == 0 && (reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(in)) % 16 == 0;
  const size_t total = (size_t)n * (vec ? width / 4 : width);
  const int grd = (int)std::min<size_t>((total + 255) / 256, 148 * 16);
  if (vec) scatter_add_rows_idx_kernel<true><<<grd, 256, 0, st>>>(dst, ld_dst, idx, n, width, in);
  else scatter_add_rows_idx_kernel<false><<<grd, 256, 0, st>>>(dst, ld_dst, idx, n, width, in);
  S7B_LAUNCH_CHECK();
  return 0;
}

int s7b_dense_linear(const float* A, const float* W, float* C, int64_t rows, int32_t K, int32_t N,
                     int32_t use_tc, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (rows <= 0 || K <= 0 || N <= 0 || rows > (1 << 24)) return fail("bad sizes");
  if (!use_tc) return dense_gemm(A, K, C, N, W, rows, kEpiNone, nullptr, nullptr, false, st);
  if (K % kTcKC != 0) return fail("tensor-core linear needs K % 32 == 0");
  std::vector<float> hw((size_t)K * N);
  S7B_CUDA_CHECK(cudaMemcpyAsync(hw.data(), W, hw.size() * sizeof(float), cudaMemcpyDeviceToHost, st));
  S7B_CUDA_CHECK(cudaStreamSynchronize(st));
  const int Ks[1] = {K}, Ns[1] = {N}, zero[1] = {0};
  return tc_linear_once(hw.data(), "tensor-core weights could not be built", A, K, zero, Ks, C, N, zero, Ns, 1,
                        (int)rows, false, st);
}

// Debug: record a timeline of CTA 0 of the NEXT tensor-core linear launches into a device buffer the caller
// reads back (tools/tc_trace.py).  cap = 0 turns tracing off.  Returns the device pointer through *buf.
int s7b_tc_trace_enable(int32_t cap, void** buf) {
  if (g_tc_trace) { cudaFree(g_tc_trace); g_tc_trace = nullptr; }
  g_tc_trace_cap = 0;
  if (cap > 0) {
    S7B_CUDA_CHECK(cudaMalloc((void**)&g_tc_trace, (8 + 3 * (size_t)cap) * sizeof(long long)));
    S7B_CUDA_CHECK(cudaMemset(g_tc_trace, 0, (8 + 3 * (size_t)cap) * sizeof(long long)));
    g_tc_trace_cap = cap;
  }
  if (buf) *buf = g_tc_trace;
  return 0;
}

// Test / utility entry: one block-diagonal irreps linear  C_l (+)= A_l W_l  (l = 0..n_l-1, block l has 2l+1
// rows per node) through the engine's GEMM kernels -- use_tc = 1: the tensor-core path exactly as the
// engine drives it (row exponents, packed weights, tensor maps), 0: the FP32 SIMT kernel.  A, C device
// pointers; W host pointer (blocks [K_l, N_l] row-major, concatenated).
int s7b_block_linear(const float* A, int32_t lda, int32_t n_nodes, int32_t n_l, const int32_t* a_off, const int32_t* a_K,
                     const float* W_host, float* C, int32_t ldc, const int32_t* c_off, const int32_t* c_N,
                     int32_t accumulate, int32_t use_tc, void* stream) {
  if (!A || !C || !W_host || !a_off || !a_K || !c_off || !c_N) return fail("null argument");
  if (n_l < 1 || n_l > kMaxL || n_nodes < 1) return fail("bad sizes");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (use_tc)
    return tc_linear_once(W_host, "shapes not supported by the tensor-core linear", A, lda, a_off, a_K, C, ldc, c_off,
                          c_N, n_l, n_nodes, accumulate != 0, st);
  size_t wn = 0;
  for (int l = 0; l < n_l; ++l) wn += (size_t)a_K[l] * c_N[l];
  float* dW = nullptr;
  S7B_CUDA_CHECK(cudaMalloc((void**)&dW, wn * sizeof(float)));
  cudaMemcpy(dW, W_host, wn * sizeof(float), cudaMemcpyHostToDevice);
  const int rc = irreps_linear(A, lda, a_off, a_K, C, ldc, c_off, c_N, n_l, dW, n_nodes, accumulate != 0, st);
  cudaStreamSynchronize(st);
  cudaFree(dW);
  return rc;
}

// Host-only: the tensor-core weight packing of tc_gemm.cuh for one [K, N] block (tests/test_tc_pack_cpu.py).
// q: 3*K*NT*ceil(N/NT) uint16 (bf16 bits; caller allocates 3*K*(N+127) and zero-fills), laid out
// [n tile][K/32][slice][canonical NT x 32]; fb: N floats; *NT_out = tile width.
int s7b_tc_pack_weights(const float* W, int32_t K, int32_t N, uint16_t* q, float* fb, int32_t* NT_out) {
  if (!W || !q || !fb) return fail("null argument");
  const int NT = tc_pick_nt(N);
  if (K <= 0 || K % kTcKC != 0 || NT == 0) return fail("unsupported shape for the tensor-core linear");
  memset(q, 0, (size_t)3 * K * NT * tc_tiles(N, NT) * sizeof(uint16_t));
  tc_pack_block(W, K, N, NT, q, fb);
  if (NT_out) *NT_out = NT;
  return 0;
}

int s7b_engine_create(const S7bModelDesc* d, S7bEngine** out) {
  if (!d || !out) return fail("null argument");
  if (d->n_layers < 1 || d->n_layers > S7B_MAX_LAYERS) return fail("n_layers out of range");
  if (d->lmax_filter < 1 || d->lmax_filter > 3) return fail("lmax_filter must be 1..3");
  if (d->n_basis < 1 || d->n_basis > 8) return fail("n_basis must be 1..8");
  S7bEngine* e = new S7bEngine();
  e->desc = *d;
  e->layers.resize(d->n_layers);
  for (int t = 0; t < d->n_layers; ++t) {
    if (d->n_l[t] < 1 || d->n_l[t] > S7B_MAX_L || d->n_l[t + 1] < 1 || d->n_l[t + 1] > S7B_MAX_L) {
      delete e;
      return fail("irreps lmax out of range");
    }
    if (build_layer_cfg(e->layers[t], d->muls[t], d->n_l[t], d->muls[t + 1], d->n_l[t + 1], d->lmax_filter)) {
      delete e;
      return 1;
    }
  }
  if (e->layers[0].n_lx != 1) {
    delete e;
    return fail("the first layer input must be scalars only");
  }
  for (const LayerCfg& L : e->layers) e->max_lx = std::max(e->max_lx, L.n_lx);
  e->ny_stride = (d->lmax_filter == 3) ? 16 : ((d->lmax_filter == 2) ? 8 : 4);
  const int T = d->n_layers;
  e->x.resize(T);
  e->g.resize(T);
  e->wbuf.resize(T);
  e->z1.resize(T);
  e->z2.resize(T);
  e->h1.resize(T);
  e->h2.resize(T);
  memset(&e->radial, 0, sizeof(e->radial));
  e->radial.cutoff = d->cutoff;
  e->radial.cutoff_fn = d->cutoff_fn;
  e->radial.cutoff_on = d->cutoff_on;
  e->radial.poly_p = d->poly_p;
  e->radial.n_basis = d->n_basis;
  e->radial.knots = d->table_knots > 0 ? d->table_knots : 1;
  e->radial.inv_h = d->table_knots > 0 ? (float)d->table_knots / d->cutoff : 1.0f;
  e->want_atomic_virial = g_opt_atomic_virial != 0;
  for (int i = 1; i < kMaxL; ++i) {
    if (cudaStreamCreateWithFlags(&e->side[i], cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->ev_join[i], cudaEventDisableTiming) != cudaSuccess) {
      delete e;
      return fail("cannot create side streams");
    }
  }
  if (cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming) != cudaSuccess) {
    delete e;
    return fail("cannot create events");
  }
  *out = e;
  return 0;
}

void s7b_engine_destroy(S7bEngine* e) {
  if (!e) return;
  for (int i = 1; i < kMaxL; ++i) {
    if (e->side[i]) cudaStreamDestroy(e->side[i]);
    if (e->ev_join[i]) cudaEventDestroy(e->ev_join[i]);
  }
  if (e->ev_fork) cudaEventDestroy(e->ev_fork);
  if (e->gexec) cudaGraphExecDestroy(e->gexec);
  for (auto& kv : e->stage_graphs) if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  if (e->gstream) cudaStreamDestroy(e->gstream);
  if (e->g_in) cudaEventDestroy(e->g_in);
  if (e->g_out) cudaEventDestroy(e->g_out);
  e->d_nE.release();
  for (auto& kv : e->params) kv.second.release();
  for (auto& L : e->layers) {
    for (auto& kv : L.params) kv.second.release();
    for (auto& kv : L.tcw)
      if (kv.second) { kv.second->q.release(); kv.second->fb.release(); delete kv.second; }
  }
  for (RowExp* r : {&e->re_mid, &e->re_h, &e->re_dg, &e->re_dx}) r->buf.release();
  DevBuf* bufs[] = {&e->rec, &e->Y, &e->rlen, &e->emb, &e->dY_acc, &e->dEdr_acc, &e->demb_acc, &e->fedge,
                    &e->mid, &e->h, &e->dh, &e->dg, &e->dx, &e->dwbuf, &e->tmpA, &e->tmpB, &e->energy,
                    &e->atomic_energy, &e->forces, &e->virial, &e->atomic_virial, &e->hs_species, &e->hs_rowptr, &e->hs_src,
                    &e->hs_vec, &e->hs_centre, &e->hs_flag, &e->nl_pos, &e->nl_wrapped, &e->nl_key, &e->nl_key_sorted,
                    &e->nl_idx, &e->nl_idx_sorted, &e->nl_bin_start, &e->nl_count, &e->nl_tmp, &e->nl_centres};
  for (DevBuf* b : bufs) b->release();
  for (auto* v : {&e->x, &e->g, &e->wbuf, &e->z1, &e->z2, &e->h1, &e->h2})
    for (auto& b : *v) b.release();
  delete e;
}

int s7b_engine_set_atomic_virial(S7bEngine* e, int enable) {
  if (!e) return fail("null engine");
  if (e->want_atomic_virial != (enable != 0)) ++g_alloc_gen;   // a captured step graph bakes the choice in
  e->want_atomic_virial = enable != 0;
  return 0;
}

int s7b_engine_set_param(S7bEngine* e, const char* name, int layer, const float* host, size_t numel) {
  if (!e || !name || !host) return fail("null argument");
  const std::string nm(name);
  if (nm == "bessel") {
    if ((int)numel != e->desc.n_basis) return fail("bessel: wrong size");
    for (int b = 0; b < e->desc.n_basis; ++b) e->radial.coeffs[b] = host[b];
    e->radial_ready = true;
    return 0;
  }
  DevBuf* dst;
  if (layer < 0) dst = &e->params[nm];
  else {
    if (layer >= e->desc.n_layers) return fail("layer out of range");
    dst = &e->layers[layer].params[nm];
  }
  if (dst->ensure(numel * sizeof(float))) return fail("cudaMalloc failed for parameter " + nm);
  S7B_CUDA_CHECK(cudaMemcpy(dst->p, host, numel * sizeof(float), cudaMemcpyHostToDevice));
  if (layer >= 0 && (nm == "si1" || nm == "si1T" || nm == "sc" || nm == "scT" || nm == "si2" || nm == "si2T")) {
    // tensor-core form: block shapes from the layer configuration
    LayerCfg& L = e->layers[layer];
    int Ks[kMaxL] = {0, 0, 0, 0}, Ns[kMaxL] = {0, 0, 0, 0}, n_l = 0;
    const bool T = nm.back() == 'T';
    if (nm.rfind("si1", 0) == 0) { n_l = L.n_lx; for (int l = 0; l < n_l; ++l) { Ks[l] = L.x_muls[l]; Ns[l] = L.x_muls[l]; } }
    else if (nm.rfind("sc", 0) == 0) { n_l = std::min(L.n_lx, L.n_lg); for (int l = 0; l < n_l; ++l) { Ks[l] = L.x_muls[l]; Ns[l] = L.g_muls[l]; } }
    else { n_l = L.n_lg; for (int l = 0; l < n_l; ++l) { Ks[l] = L.mid_K[l]; Ns[l] = L.g_muls[l]; } }
    if (T) for (int l = 0; l < n_l; ++l) std::swap(Ks[l], Ns[l]);
    size_t expect = 0;
    for (int l = 0; l < n_l; ++l) expect += (size_t)Ks[l] * Ns[l];
    if (expect != numel) return fail("parameter " + nm + ": size does not match the layer configuration");
    TcWeights*& w = L.tcw[nm];
    if (!w) w = new TcWeights();
    if (tc_build_weights(*w, host, Ks, Ns, n_l)) return 1;
    ++g_alloc_gen;
  }
  return 0;
}

static const float* lparam(const S7bEngine* e, int t, const char* name) {
  auto it = e->layers[t].params.find(name);
  return it == e->layers[t].params.end() ? nullptr : it->second.as<float>();
}
static const float* gparam(const S7bEngine* e, const char* name) {
  auto it = e->params.find(name);
  return it == e->params.end() ? nullptr : it->second.as<float>();
}

int s7b_engine_set_graph(S7bEngine* e, int32_t n_nodes, int32_t n_local, int64_t n_edges,
                         const int32_t* d_species, const int32_t* d_rowptr, const int32_t* d_src,
                         const float* d_edge_vec, void* stream) {
  if (!e) return fail("null engine");
  if (n_local < 0 || n_nodes < n_local || n_edges < 0) return fail("bad graph sizes");
  if (n_edges >= ((int64_t)1 << 31)) return fail("more than 2^31-1 edges per GPU are not supported");
  e->n_nodes = n_nodes;
  e->n_local = n_local;
  e->n_interior = n_local;
  e->n_edges = n_edges;
  e->d_species = d_species;
  e->d_rowptr = d_rowptr;
  e->d_src = d_src;
  e->d_edge_vec = d_edge_vec;
  const bool table = e->desc.table_knots > 0;
  if (n_edges > e->E_cap || 2 * n_edges < e->E_cap)   // a little headroom, so MD-step fluctuations keep the capacity
    e->E_cap = (n_edges + n_edges / 32 + 1024) / 1024 * 1024;
  if (e->d_nE.ensure(sizeof(int64_t))) return fail("cudaMalloc failed");
  set_i64_kernel<<<1, 1, 0, reinterpret_cast<cudaStream_t>(stream)>>>(e->d_nE.as<int64_t>(), n_edges);
  S7B_LAUNCH_CHECK();
  const size_t E = (size_t)e->E_cap, Nn = (size_t)std::max(n_nodes, 1), Nl = (size_t)std::max(n_local, 1);
  const int T = e->desc.n_layers;
  int rc = 0;
  rc |= e->rec.ensure(E * sizeof(int4));
  rc |= e->Y.ensure(E * e->ny_stride * sizeof(float));
  rc |= e->rlen.ensure(E * sizeof(float));
  rc |= e->dY_acc.ensure((size_t)e->max_lx * E * e->ny_stride * sizeof(float));
  rc |= e->dEdr_acc.ensure((size_t)e->max_lx * E * sizeof(float));
  rc |= e->fedge.ensure(E * 3 * sizeof(float));
  size_t max_mid = 0, max_h = 0, max_g = 0, max_x = 0, max_W = 0;
  for (int t = 0; t < T; ++t) {
    const LayerCfg& L = e->layers[t];
    rc |= e->x[t].ensure(Nn * L.dim_x * sizeof(float));
    rc |= e->g[t].ensure(Nl * L.dim_g * sizeof(float));
    max_mid = std::max(max_mid, (size_t)L.dim_mid);
    max_h = std::max(max_h, (size_t)L.dim_h);
    max_g = std::max(max_g, (size_t)L.dim_g);
    max_x = std::max(max_x, (size_t)L.dim_x);
    max_W = std::max(max_W, (size_t)L.W);
    if (!table) {
      const int h0 = e->desc.radial_hidden[0], h1 = e->desc.radial_hidden[1];
      rc |= e->wbuf[t].ensure(E * L.W * sizeof(float));
      rc |= e->z1[t].ensure(E * h0 * sizeof(float));
      rc |= e->h1[t].ensure(E * h0 * sizeof(float));
      rc |= e->z2[t].ensure(E * h1 * sizeof(float));
      rc |= e->h2[t].ensure(E * h1 * sizeof(float));
    }
  }
  if (!table) {
    rc |= e->emb.ensure(E * e->desc.n_basis * sizeof(float));
    rc |= e->demb_acc.ensure(E * e->desc.n_basis * sizeof(float));
    rc |= e->dwbuf.ensure(E * max_W * sizeof(float));
    const size_t hh = (size_t)std::max(e->desc.radial_hidden[0], e->desc.radial_hidden[1]);
    rc |= e->tmpA.ensure(E * hh * sizeof(float));
    rc |= e->tmpB.ensure(E * hh * sizeof(float));
  }
  rc |= e->mid.ensure(Nl * max_mid * sizeof(float));
  rc |= e->h.ensure(Nl * std::max(max_h, max_x) * sizeof(float));
  rc |= e->dh.ensure(Nl * std::max(max_h, max_x) * sizeof(float));
  rc |= e->dg.ensure(Nl * max_g * sizeof(float));
  rc |= e->dx.ensure(Nn * max_x * sizeof(float));
  // row exponents of the tensor-core GEMM inputs (at most 1+3+5+7 rows per node); sized here because the
  // step may be recorded into a CUDA graph, where cudaMalloc is not allowed
  for (RowExp* r : {&e->re_mid, &e->re_h, &e->re_dg, &e->re_dx}) rc |= r->buf.ensure(Nn * 16 * sizeof(int));
  rc |= e->energy.ensure(sizeof(double));
  rc |= e->virial.ensure(6 * sizeof(double));
  rc |= e->atomic_energy.ensure(Nl * sizeof(float));
  rc |= e->forces.ensure(Nn * 3 * sizeof(float));
  if (e->want_atomic_virial) rc |= e->atomic_virial.ensure(Nn * 6 * sizeof(float));
  if (rc) return fail("cudaMalloc failed while sizing step buffers");
  return 0;
}

int s7b_engine_set_interior(S7bEngine* e, int32_t n_interior) {
  if (!e) return fail("null engine");
  if (n_interior < 0 || n_interior > e->n_local) return fail("n_interior out of range");
  e->n_interior = n_interior;
  return 0;
}

static ConvArgs make_conv_args(const S7bEngine* e, int t, const float* x) {
  const LayerCfg& L = e->layers[t];
  ConvArgs a;
  memset(&a, 0, sizeof(a));
  a.rowptr = e->d_rowptr;
  a.rec = e->rec.as<int4>();
  a.Y = e->Y.as<float>();
  a.x = x;
  a.table = reinterpret_cast<const float4*>(lparam(e, t, "table"));
  a.table23 = reinterpret_cast<const uint2*>(lparam(e, t, "table23"));
  a.w = e->desc.table_knots > 0 ? nullptr : e->wbuf[t].as<float>();
  a.n_dst = e->n_local;
  a.dim_x = L.dim_x;
  a.dim_mid = L.dim_mid;
  a.w_numel = L.W;
  a.ny_stride = e->ny_stride;
  a.inv_h = e->radial.inv_h;
  return a;
}

static int grid1d(size_t total, int block) {
  size_t g = (total + block - 1) / block;
  if (g > 148 * 64) g = 148 * 64;
  if (g < 1) g = 1;
  return (int)g;
}

static int require(const void* p, const char* what) {
  if (p) return 0;
  return fail(std::string("missing parameter: ") + what);
}

static int run_stage_impl(S7bEngine* e, int stage, int t, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int T = e->desc.n_layers;
  const int Nn = e->n_nodes, Nl = e->n_local;
  const int64_t E = e->n_edges;
  const int64_t Ecap = e->E_cap;          // stride of the per-l1 parts of dY_acc / dEdr_acc, grid of the edge kernels
  const int64_t* nE = e->d_nE.as<int64_t>();
  const bool table = e->desc.table_knots > 0;
  const int LF = e->desc.lmax_filter;
  if (!e->radial_ready) return fail("parameter 'bessel' was not set");

  switch (stage) {
    case S7B_STAGE_FWD_BEGIN: {
      if (E > 0) {
        const int blk = 256;
        const int grd = (int)((Ecap + blk - 1) / blk);
        float* emb = table ? nullptr : e->emb.as<float>();
        ProfScope ps(e->prof, st, "edge_fwd");
        if (LF == 1) edge_fwd_kernel<1><<<grd, blk, 0, st>>>(e->radial, e->d_edge_vec, e->d_src, nE, e->ny_stride, e->rec.as<int4>(), e->Y.as<float>(), e->rlen.as<float>(), emb);
        else if (LF == 2) edge_fwd_kernel<2><<<grd, blk, 0, st>>>(e->radial, e->d_edge_vec, e->d_src, nE, e->ny_stride, e->rec.as<int4>(), e->Y.as<float>(), e->rlen.as<float>(), emb);
        else edge_fwd_kernel<3><<<grd, blk, 0, st>>>(e->radial, e->d_edge_vec, e->d_src, nE, e->ny_stride, e->rec.as<int4>(), e->Y.as<float>(), e->rlen.as<float>(), emb);
        S7B_LAUNCH_CHECK();
        S7B_CUDA_CHECK(cudaMemsetAsync(e->dY_acc.p, 0, (size_t)e->max_lx * Ecap * e->ny_stride * sizeof(float), st));
        S7B_CUDA_CHECK(cudaMemsetAsync(e->dEdr_acc.p, 0, (size_t)e->max_lx * Ecap * sizeof(float), st));
        if (!table) S7B_CUDA_CHECK(cudaMemsetAsync(e->demb_acc.p, 0, (size_t)E * e->desc.n_basis * sizeof(float), st));
      }
      const LayerCfg& L0 = e->layers[0];
      const float* ex = gparam(e, "embed_x0");
      const float* eg = gparam(e, "embed_g0");
      if (require(ex, "embed_x0") || require(eg, "embed_g0")) return 1;
      ProfScope ps(e->prof, st, "embed_gather");
      if (Nn > 0) {
        gather_rows_kernel<<<grid1d((size_t)Nn * L0.dim_x, 256), 256, 0, st>>>(ex, e->d_species, e->x[0].as<float>(), Nn, L0.dim_x, L0.dim_x);
        S7B_LAUNCH_CHECK();
      }
      if (Nl > 0) {
        gather_rows_kernel<<<grid1d((size_t)Nl * L0.dim_g, 256), 256, 0, st>>>(eg, e->d_species, e->g[0].as<float>(), Nl, L0.dim_g, L0.dim_g);
        S7B_LAUNCH_CHECK();
      }
      return 0;
    }
    case S7B_STAGE_FWD_LAYER:
    case S7B_STAGE_FWD_LAYER_A:
    case S7B_STAGE_FWD_CONV_INTERIOR:
    case S7B_STAGE_FWD_LAYER_A2: {
      if (t < 0 || t >= T) return fail("layer out of range");
      const LayerCfg& L = e->layers[t];
      if (Nl == 0) return 0;
      const bool head = stage != S7B_STAGE_FWD_LAYER_A2;
      if (head && !table && E > 0) {
        // exact radial MLP (convolution.py:121): emb -> h1 -> h2 -> w
        const float *w0 = lparam(e, t, "mlp0"), *w1 = lparam(e, t, "mlp1"), *w2 = lparam(e, t, "mlp2");
        if (require(w0, "mlp0") || require(w1, "mlp1") || require(w2, "mlp2")) return 1;
        const int nb = e->desc.n_basis, h0 = e->desc.radial_hidden[0], h1 = e->desc.radial_hidden[1];
        ProfScope ps(e->prof, st, "radial_mlp_fwd", t);
        if (dense_gemm(e->emb.as<float>(), nb, e->h1[t].as<float>(), h0, w0, E, kEpiSiluStoreZ, nullptr, e->z1[t].as<float>(), false, st)) return 1;
        if (dense_gemm(e->h1[t].as<float>(), h0, e->h2[t].as<float>(), h1, w1, E, kEpiSiluStoreZ, nullptr, e->z2[t].as<float>(), false, st)) return 1;
        if (dense_gemm(e->h2[t].as<float>(), h1, e->wbuf[t].as<float>(), L.W, w2, E, kEpiNone, nullptr, nullptr, false, st)) return 1;
      } else if (head && table) {
        if (require(lparam(e, t, "table"), "table") || require(lparam(e, t, "table23"), "table23")) return 1;
      }
      // convolution: gather + tensor product + scatter (raw sums; 1/denominator is folded into si2)
      ConvArgs ca = make_conv_args(e, t, e->x[t].as<float>());
      if (stage == S7B_STAGE_FWD_CONV_INTERIOR) ca.n_dst = e->n_interior;
      if (stage == S7B_STAGE_FWD_LAYER_A2) ca.n_begin = e->n_interior;
      // the convolution kernels also leave the row maxima of `mid` for the tensor-core self_interaction_2
      const bool fused_rows = tc_ready(L, "si2");
      if (fused_rows) {
        e->re_mid.rows_per_node = L.n_lg * L.n_lg;
        e->re_mid.bits = true;
        if (head) S7B_CUDA_CHECK(cudaMemsetAsync(e->re_mid.buf.p, 0, (size_t)Nl * e->re_mid.rows_per_node * sizeof(int), st));
        ca.row_max = e->re_mid.buf.as<unsigned int>();
        ca.rows_per_node = e->re_mid.rows_per_node;
      }
      if (fork_join_l1(e, L, st, "conv_fwd", t, [&](int l1, cudaStream_t s1) {
            return launch_conv_fwd(l1, LF, L.lmax_out, table, ca, L.roles[l1], e->mid.as<float>(), s1);
          }))
        return 1;
      if (stage == S7B_STAGE_FWD_CONV_INTERIOR) return 0;
      // self_interaction_2 accumulated onto the self-connection already stored in g[t]
      const float* si2 = lparam(e, t, "si2");
      if (require(si2, "si2")) return 1;
      {
        ProfScope ps(e->prof, st, "si2_gemm", t);
        if (node_linear(L, "si2", e->re_mid, !fused_rows, L.n_lg, e->mid.as<float>(), L.dim_mid, L.mid_off, L.mid_K, e->g[t].as<float>(), L.dim_g, L.g_off, L.g_muls, L.n_lg, si2, Nl, true, st)) return 1;
      }
      // gate
      // gate; with the tensor-core linears the kernel also leaves the row exponents of h for self_interaction_1 / sc
      const bool h_rows = t + 1 < T && tc_ready(e->layers[t + 1], "si1") && L.n_lg * L.n_lg <= 16;
      {
        ProfScope ps(e->prof, st, "gate_fwd", t);
        if (h_rows) {
          e->re_h.rows_per_node = L.n_lg * L.n_lg;
          e->re_h.bits = false;
          gate_fwd_rows_kernel<<<(Nl + 7) / 8, 256, 0, st>>>(L.gate, e->g[t].as<float>(), e->h.as<float>(), Nl, e->re_h.buf.as<int>(), e->re_h.rows_per_node, kTcZeroRow);
        } else {
          gate_fwd_kernel<<<grid1d((size_t)Nl * L.dim_h, 256), 256, 0, st>>>(L.gate, e->g[t].as<float>(), e->h.as<float>(), Nl);
        }
        S7B_LAUNCH_CHECK();
      }
      if (t + 1 < T) {
        const LayerCfg& N = e->layers[t + 1];
        const float* si1 = lparam(e, t + 1, "si1");
        if (require(si1, "si1")) return 1;
        ProfScope ps(e->prof, st, "si1_gemm", t + 1);
        // self_interaction_1 of the next layer -> local rows of x[t+1] (ghost rows: caller's exchange)
        if (node_linear(N, "si1", e->re_h, !h_rows, N.n_lx, e->h.as<float>(), N.dim_x, N.x_off, N.x_muls, e->x[t + 1].as<float>(), N.dim_x, N.x_off, N.x_muls, N.n_lx, si1, Nl, false, st)) return 1;
      }
      if (stage != S7B_STAGE_FWD_LAYER) return 0;
    }
    // fall through: FWD_LAYER = FWD_LAYER_A + FWD_LAYER_SC
    case S7B_STAGE_FWD_LAYER_SC: {
      if (t < 0 || t >= T) return fail("layer out of range");
      if (Nl == 0 || t + 1 >= T) return 0;
      const LayerCfg& N = e->layers[t + 1];
      const float* sc = lparam(e, t + 1, "sc");
      if (require(sc, "sc")) return 1;
      ProfScope ps(e->prof, st, "sc_gemm", t + 1);
      // self_connection_intro of the next layer -> initial value of g[t+1]; independent of the ghost
      // exchange of x[t+1], so multi-GPU callers overlap the two
      S7B_CUDA_CHECK(cudaMemsetAsync(e->g[t + 1].p, 0, (size_t)Nl * N.dim_g * sizeof(float), st));
      const int n_sc = std::min(N.n_lx, N.n_lg);
      if (node_linear(N, "sc", e->re_h, false, N.n_lx, e->h.as<float>(), N.dim_x, N.x_off, N.x_muls, e->g[t + 1].as<float>(), N.dim_g, N.g_off, N.g_muls, n_sc, sc, Nl, false, st)) return 1;
      return 0;
    }
    case S7B_STAGE_FWD_END: {
      const LayerCfg& L = e->layers[T - 1];
      const float *wr = gparam(e, "readout"), *scale = gparam(e, "scale"), *shift = gparam(e, "shift");
      if (require(wr, "readout") || require(scale, "scale") || require(shift, "shift")) return 1;
      S7B_CUDA_CHECK(cudaMemsetAsync(e->energy.p, 0, sizeof(double), st));
      if (Nl > 0) {
        const int blk = 256;
        ProfScope ps(e->prof, st, "readout");
        readout_kernel<<<(Nl * 32 + blk - 1) / blk, blk, 0, st>>>(e->h.as<float>(), wr, gparam(e, "readout_lo"), scale, shift, e->d_species, Nl, L.dim_h, e->atomic_energy.as<float>(), e->energy.as<double>(), e->dh.as<float>());
        S7B_LAUNCH_CHECK();
      }
      return 0;
    }
    case S7B_STAGE_BWD_LAYER_A:
    case S7B_STAGE_BWD_LAYER_A1:
    case S7B_STAGE_BWD_LAYER_A2: {
      if (t < 0 || t >= T) return fail("layer out of range");
      const LayerCfg& L = e->layers[t];
      const bool head = stage != S7B_STAGE_BWD_LAYER_A2, tail = stage != S7B_STAGE_BWD_LAYER_A1;
      if (head && t > 0 && Nn > 0) S7B_CUDA_CHECK(cudaMemsetAsync(e->dx.p, 0, (size_t)Nn * L.dim_x * sizeof(float), st));
      if (Nl == 0) return 0;
      if (head) {
        const bool dg_rows = g_opt_gate_bwd_rows && tc_ready(L, "si2T") && L.n_lg * L.n_lg <= 16;
        {
          ProfScope ps(e->prof, st, "gate_bwd", t);
          if (dg_rows) {      // ... and the row exponents of dg for si2^T / sc^T
            e->re_dg.rows_per_node = L.n_lg * L.n_lg;
            e->re_dg.bits = true;
            S7B_CUDA_CHECK(cudaMemsetAsync(e->re_dg.buf.p, 0, (size_t)Nl * e->re_dg.rows_per_node * sizeof(int), st));
            gate_bwd_rows_kernel<<<grid1d((size_t)Nl * L.dim_g, 256), 256, 0, st>>>(L.gate, e->g[t].as<float>(), e->dh.as<float>(), e->dg.as<float>(), Nl, e->re_dg.buf.as<unsigned int>(), e->re_dg.rows_per_node);
          } else {
            gate_bwd_kernel<<<grid1d((size_t)Nl * L.dim_g, 256), 256, 0, st>>>(L.gate, e->g[t].as<float>(), e->dh.as<float>(), e->dg.as<float>(), Nl);
          }
          S7B_LAUNCH_CHECK();
        }
        const float* si2T = lparam(e, t, "si2T");
        if (require(si2T, "si2T")) return 1;
        // d(mid) = dg * si2^T
        ProfScope ps(e->prof, st, "si2T_gemm", t);
        if (node_linear(L, "si2T", e->re_dg, !dg_rows, L.n_lg, e->dg.as<float>(), L.dim_g, L.g_off, L.g_muls, e->mid.as<float>(), L.dim_mid, L.mid_off, L.mid_K, L.n_lg, si2T, Nl, false, st)) return 1;
      }
      if (E > 0) {
        ConvArgs ca = make_conv_args(e, t, e->x[t].as<float>());
        if (stage == S7B_STAGE_BWD_LAYER_A1) ca.n_begin = e->n_interior;     // boundary atoms first: they own the ghost rows of dx
        if (stage == S7B_STAGE_BWD_LAYER_A2) ca.n_dst = e->n_interior;
        if (fork_join_l1(e, L, st, "conv_bwd", t, [&](int l1, cudaStream_t s1) {
              float* dY = e->dY_acc.as<float>() + (size_t)l1 * Ecap * e->ny_stride;
              float* dEdr = e->dEdr_acc.as<float>() + (size_t)l1 * Ecap;
              return launch_conv_bwd(l1, LF, L.lmax_out, table, t > 0, ca, L.roles[l1], e->mid.as<float>(), e->dx.as<float>(), dY, dEdr, table ? nullptr : e->dwbuf.as<float>(), s1);
            }))
          return 1;
        if (!table && tail) {
          // radial MLP backward: dw -> demb (accumulated over layers)
          const float *w0T = lparam(e, t, "mlp0T"), *w1T = lparam(e, t, "mlp1T"), *w2T = lparam(e, t, "mlp2T");
          if (require(w0T, "mlp0T") || require(w1T, "mlp1T") || require(w2T, "mlp2T")) return 1;
          const int nb = e->desc.n_basis, h0 = e->desc.radial_hidden[0], h1 = e->desc.radial_hidden[1];
          ProfScope ps(e->prof, st, "radial_mlp_bwd", t);
          if (dense_gemm(e->dwbuf.as<float>(), L.W, e->tmpA.as<float>(), h1, w2T, E, kEpiMulDsilu, e->z2[t].as<float>(), nullptr, false, st)) return 1;
          if (dense_gemm(e->tmpA.as<float>(), h1, e->tmpB.as<float>(), h0, w1T, E, kEpiMulDsilu, e->z1[t].as<float>(), nullptr, false, st)) return 1;
          if (dense_gemm(e->tmpB.as<float>(), h0, e->demb_acc.as<float>(), nb, w0T, E, kEpiNone, nullptr, nullptr, true, st)) return 1;
        }
      }
      return 0;
    }
    case S7B_STAGE_BWD_LAYER_B:
    case S7B_STAGE_BWD_LAYER_B1:
    case S7B_STAGE_BWD_LAYER_B2: {
      if (t <= 0 || t >= T) return fail("BWD_LAYER_B needs 1 <= layer < n_layers");
      const LayerCfg& L = e->layers[t];
      if (Nl == 0) return 0;
      const float *si1T = lparam(e, t, "si1T"), *scT = lparam(e, t, "scT");
      if (require(si1T, "si1T") || require(scT, "scT")) return 1;
      // dE/dh(t) = dg(t) * sc^T + dx(t) * si1^T     (h(t) = gate output of layer t-1).  B1 (the self-
      // connection term) does not need the reverse ghost exchange of dx and can overlap it; B2 adds the rest.
      ProfScope ps(e->prof, st, "si1T_scT_gemm", t);
      if (stage != S7B_STAGE_BWD_LAYER_B2) {
        const int n_sc = std::min(L.n_lx, L.n_lg);
        S7B_CUDA_CHECK(cudaMemsetAsync(e->dh.p, 0, (size_t)Nl * L.dim_x * sizeof(float), st));
        if (node_linear(L, "scT", e->re_dg, false, L.n_lg, e->dg.as<float>(), L.dim_g, L.g_off, L.g_muls, e->dh.as<float>(), L.dim_x, L.x_off, L.x_muls, n_sc, scT, Nl, false, st)) return 1;
      }
      if (stage != S7B_STAGE_BWD_LAYER_B1) {
        if (node_linear(L, "si1T", e->re_dx, true, L.n_lx, e->dx.as<float>(), L.dim_x, L.x_off, L.x_muls, e->dh.as<float>(), L.dim_x, L.x_off, L.x_muls, L.n_lx, si1T, Nl, true, st)) return 1;
      }
      return 0;
    }
    case S7B_STAGE_BWD_END: {
      S7B_CUDA_CHECK(cudaMemsetAsync(e->forces.p, 0, (size_t)std::max(Nn, 1) * 3 * sizeof(float), st));
      S7B_CUDA_CHECK(cudaMemsetAsync(e->virial.p, 0, 6 * sizeof(double), st));
      const bool av = e->want_atomic_virial && e->atomic_virial.p != nullptr;
      if (av) S7B_CUDA_CHECK(cudaMemsetAsync(e->atomic_virial.p, 0, (size_t)std::max(Nn, 1) * 6 * sizeof(float), st));
      if (E > 0 && Nl > 0) {
        const int blk = 256;
        const int grd = (int)((Ecap + blk - 1) / blk);
        const float* dEdr = table ? e->dEdr_acc.as<float>() : nullptr;
        const float* demb = table ? nullptr : e->demb_acc.as<float>();
        ProfScope ps(e->prof, st, "edge_bwd_force_scatter");
        if (LF == 1) edge_bwd_kernel<1><<<grd, blk, 0, st>>>(e->radial, e->d_edge_vec, nE, Ecap, e->ny_stride, e->max_lx, e->dY_acc.as<float>(), dEdr, demb, e->fedge.as<float>());
        else if (LF == 2) edge_bwd_kernel<2><<<grd, blk, 0, st>>>(e->radial, e->d_edge_vec, nE, Ecap, e->ny_stride, e->max_lx, e->dY_acc.as<float>(), dEdr, demb, e->fedge.as<float>());
        else edge_bwd_kernel<3><<<grd, blk, 0, st>>>(e->radial, e->d_edge_vec, nE, Ecap, e->ny_stride, e->max_lx, e->dY_acc.as<float>(), dEdr, demb, e->fedge.as<float>());
        S7B_LAUNCH_CHECK();
        force_scatter_kernel<<<(Nl * 32 + blk - 1) / blk, blk, 0, st>>>(e->d_rowptr, e->d_src, e->d_edge_vec, e->fedge.as<float>(), Nl, e->forces.as<float>(), e->virial.as<double>(), av ? e->atomic_virial.as<float>() : nullptr);
        S7B_LAUNCH_CHECK();
      }
      return 0;
    }
    default:
      return fail("unknown stage");
  }
}

// everything a captured graph bakes in: sizes, edge capacity, graph-array pointers, any (re)allocation, the options
static std::vector<int64_t> graph_key(const S7bEngine* e) {
  return {e->n_nodes, e->n_local, e->n_interior, e->E_cap, e->n_edges > 0 ? 1 : 0, (int64_t)(uintptr_t)e->d_species,
          (int64_t)(uintptr_t)e->d_rowptr, (int64_t)(uintptr_t)e->d_src, (int64_t)(uintptr_t)e->d_edge_vec,
          g_alloc_gen, g_opt_concurrent, g_opt_tc_gemm + 2 * g_opt_tc_swizzle + 4 * g_opt_gate_bwd_rows, e->concurrent ? 1 : 0,
          e->want_atomic_virial ? 1 : 0};
}

static int ensure_graph_stream(S7bEngine* e) {
  if (e->gstream) return 0;
  S7B_CUDA_CHECK(cudaStreamCreateWithFlags(&e->gstream, cudaStreamNonBlocking));
  S7B_CUDA_CHECK(cudaEventCreateWithFlags(&e->g_in, cudaEventDisableTiming));
  S7B_CUDA_CHECK(cudaEventCreateWithFlags(&e->g_out, cudaEventDisableTiming));
  return 0;
}

// capture fn(gstream) into an executable graph; *launches = kernels recorded
static int capture_graph(S7bEngine* e, const std::function<int(cudaStream_t)>& fn, cudaGraphExec_t* exec, int64_t* launches) {
  const int64_t before = g_launches + g_conv_launches;
  S7B_CUDA_CHECK(cudaStreamBeginCapture(e->gstream, cudaStreamCaptureModeThreadLocal));
  e->capturing = true;
  const int rc = fn(e->gstream);
  e->capturing = false;
  cudaGraph_t graph = nullptr;
  const cudaError_t ce = cudaStreamEndCapture(e->gstream, &graph);
  *launches = g_launches + g_conv_launches - before;
  g_launches -= *launches;                 // recorded, not launched
  if (rc) { if (graph) cudaGraphDestroy(graph); return 1; }
  if (ce != cudaSuccess) { cudaGetLastError(); return fail(std::string("CUDA graph capture failed: ") + cudaGetErrorString(ce)); }
  const cudaError_t ci = cudaGraphInstantiate(exec, graph, 0);
  cudaGraphDestroy(graph);
  if (ci != cudaSuccess) { *exec = nullptr; cudaGetLastError(); return fail(std::string("cudaGraphInstantiate failed: ") + cudaGetErrorString(ci)); }
  return 0;
}

// A caller that drives the stages itself (multi-GPU runner: ghost exchanges between the stages; LAMMPS
// front-ends) cannot replay the whole step as one graph, but every stage between two exchanges still is a
// fixed launch sequence: with option "stage_graphs" each (stage, layer) is captured once and replayed on the
// caller's stream -- ~22 graph launches per step instead of ~170 kernel launches.  An entry whose key keeps
// changing (positions-in MD: new graph arrays every step) stops capturing after three wasted captures.
int s7b_engine_run_stage(S7bEngine* e, int stage, int t, void* stream) {
  if (!e) return fail("null engine");
  const bool table = e->desc.table_knots > 0;
  if (!g_opt_stage_graphs || e->capturing || !table || e->prof.enabled || !e->radial_ready)
    return run_stage_impl(e, stage, t, stream);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) { cudaGetLastError(); return run_stage_impl(e, stage, t, stream); }
  if (cs != cudaStreamCaptureStatusNone) return run_stage_impl(e, stage, t, stream);    // the caller is capturing already
  S7bEngine::StageGraph& sg = e->stage_graphs[stage * 64 + t];
  if (sg.thrash >= 3) return run_stage_impl(e, stage, t, stream);
  const std::vector<int64_t> key = graph_key(e);
  if (!sg.exec || key != sg.key) {
    if (sg.exec) {
      cudaGraphExecDestroy(sg.exec);
      sg.exec = nullptr;
      if (sg.replays_since_capture < 2 && ++sg.thrash >= 3) return run_stage_impl(e, stage, t, stream);
    }
    if (ensure_graph_stream(e)) return 1;
    if (capture_graph(e, [&](cudaStream_t s) { return run_stage_impl(e, stage, t, s); }, &sg.exec, &sg.launches)) {
      sg.exec = nullptr;                 // a stage that cannot be captured keeps its direct launches
      sg.thrash = 3;
      return run_stage_impl(e, stage, t, stream);
    }
    sg.key = key;
    sg.replays_since_capture = 0;
    ++e->sg_captures;
  }
  S7B_CUDA_CHECK(cudaGraphLaunch(sg.exec, st));
  g_launches += sg.launches;
  ++sg.replays_since_capture;
  ++e->sg_replays;
  return 0;
}

static int run_all_stages(S7bEngine* e, void* stream) {
  const int T = e->desc.n_layers;
  if (run_stage_impl(e, S7B_STAGE_FWD_BEGIN, 0, stream)) return 1;
  for (int t = 0; t < T; ++t)
    if (run_stage_impl(e, S7B_STAGE_FWD_LAYER, t, stream)) return 1;
  if (run_stage_impl(e, S7B_STAGE_FWD_END, 0, stream)) return 1;
  for (int t = T - 1; t >= 0; --t) {
    if (run_stage_impl(e, S7B_STAGE_BWD_LAYER_A, t, stream)) return 1;
    if (t > 0 && run_stage_impl(e, S7B_STAGE_BWD_LAYER_B, t, stream)) return 1;
  }
  return run_stage_impl(e, S7B_STAGE_BWD_END, 0, stream);
}

// The whole step is ~75 launches; below a few thousand atoms their launch latency, not the kernels, sets
// the step time.  The step is therefore captured once into a CUDA graph (on an engine-owned stream,
// side-stream fork/joins included) and replayed for as long as nothing baked into it changes: sizes,
// edge capacity, graph-array pointers, any (re)allocation, the options.  The live edge count is read
// from device memory by the edge kernels (see S7bEngine::E_cap), so MD steps with a drifting
// neighbour count replay the same graph.
int s7b_engine_compute(S7bEngine* e, void* stream) {
  if (!e) return fail("null engine");
  const bool table = e->desc.table_knots > 0;
  if (!g_opt_cuda_graph || !table || e->prof.enabled) return run_all_stages(e, stream);
  if (!e->radial_ready) return fail("parameter 'bessel' was not set");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (ensure_graph_stream(e)) return 1;
  const std::vector<int64_t> key = graph_key(e);
  if (!e->gexec || key != e->g_key) {
    if (e->gexec) { cudaGraphExecDestroy(e->gexec); e->gexec = nullptr; }
    if (capture_graph(e, [&](cudaStream_t s) { return run_all_stages(e, s); }, &e->gexec, &e->g_launches_per_replay)) return 1;
    e->g_key = key;
    ++e->g_captures;
  }
  S7B_CUDA_CHECK(cudaEventRecord(e->g_in, st));
  S7B_CUDA_CHECK(cudaStreamWaitEvent(e->gstream, e->g_in, 0));
  S7B_CUDA_CHECK(cudaGraphLaunch(e->gexec, e->gstream));
  S7B_CUDA_CHECK(cudaEventRecord(e->g_out, e->gstream));
  S7B_CUDA_CHECK(cudaStreamWaitEvent(st, e->g_out, 0));
  g_launches += e->g_launches_per_replay;
  ++e->g_replays;
  return 0;
}

int s7b_engine_graph_stats(S7bEngine* e, int64_t* captures, int64_t* replays) {
  if (!e) return fail("null engine");
  if (captures) *captures = e->g_captures;
  if (replays) *replays = e->g_replays;
  return 0;
}

int s7b_engine_stage_graph_stats(S7bEngine* e, int64_t* captures, int64_t* replays) {
  if (!e) return fail("null engine");
  if (captures) *captures = e->sg_captures;
  if (replays) *replays = e->sg_replays;
  return 0;
}

int s7b_engine_set_profiling(S7bEngine* e, int enable) {
  if (!e) return fail("null engine");
  e->prof.clear();
  e->prof.enabled = enable != 0;
  return 0;
}

int s7b_engine_profile_count(S7bEngine* e) {
  if (!e) return 0;
  e->prof.collect();
  return (int)e->prof.totals.size();
}

int s7b_engine_profile_entry(S7bEngine* e, int index, char* name, size_t name_len, double* total_ms,
                             int64_t* calls) {
  if (!e) return fail("null engine");
  e->prof.collect();
  if (index < 0 || index >= (int)e->prof.totals.size()) return fail("profile index out of range");
  auto it = e->prof.totals.begin();
  std::advance(it, index);
  if (name && name_len > 0) snprintf(name, name_len, "%s", it->first.c_str());
  if (total_ms) *total_ms = it->second.first;
  if (calls) *calls = it->second.second;
  return 0;
}

void* s7b_engine_buffer(S7bEngine* e, const char* name, int layer, size_t* numel) {
  if (!e || !name) return nullptr;
  const std::string nm(name);
  const int T = e->desc.n_layers;
  size_t n = 0;
  void* p = nullptr;
  auto in_range = [&](int t) { return t >= 0 && t < T; };
  if (nm == "x" && in_range(layer)) { p = e->x[layer].p; n = (size_t)e->n_nodes * e->layers[layer].dim_x; }
  else if (nm == "gate_in" && in_range(layer)) { p = e->g[layer].p; n = (size_t)e->n_local * e->layers[layer].dim_g; }
  else if (nm == "weight" && in_range(layer)) { p = e->wbuf[layer].p; n = (size_t)e->n_edges * e->layers[layer].W; }
  else if (nm == "dx" && in_range(layer)) { p = e->dx.p; n = (size_t)e->n_nodes * e->layers[layer].dim_x; }
  else if (nm == "dg" && in_range(layer)) { p = e->dg.p; n = (size_t)e->n_local * e->layers[layer].dim_g; }
  else if (nm == "mid" && in_range(layer)) { p = e->mid.p; n = (size_t)e->n_local * e->layers[layer].dim_mid; }
  else if (nm == "h" && in_range(layer)) { p = e->h.p; n = (size_t)e->n_local * e->layers[layer].dim_h; }
  else if (nm == "dh" && in_range(layer)) { p = e->dh.p; n = (size_t)e->n_local * e->layers[layer].dim_x; }
  else if (nm == "energy") { p = e->energy.p; n = 1; }
  else if (nm == "virial") { p = e->virial.p; n = 6; }
  else if (nm == "atomic_energy") { p = e->atomic_energy.p; n = (size_t)e->n_local; }
  else if (nm == "atomic_virial" && e->want_atomic_virial) { p = e->atomic_virial.p; n = (size_t)e->n_nodes * 6; }
  else if (nm == "forces") { p = e->forces.p; n = (size_t)e->n_nodes * 3; }
  else if (nm == "edge_force") { p = e->fedge.p; n = (size_t)e->n_edges * 3; }
  else if (nm == "edge_Y") { p = e->Y.p; n = (size_t)e->n_edges * e->ny_stride; }
  else if (nm == "edge_rec") { p = e->rec.p; n = (size_t)e->n_edges * 4; }
  else if (nm == "graph_rowptr") { p = (void*)e->d_rowptr; n = (size_t)e->n_local + 1; }
  else if (nm == "graph_src") { p = (void*)e->d_src; n = (size_t)e->n_edges; }
  else if (nm == "graph_edge_vec") { p = (void*)e->d_edge_vec; n = (size_t)e->n_edges * 3; }
  else if (nm == "nl_rowptr") { p = e->hs_rowptr.p; n = (size_t)e->nl_n_centres + 1; }
  else if (nm == "nl_src") { p = e->hs_src.p; n = (size_t)e->nl_n_edges; }
  else if (nm == "nl_vec") { p = e->hs_vec.p; n = (size_t)e->nl_n_edges * 3; }
  else if (nm == "edge_len") { p = e->rlen.p; n = (size_t)e->n_edges; }
  else if (nm == "edge_emb") { p = e->emb.p; n = (size_t)e->n_edges * e->desc.n_basis; }
  else if (nm == "dY_acc") { p = e->dY_acc.p; n = (size_t)e->n_edges * e->ny_stride; }
  else if (nm == "dEdr_acc") { p = e->dEdr_acc.p; n = (size_t)e->n_edges; }
  if (numel) *numel = n;
  return p;
}

int s7b_engine_compute_host(S7bEngine* e, int32_t n_nodes, int64_t n_edges, const int32_t* species,
                            const int32_t* edge_centre, const int32_t* edge_neighbour,
                            const float* edge_vec, double* energy, float* atomic_energy, float* forces,
                            double* virial, void* stream) {
  if (!e) return fail("null engine");
  if (n_nodes < 0 || n_edges < 0) return fail("bad sizes");
  if (n_nodes > 0 && !species) return fail("null species");
  if (n_edges > 0 && (!edge_centre || !edge_neighbour || !edge_vec)) return fail("null edge arrays");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // H2D of the caller's arrays; the CSR over centres is built (and the edge list validated) on the
  // device.  The caller promises centre-major order, as pair_e3gnn.cpp:136-170 emits.
  const size_t E = (size_t)std::max<int64_t>(n_edges, 1), N = (size_t)std::max(n_nodes, 1);
  if (e->hs_species.ensure(N * sizeof(int)) || e->hs_rowptr.ensure((N + 1) * sizeof(int)) ||
      e->hs_src.ensure(E * sizeof(int)) || e->hs_vec.ensure(E * 3 * sizeof(float)) ||
      e->hs_centre.ensure(E * sizeof(int)) || e->hs_flag.ensure(sizeof(int)))
    return fail("cudaMalloc failed for staging buffers");
  if (n_nodes > 0) S7B_CUDA_CHECK(cudaMemcpyAsync(e->hs_species.p, species, (size_t)n_nodes * sizeof(int), cudaMemcpyHostToDevice, st));
  S7B_CUDA_CHECK(cudaMemsetAsync(e->hs_flag.p, 0, sizeof(int), st));
  if (n_edges > 0) {
    S7B_CUDA_CHECK(cudaMemcpyAsync(e->hs_centre.p, edge_centre, (size_t)n_edges * sizeof(int), cudaMemcpyHostToDevice, st));
    S7B_CUDA_CHECK(cudaMemcpyAsync(e->hs_src.p, edge_neighbour, (size_t)n_edges * sizeof(int), cudaMemcpyHostToDevice, st));
    S7B_CUDA_CHECK(cudaMemcpyAsync(e->hs_vec.p, edge_vec, (size_t)n_edges * 3 * sizeof(float), cudaMemcpyHostToDevice, st));
  }
  {
    const int64_t nthreads = n_edges + 1;
    csr_from_sorted_kernel<<<(int)((nthreads + 255) / 256), 256, 0, st>>>(e->hs_centre.as<int>(), e->hs_src.as<int>(), n_edges, n_nodes, e->hs_rowptr.as<int>(), e->hs_flag.as<int>());
    S7B_LAUNCH_CHECK();
    int flag = 0;
    S7B_CUDA_CHECK(cudaMemcpyAsync(&flag, e->hs_flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    S7B_CUDA_CHECK(cudaStreamSynchronize(st));
    if (flag & 1) return fail("edges must be sorted by centre and centres must be < n_nodes");
    if (flag & 2) return fail("edge neighbour index out of range");
  }
  if (s7b_engine_set_graph(e, n_nodes, n_nodes, n_edges, e->hs_species.as<int>(), e->hs_rowptr.as<int>(), e->hs_src.as<int>(), e->hs_vec.as<float>(), stream)) return 1;
  if (s7b_engine_compute(e, stream)) return 1;
  if (energy) S7B_CUDA_CHECK(cudaMemcpyAsync(energy, e->energy.p, sizeof(double), cudaMemcpyDeviceToHost, st));
  if (virial) S7B_CUDA_CHECK(cudaMemcpyAsync(virial, e->virial.p, 6 * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (atomic_energy && n_nodes > 0) S7B_CUDA_CHECK(cudaMemcpyAsync(atomic_energy, e->atomic_energy.p, (size_t)n_nodes * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (forces && n_nodes > 0) S7B_CUDA_CHECK(cudaMemcpyAsync(forces, e->forces.p, (size_t)n_nodes * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
  S7B_CUDA_CHECK(cudaStreamSynchronize(st));
  return 0;
}

// ---- positions in: device neighbour list + graph build (SURVEY 8(f).1) ------------------------
static int invert3(const double* m, double* inv) {
  const double det = m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * m[7] - m[4] * m[6]);
  if (fabs(det) < 1e-12) return 1;
  const double id = 1.0 / det;
  inv[0] = (m[4] * m[8] - m[5] * m[7]) * id; inv[1] = (m[2] * m[7] - m[1] * m[8]) * id; inv[2] = (m[1] * m[5] - m[2] * m[4]) * id;
  inv[3] = (m[5] * m[6] - m[3] * m[8]) * id; inv[4] = (m[0] * m[8] - m[2] * m[6]) * id; inv[5] = (m[2] * m[3] - m[0] * m[5]) * id;
  inv[6] = (m[3] * m[7] - m[4] * m[6]) * id; inv[7] = (m[1] * m[6] - m[0] * m[7]) * id; inv[8] = (m[0] * m[4] - m[1] * m[3]) * id;
  return 0;
}

// Neighbour list of `n_centres` centre atoms (centres == nullptr: all n_atoms atoms) against all atoms;
// leaves species / rowptr [n_centres + 1] / src (indices into the n_atoms atoms) / edge_vec in the hs_* buffers.
static int build_neighbor_list(S7bEngine* e, int32_t n_atoms, const int32_t* species, const double* positions,
                               const double* cell9, const int32_t* pbc3, int32_t n_centres, const int32_t* centres_host,
                               int64_t* n_edges_out, void* stream) {
  if (!e) return fail("null engine");
  if (n_atoms < 0 || (n_atoms > 0 && (!species || !positions))) return fail("bad arguments");
  if (centres_host == nullptr) n_centres = n_atoms;
  if (n_centres < 0 || n_centres > n_atoms) return fail("bad centre count");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NLGrid g;
  memset(&g, 0, sizeof(g));
  const double cutoff = (double)e->desc.cutoff;
  g.cutoff2 = cutoff * cutoff;
  for (int a = 0; a < 3; ++a) g.pbc[a] = (pbc3 && pbc3[a]) ? 1 : 0;
  for (int k = 0; k < 9; ++k) g.cell[k] = cell9 ? cell9[k] : 0.0;
  for (int a = 0; a < 3; ++a) {      // complete missing lattice vectors of non-periodic directions
    const double* v = g.cell + 3 * a;
    if (v[0] * v[0] + v[1] * v[1] + v[2] * v[2] < 1e-20) {
      if (g.pbc[a]) return fail("periodic direction with a zero lattice vector");
      g.cell[3 * a + a] = 1.0;
    }
  }
  if (invert3(g.cell, g.inv)) return fail("singular cell");
  // plane spacings
  double height[3];
  for (int a = 0; a < 3; ++a) {      // |row a of inv^T| = 1 / height_a
    const double nx = g.inv[0 * 3 + a], ny = g.inv[1 * 3 + a], nz = g.inv[2 * 3 + a];
    height[a] = 1.0 / sqrt(nx * nx + ny * ny + nz * nz);
  }
  // fractional bounding range of non-periodic directions (host pass over the caller's positions)
  for (int a = 0; a < 3; ++a) { g.fmin[a] = 0.0; g.fspan[a] = 1.0; }
  if (!(g.pbc[0] && g.pbc[1] && g.pbc[2]) && n_atoms > 0) {
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    for (int i = 0; i < n_atoms; ++i)
      for (int a = 0; a < 3; ++a) {
        const double f = positions[3 * i] * g.inv[0 * 3 + a] + positions[3 * i + 1] * g.inv[1 * 3 + a] + positions[3 * i + 2] * g.inv[2 * 3 + a];
        lo[a] = std::min(lo[a], f);
        hi[a] = std::max(hi[a], f);
      }
    for (int a = 0; a < 3; ++a)
      if (!g.pbc[a]) { g.fmin[a] = lo[a]; g.fspan[a] = std::max(hi[a] - lo[a], 1e-9) * (1.0 + 1e-9); }
  }
  long long nbins = 1;
  for (int a = 0; a < 3; ++a) {
    const double extent = height[a] * g.fspan[a];
    int nb = (int)floor(extent / cutoff);
    nb = std::max(1, std::min(nb, 512));
    g.nb[a] = nb;
    g.R[a] = g.pbc[a] ? (int)ceil(cutoff / (extent / nb) - 1e-12) : std::min(nb - 1, (int)ceil(cutoff / (extent / nb) - 1e-12));
    if (g.R[a] < 0) g.R[a] = 0;
    nbins *= nb;
  }
  if (nbins > (1LL << 26)) return fail("neighbour grid too large");
  const size_t N = (size_t)std::max(n_atoms, 1);
  int rc = 0;
  rc |= e->hs_species.ensure(N * sizeof(int));
  rc |= e->hs_rowptr.ensure((N + 1) * sizeof(int));
  rc |= e->nl_pos.ensure(N * 3 * sizeof(double));
  rc |= e->nl_wrapped.ensure(N * 3 * sizeof(double));
  rc |= e->nl_key.ensure(N * sizeof(int));
  rc |= e->nl_key_sorted.ensure(N * sizeof(int));
  rc |= e->nl_idx.ensure(N * sizeof(int));
  rc |= e->nl_idx_sorted.ensure(N * sizeof(int));
  rc |= e->nl_bin_start.ensure(((size_t)nbins + 1) * sizeof(int));
  rc |= e->nl_count.ensure((N + 1) * sizeof(int));
  rc |= e->nl_centres.ensure(N * sizeof(int));
  if (rc) return fail("cudaMalloc failed for the neighbour list");
  int64_t n_edges = 0;
  const int* d_centres = nullptr;
  if (centres_host != nullptr && n_centres > 0) {
    S7B_CUDA_CHECK(cudaMemcpyAsync(e->nl_centres.p, centres_host, (size_t)n_centres * sizeof(int), cudaMemcpyHostToDevice, st));
    d_centres = e->nl_centres.as<int>();
  }
  if (n_atoms > 0) {
    S7B_CUDA_CHECK(cudaMemcpyAsync(e->hs_species.p, species, (size_t)n_atoms * sizeof(int), cudaMemcpyHostToDevice, st));
    S7B_CUDA_CHECK(cudaMemcpyAsync(e->nl_pos.p, positions, (size_t)n_atoms * 3 * sizeof(double), cudaMemcpyHostToDevice, st));
    const int blk = 128, grd = (n_atoms + blk - 1) / blk;
    nl_bin_kernel<<<grd, blk, 0, st>>>(g, e->nl_pos.as<double>(), n_atoms, e->nl_key.as<int>(), e->nl_idx.as<int>(), e->nl_wrapped.as<double>());
    S7B_LAUNCH_CHECK();
    size_t tmp_sort = 0, tmp_scan = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp_sort, e->nl_key.as<int>(), e->nl_key_sorted.as<int>(), e->nl_idx.as<int>(), e->nl_idx_sorted.as<int>(), n_atoms, 0, 32, st);
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_scan, e->nl_count.as<int>(), e->hs_rowptr.as<int>(), n_atoms + 1, st);
    if (e->nl_tmp.ensure(std::max(tmp_sort, tmp_scan) + 256)) return fail("cudaMalloc failed for cub workspace");
    size_t tmp = e->nl_tmp.bytes;
    S7B_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(e->nl_tmp.p, tmp, e->nl_key.as<int>(), e->nl_key_sorted.as<int>(), e->nl_idx.as<int>(), e->nl_idx_sorted.as<int>(), n_atoms, 0, 32, st));
    ++g_launches;
    nl_bin_start_kernel<<<(n_atoms + 1 + 255) / 256, 256, 0, st>>>(e->nl_key_sorted.as<int>(), n_atoms, (int)nbins, e->nl_bin_start.as<int>());
    S7B_LAUNCH_CHECK();
    S7B_CUDA_CHECK(cudaMemsetAsync(e->nl_count.p, 0, ((size_t)n_atoms + 1) * sizeof(int), st));
    const int grd_c = std::max(1, (n_centres + blk - 1) / blk);
    nl_pairs_kernel<false><<<grd_c, blk, 0, st>>>(g, e->nl_wrapped.as<double>(), e->nl_key.as<int>(), e->nl_idx_sorted.as<int>(), e->nl_bin_start.as<int>(), n_centres, e->nl_count.as<int>(), nullptr, nullptr, nullptr, d_centres);
    S7B_LAUNCH_CHECK();
    tmp = e->nl_tmp.bytes;
    S7B_CUDA_CHECK(cub::DeviceScan::ExclusiveSum(e->nl_tmp.p, tmp, e->nl_count.as<int>(), e->hs_rowptr.as<int>(), n_centres + 1, st));
    ++g_launches;
    int total = 0;
    S7B_CUDA_CHECK(cudaMemcpyAsync(&total, e->hs_rowptr.as<int>() + n_centres, sizeof(int), cudaMemcpyDeviceToHost, st));
    S7B_CUDA_CHECK(cudaStreamSynchronize(st));
    n_edges = total;
    const size_t E = (size_t)std::max<int64_t>(n_edges, 1);
    if (e->hs_src.ensure(E * sizeof(int)) || e->hs_vec.ensure(E * 3 * sizeof(float))) return fail("cudaMalloc failed for the edge list");
    if (n_edges > 0) {
      nl_pairs_kernel<true><<<grd_c, blk, 0, st>>>(g, e->nl_wrapped.as<double>(), e->nl_key.as<int>(), e->nl_idx_sorted.as<int>(), e->nl_bin_start.as<int>(), n_centres, nullptr, e->hs_rowptr.as<int>(), e->hs_src.as<int>(), e->hs_vec.as<float>(), d_centres);
      S7B_LAUNCH_CHECK();
    }
  } else {
    S7B_CUDA_CHECK(cudaMemsetAsync(e->hs_rowptr.p, 0, sizeof(int), st));
  }
  e->nl_n_centres = n_centres;
  e->nl_n_edges = n_edges;
  if (n_edges_out) *n_edges_out = n_edges;
  return 0;
}

// ---- host-staged pieces of the stage protocol (a LAMMPS pair style without CUDA headers: pair_e3gnn_parallel.cpp
// does the same staging through CPU tensors unless MPI is CUDA-aware, :698-799) -----------------------------------
// Graph with ghosts from host arrays: the upload of s7b_engine_compute_host, but n_local <= n_nodes and no compute.
int s7b_engine_set_graph_host(S7bEngine* e, int32_t n_nodes, int32_t n_local, int64_t n_edges, const int32_t* species,
                              const int32_t* edge_centre, const int32_t* edge_neighbour, const float* edge_vec,
                              void* stream) {
  if (!e) return fail("null engine");
  if (n_nodes < 0 || n_local < 0 || n_local > n_nodes || n_edges < 0) return fail("bad sizes");
  if (n_nodes > 0 && !species) return fail("null species");
  if (n_edges > 0 && (!edge_centre || !edge_neighbour || !edge_vec)) return fail("null edge arrays");
  for (int64_t k = 0; k < n_edges; ++k)
    if (edge_centre[k] < 0 || edge_centre[k] >= n_local) return fail("edge centres must be owned atoms (< n_local)");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const size_t E = (size_t)std::max<int64_t>(n_edges, 1), N = (size_t)std::max(n_nodes, 1);
  if (e->hs_species.ensure(N * sizeof(int)) || e->hs_rowptr.ensure((N + 1) * sizeof(int)) ||
      e->hs_src.ensure(E * sizeof(int)) || e->hs_vec.ensure(E * 3 * sizeof(float)) ||
      e->hs_centre.ensure(E * sizeof(int)) || e->hs_flag.ensure(sizeof(int)))
    return fail("cudaMalloc failed for staging buffers");
  if (n_nodes > 0) S7B_CUDA_CHECK(cudaMemcpyAsync(e->hs_species.p, species, (size_t)n_nodes * sizeof(int), cudaMemcpyHostToDevice, st));
  S7B_CUDA_CHECK(cudaMemsetAsync(e->hs_flag.p, 0, sizeof(int), st));
  if (n_edges > 0) {
    S7B_CUDA_CHECK(cudaMemcpyAsync(e->hs_centre.p, edge_centre, (size_t)n_edges * sizeof(int), cudaMemcpyHostToDevice, st));
    S7B_CUDA_CHECK(cudaMemcpyAsync(e->hs_src.p, edge_neighbour, (size_t)n_edges * sizeof(int), cudaMemcpyHostToDevice, st));
    S7B_CUDA_CHECK(cudaMemcpyAsync(e->hs_vec.p, edge_vec, (size_t)n_edges * 3 * sizeof(float), cudaMemcpyHostToDevice, st));
  }
  // CSR over all n_nodes rows (ghost rows are empty, so its first n_local + 1 entries are the CSR over the owned atoms)
  const int64_t nthreads = n_edges + 1;
  csr_from_sorted_kernel<<<(int)((nthreads + 255) / 256), 256, 0, st>>>(e->hs_centre.as<int>(), e->hs_src.as<int>(), n_edges, n_nodes, e->hs_rowptr.as<int>(), e->hs_flag.as<int>());
  S7B_LAUNCH_CHECK();
  int flag = 0;
  S7B_CUDA_CHECK(cudaMemcpyAsync(&flag, e->hs_flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  S7B_CUDA_CHECK(cudaStreamSynchronize(st));
  if (flag & 1) return fail("edges must be sorted by centre");
  if (flag & 2) return fail("edge neighbour index out of range");
  return s7b_engine_set_graph(e, n_nodes, n_local, n_edges, e->hs_species.as<int>(), e->hs_rowptr.as<int>(), e->hs_src.as<int>(), e->hs_vec.as<float>(), stream);
}

// rows [row_begin, row_begin + n_rows) of a 2-D engine buffer <-> host (fp32 buffers only; synchronous)
static int rows_host_copy(S7bEngine* e, const char* name, int layer, int32_t row_begin, int32_t n_rows, int32_t width,
                          float* host, bool to_host, void* stream) {
  if (!e) return fail("null engine");
  if (n_rows <= 0) return 0;
  if (!host || width <= 0 || row_begin < 0) return fail("bad row range");
  const std::string nm(name ? name : "");
  if (nm == "energy" || nm == "virial") return fail("energy / virial are doubles: read them with s7b_engine_buffer");
  size_t numel = 0;
  float* base = static_cast<float*>(s7b_engine_buffer(e, name, layer, &numel));
  if (!base) return fail(std::string("no such buffer: ") + nm);
  if ((size_t)(row_begin + (int64_t)n_rows) * width > numel) return fail("row range exceeds the buffer");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  float* dev = base + (size_t)row_begin * width;
  const size_t bytes = (size_t)n_rows * width * sizeof(float);
  if (to_host) S7B_CUDA_CHECK(cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, st));
  else S7B_CUDA_CHECK(cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, st));
  S7B_CUDA_CHECK(cudaStreamSynchronize(st));
  return 0;
}

int s7b_engine_read_rows_host(S7bEngine* e, const char* name, int layer, int32_t row_begin, int32_t n_rows, int32_t width,
                              float* host_out, void* stream) {
  return rows_host_copy(e, name, layer, row_begin, n_rows, width, host_out, true, stream);
}

int s7b_engine_write_rows_host(S7bEngine* e, const char* name, int layer, int32_t row_begin, int32_t n_rows, int32_t width,
                               const float* host_in, void* stream) {
  return rows_host_copy(e, name, layer, row_begin, n_rows, width, const_cast<float*>(host_in), false, stream);
}

int s7b_engine_read_scalars_host(S7bEngine* e, double* energy, double* virial6, void* stream) {
  if (!e) return fail("null engine");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (energy) S7B_CUDA_CHECK(cudaMemcpyAsync(energy, e->energy.p, sizeof(double), cudaMemcpyDeviceToHost, st));
  if (virial6) S7B_CUDA_CHECK(cudaMemcpyAsync(virial6, e->virial.p, 6 * sizeof(double), cudaMemcpyDeviceToHost, st));
  S7B_CUDA_CHECK(cudaStreamSynchronize(st));
  return 0;
}


int s7b_engine_set_positions_host(S7bEngine* e, int32_t n_atoms, const int32_t* species, const double* positions,
                                  const double* cell9, const int32_t* pbc3, void* stream) {
  int64_t n_edges = 0;
  if (build_neighbor_list(e, n_atoms, species, positions, cell9, pbc3, n_atoms, nullptr, &n_edges, stream)) return 1;
  return s7b_engine_set_graph(e, n_atoms, n_atoms, n_edges, e->hs_species.as<int>(), e->hs_rowptr.as<int>(), e->hs_src.as<int>(), e->hs_vec.as<float>(), stream);
}

// Multi-GPU front-end (SURVEY 8(f), pair_e3gnn_parallel.cpp:194-340): the rows of a SUBSET of centre atoms
// (a rank's own atoms) against all atoms of the system, built on the device.  Nothing becomes the engine's
// graph; the caller reads "nl_rowptr" [n_centres + 1], "nl_src" [E] (indices into the n_atoms atoms) and
// "nl_vec" [E, 3] with s7b_engine_buffer, maps neighbours to local / ghost rows and calls s7b_engine_set_graph.
int s7b_engine_neighbor_rows_host(S7bEngine* e, int32_t n_atoms, const int32_t* species, const double* positions,
                                  const double* cell9, const int32_t* pbc3, int32_t n_centres, const int32_t* centres,
                                  int64_t* n_edges_out, void* stream) {
  if (!centres && n_centres > 0) return fail("null centre list");
  return build_neighbor_list(e, n_atoms, species, positions, cell9, pbc3, n_centres, centres, n_edges_out, stream);
}

int s7b_engine_compute_positions_host(S7bEngine* e, int32_t n_atoms, const int32_t* species, const double* positions,
                                      const double* cell9, const int32_t* pbc3, double* energy, float* atomic_energy,
                                      float* forces, double* virial, int64_t* n_edges_out, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (s7b_engine_set_positions_host(e, n_atoms, species, positions, cell9, pbc3, stream)) return 1;
  if (n_edges_out) *n_edges_out = e->n_edges;
  if (s7b_engine_compute(e, stream)) return 1;
  if (energy) S7B_CUDA_CHECK(cudaMemcpyAsync(energy, e->energy.p, sizeof(double), cudaMemcpyDeviceToHost, st));
  if (virial) S7B_CUDA_CHECK(cudaMemcpyAsync(virial, e->virial.p, 6 * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (atomic_energy && n_atoms > 0) S7B_CUDA_CHECK(cudaMemcpyAsync(atomic_energy, e->atomic_energy.p, (size_t)n_atoms * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (forces && n_atoms > 0) S7B_CUDA_CHECK(cudaMemcpyAsync(forces, e->forces.p, (size_t)n_atoms * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
  S7B_CUDA_CHECK(cudaStreamSynchronize(st));
  return 0;
}

// ---- operator-level plug-in -----------------------------------------------------------------
int s7b_conv_plan_create(int32_t n_l_x, const int32_t* x_muls, int32_t lmax_filter, int32_t lmax_out,
                         S7bConvPlan** out) {
  if (!x_muls || !out) return fail("null argument");
  if (n_l_x < 1 || n_l_x > S7B_MAX_L || lmax_filter < 1 || lmax_filter > 3 || lmax_out < 0 || lmax_out > 3)
    return fail("irreps out of the supported range (l <= 3)");
  S7bConvPlan* p = new S7bConvPlan();
  int out_muls[kMaxL] = {32, 32, 32, 32};   // only lmax_out matters for the path set
  if (build_layer_cfg(p->cfg, x_muls, n_l_x, out_muls, lmax_out + 1, lmax_filter)) {
    delete p;
    return 1;
  }
  p->lmax_filter = lmax_filter;
  p->ny_stride = (lmax_filter == 3) ? 16 : ((lmax_filter == 2) ? 8 : 4);
  *out = p;
  return 0;
}

void s7b_conv_plan_destroy(S7bConvPlan* p) { delete p; }

int s7b_conv_plan_dims(const S7bConvPlan* p, int32_t* dim_x, int32_t* dim_mid, int32_t* weight_numel,
                       int32_t* n_sh) {
  if (!p) return fail("null plan");
  if (dim_x) *dim_x = p->cfg.dim_x;
  if (dim_mid) *dim_mid = p->cfg.dim_mid;
  if (weight_numel) *weight_numel = p->cfg.W;
  if (n_sh) *n_sh = (p->lmax_filter + 1) * (p->lmax_filter + 1);
  return 0;
}

}  // extern "C"

namespace s7b {

// rec[e] = {src, 0, 0, 0};  Ypk[e, :] = sh[e, 1:]
__global__ void conv_pack_kernel(const int* __restrict__ src, const float* __restrict__ sh, int n_sh,
                                 int ny_stride, int64_t n_edges, int4* __restrict__ rec,
                                 float* __restrict__ Ypk) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_edges) return;
  rec[e] = make_int4(src[e], 0, 0, 0);
  for (int j = 0; j < ny_stride; ++j) Ypk[e * ny_stride + j] = (j + 1 < n_sh) ? sh[e * n_sh + j + 1] : 0.0f;
}

// grad_sh[e, 0] = 0; grad_sh[e, j] = sum_parts dY_acc[part, e, j-1]
__global__ void conv_unpack_grad_kernel(const float* __restrict__ dY_acc, int n_part, int n_sh,
                                        int ny_stride, int64_t n_edges, float* __restrict__ grad_sh) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_edges) return;
  grad_sh[e * n_sh] = 0.0f;
  for (int j = 1; j < n_sh; ++j) {
    float s = 0.0f;
    for (int p = 0; p < n_part; ++p) s += dY_acc[((size_t)p * n_edges + e) * ny_stride + j - 1];
    grad_sh[e * n_sh + j] = s;
  }
}

}  // namespace s7b

extern "C" {

int s7b_conv_forward(const S7bConvPlan* p, const float* x, const float* sh, const float* weight,
                     const int32_t* rowptr, const int32_t* src, int32_t n_nodes, int32_t n_dst,
                     int64_t n_edges, float* out, void* stream) {
  if (!p) return fail("null plan");
  (void)n_nodes;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const LayerCfg& L = p->cfg;
  if (n_dst <= 0) return 0;
  if (n_edges == 0) {   // reference convolution.py:265-268: no launch, zeros out
    S7B_CUDA_CHECK(cudaMemsetAsync(out, 0, (size_t)n_dst * L.dim_mid * sizeof(float), st));
    return 0;
  }
  const int n_sh = (p->lmax_filter + 1) * (p->lmax_filter + 1);
  int4* rec = nullptr;
  float* Ypk = nullptr;
  S7B_CUDA_CHECK(cudaMallocAsync((void**)&rec, (size_t)n_edges * sizeof(int4), st));
  S7B_CUDA_CHECK(cudaMallocAsync((void**)&Ypk, (size_t)n_edges * p->ny_stride * sizeof(float), st));
  conv_pack_kernel<<<(int)((n_edges + 255) / 256), 256, 0, st>>>(src, sh, n_sh, p->ny_stride, n_edges, rec, Ypk);
  S7B_LAUNCH_CHECK();
  ConvArgs a;
  memset(&a, 0, sizeof(a));
  a.rowptr = rowptr;
  a.rec = rec;
  a.Y = Ypk;
  a.x = x;
  a.w = weight;
  a.n_dst = n_dst;
  a.dim_x = L.dim_x;
  a.dim_mid = L.dim_mid;
  a.w_numel = L.W;
  a.ny_stride = p->ny_stride;
  a.inv_h = 1.0f;
  int rc = conv_forward(L, p->lmax_filter, false, a, out, st);
  cudaFreeAsync(rec, st);
  cudaFreeAsync(Ypk, st);
  return rc;
}

int s7b_conv_backward(const S7bConvPlan* p, const float* x, const float* sh, const float* weight,
                      const int32_t* rowptr, const int32_t* src, int32_t n_nodes, int32_t n_dst,
                      int64_t n_edges, const float* grad_out, float* grad_x, float* grad_sh,
                      float* grad_weight, void* stream) {
  if (!p) return fail("null plan");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const LayerCfg& L = p->cfg;
  const int n_sh = (p->lmax_filter + 1) * (p->lmax_filter + 1);
  if (n_nodes > 0) S7B_CUDA_CHECK(cudaMemsetAsync(grad_x, 0, (size_t)n_nodes * L.dim_x * sizeof(float), st));
  if (n_edges == 0 || n_dst <= 0) return 0;
  int4* rec = nullptr;
  float *Ypk = nullptr, *dY = nullptr;
  S7B_CUDA_CHECK(cudaMallocAsync((void**)&rec, (size_t)n_edges * sizeof(int4), st));
  S7B_CUDA_CHECK(cudaMallocAsync((void**)&Ypk, (size_t)n_edges * p->ny_stride * sizeof(float), st));
  S7B_CUDA_CHECK(cudaMallocAsync((void**)&dY, (size_t)L.n_lx * n_edges * p->ny_stride * sizeof(float), st));
  S7B_CUDA_CHECK(cudaMemsetAsync(dY, 0, (size_t)L.n_lx * n_edges * p->ny_stride * sizeof(float), st));
  conv_pack_kernel<<<(int)((n_edges + 255) / 256), 256, 0, st>>>(src, sh, n_sh, p->ny_stride, n_edges, rec, Ypk);
  S7B_LAUNCH_CHECK();
  ConvArgs a;
  memset(&a, 0, sizeof(a));
  a.rowptr = rowptr;
  a.rec = rec;
  a.Y = Ypk;
  a.x = x;
  a.w = weight;
  a.n_dst = n_dst;
  a.dim_x = L.dim_x;
  a.dim_mid = L.dim_mid;
  a.w_numel = L.W;
  a.ny_stride = p->ny_stride;
  a.inv_h = 1.0f;
  int rc = 0;
  for (int l1 = 0; l1 < L.n_lx && !rc; ++l1)
    rc = launch_conv_bwd(l1, p->lmax_filter, L.lmax_out, false, true, a, L.roles[l1], grad_out, grad_x,
                         dY + (size_t)l1 * n_edges * p->ny_stride, nullptr, grad_weight, st);
  if (!rc) {
    conv_unpack_grad_kernel<<<(int)((n_edges + 255) / 256), 256, 0, st>>>(dY, L.n_lx, n_sh, p->ny_stride, n_edges, grad_sh);
    ++g_launches;
    if (cudaGetLastError() != cudaSuccess) rc = fail("conv_unpack_grad_kernel launch failed");
  }
  cudaFreeAsync(rec, st);
  cudaFreeAsync(Ypk, st);
  cudaFreeAsync(dY, st);
  return rc;
}

}  // extern "C"

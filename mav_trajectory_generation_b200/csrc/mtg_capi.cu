// mtg_capi.cu -- the C-ABI (include/mtg_b200.h): handle, host-side constraint layout,
// kernel routing and the pipelined host-buffer entry points.  No CPU compute path exists
// here: every mtg_*_batch_* call launches sm_100a kernels or returns an error.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/mtg_b200.h"
#include "mtg_generic_kernel.cuh"
#include "mtg_twisted_kernel.cuh"
#include "mtg_twisted_tmem_kernel.cuh"
#include "mtg_twisted_tmem_v4_kernel.cuh"
#include "mtg_twisted_chunked_kernel.cuh"
#include "mtg_twisted_tmem_v5_kernel.cuh"
#include "mtg_masked_block_kernel.cuh"
#include "mtg_waypoint_kernel.cuh"

namespace {

thread_local std::string g_create_error;

struct Layout {
  int n_all = 0, n_fixed = 0, n_free = 0, bw = 0;
  bool waypoint = false;
  std::vector<int32_t> slot_col;
  std::vector<int32_t> vcol;  // [(K+1)*h] column of (vertex, derivative)
};

struct CachedTopology {
  std::vector<uint8_t> mask;  // canonical mask
  int N = 0, K = 0;
  Layout layout;
  int32_t* d_slot_col = nullptr;
  int32_t* d_vcol = nullptr;
};

}  // namespace

struct mtg_handle {
  int device = 0;
  int sm_count = 0;
  int cc_major = 0;
  size_t smem_optin = 0;
  std::string error;
  int64_t launches = 0;
  int waypoint_variant = 0;  // MTG_OPT_WAYPOINT_VARIANT
  int ring_depth = 3;        // MTG_OPT_RING_DEPTH (v4 kernel: cp.async input ring buffers, 2..4)
  int early_steps = 0;       // MTG_OPT_EARLY_REFILL (v5, single tile buffer): 0 = on (kV5Early steps of lead), -1 = off
  int v5_static_shape = 0;   // MTG_OPT_V5_STATIC_SHAPE: 0 = on (compile-time-shape v5 kernel where one is built), -1 = off
  int ctas_per_sm = 0;       // MTG_OPT_CTAS_PER_SM (v4 kernel: 0 = as many as fit, 9 = one CTA per tile, not persistent)
  int stagger_us = 0;        // MTG_OPT_STAGGER_US (v4 kernel: CTA start times spread over this many microseconds)
  int tma_inputs = 2;        // MTG_OPT_TMA_INPUTS (default routing prefers the TMA-input kernel v5 when eligible)
  int mellinger_unfused = 0; // MTG_OPT_MELLINGER_UNFUSED (1 = expand + solve + cost kernels, the round-1 path)
  int generic_variant = 0;   // MTG_OPT_GENERIC_VARIANT (0 = masked block kernel, 1 = banded kernel in global scratch)
  int chunk_blocks = 0;      // MTG_OPT_CHUNK_BLOCKS (chunked kernel: resident vertex blocks per lane, 0 = auto)
  int dynamic_tiles = 0;     // MTG_OPT_DYNAMIC_TILES (v4 kernel: warps draw tiles from a global counter)
  std::vector<CachedTopology> topologies;
  // host-pointer pipeline
  static constexpr int kPipe = 3;
  // Scratch arenas are PER PIPELINE SLOT (index kPipe = launches on a caller-supplied stream): two chunks
  // of the host pipeline run concurrently on different streams and must never share band / pack scratch.
  // On the caller-stream slot consecutive users on DIFFERENT streams are ordered with an event.
  struct Arena {
    double* p = nullptr;
    size_t bytes = 0;
    cudaEvent_t ev = nullptr;       // recorded after the last kernel that used the arena
    cudaStream_t last = nullptr;
    bool used = false;
  };
  Arena scratch[kPipe + 1];  // generic kernel: banded factor + right-hand sides
  Arena pack[kPipe + 1];     // times + d_fixed produced by nfabian_pack_kernel; Mellinger expansion
  Arena counters[kPipe + 1]; // dynamic tile counter of the persistent kernels (event-ordered like the scratch arenas: two
                             // launches of one slot on different caller streams must not share a live counter)
  // cached launch plans of the TMEM kernel (per waypoint entry and K): attributes are set once
  struct TmemPlan {
    const void* entry = nullptr;
    int K = 0;
    int cols = 0, ntm = 0, ctas = 0;
    size_t smem = 0;
    bool attr_plain = false, attr_fused = false;
  };
  std::vector<TmemPlan> plans;
  // cudaFuncAttributeMaxDynamicSharedMemorySize is a property of the FUNCTION (shared by every K routed to it):
  // remember the largest value set so far and only ever raise it
  std::vector<std::pair<const void*, size_t>> smem_set;
  std::vector<std::pair<const void*, int>> regs_of;  // cudaFuncGetAttributes().numRegs, queried once per function
  // last encoded tensor map (B = 1 solveLinear() calls re-use the same output buffer)
  struct TmapKey {
    const void* base = nullptr;
    int64_t B = 0;
    int K = 0, D = 0, N = 0;
  } tmap_key;
  CUtensorMap tmap_cached;
  cudaStream_t streams[kPipe] = {nullptr, nullptr, nullptr};
  void* dev_buf[kPipe] = {nullptr, nullptr, nullptr};
  size_t dev_buf_bytes[kPipe] = {0, 0, 0};
};

namespace {

bool set_err(mtg_handle* h, const char* what, cudaError_t e) {
  if (e == cudaSuccess) return false;
  if (h) h->error = std::string(what) + ": " + cudaGetErrorString(e);
  return true;
}

#define MTG_CUDA(h, call)                         \
  do {                                            \
    cudaError_t e__ = (call);                     \
    if (set_err(h, #call, e__)) return MTG_ERR_CUDA; \
  } while (0)

bool valid_problem(const mtg_problem* p) {
  if (!p) return false;
  if (p->N < 2 || p->N > MTG_MAX_N || (p->N & 1)) return false;
  if (p->r < 0 || p->r > p->N / 2 - 1) return false;  // CHECK at linear_impl.h:60
  if (p->K < 1 || p->D < 1) return false;
  return true;
}

std::vector<uint8_t> canonical_mask(const mtg_problem* p) {
  const int h = p->N / 2;
  std::vector<uint8_t> m(size_t(p->K + 1) * h, 0);
  if (p->fixed_mask) {
    for (size_t i = 0; i < m.size(); ++i) m[i] = p->fixed_mask[i] ? 1 : 0;
  } else {
    for (int v = 0; v <= p->K; ++v) {
      m[size_t(v) * h] = 1;
      if (v == 0 || v == p->K)
        for (int k = 1; k < h; ++k) m[size_t(v) * h + k] = 1;
    }
  }
  return m;
}

// The constraint reordering of linear_impl.h:181-260 in O(n): columns are the ranks of
// (vertex, derivative) inside the sorted fixed / free sets (linear.h:287-295); row i*N+s is
// slot s of segment i (s < h: vertex i, s >= h: vertex i+1; interior vertices appear twice,
// :202-205).
void compute_layout(int N, int K, const std::vector<uint8_t>& mask, Layout* L) {
  const int h = N / 2;
  std::vector<int32_t> col(size_t(K + 1) * h);
  int nf = 0, np = 0;
  for (size_t i = 0; i < mask.size(); ++i) (mask[i] ? nf : np)++;
  int cf = 0, cp = 0;
  for (size_t i = 0; i < mask.size(); ++i) col[i] = mask[i] ? cf++ : nf + cp++;
  L->vcol = col;
  L->n_all = K * N;
  L->n_fixed = nf;
  L->n_free = np;
  L->slot_col.resize(size_t(K) * N);
  L->bw = 0;
  for (int i = 0; i < K; ++i) {
    int lo = 1 << 30, hi = -1;
    for (int s = 0; s < N; ++s) {
      const int v = s < h ? i : i + 1, k = s < h ? s : s - h;
      const int c = col[size_t(v) * h + k];
      L->slot_col[size_t(i) * N + s] = c;
      if (c >= nf) { lo = std::min(lo, c); hi = std::max(hi, c); }
    }
    if (hi >= lo) L->bw = std::max(L->bw, hi - lo);
  }
  bool wp = K >= 2;
  for (int v = 0; v <= K && wp; ++v)
    for (int k = 0; k < h; ++k) {
      const bool want = (k == 0) || v == 0 || v == K;
      if ((mask[size_t(v) * h + k] != 0) != want) { wp = false; break; }
    }
  L->waypoint = wp && h >= 2;
}

// ---- waypoint kernel registry ---------------------------------------------------------
typedef void (*WaypointKernel)(const mtg::WaypointParams);
struct WaypointEntry {
  int N, R, D, slots;
  WaypointKernel fn;          // one thread per trajectory
  WaypointKernel fn_twisted;  // two lanes per trajectory (twisted factorisation)
  void (*fn_tmem)(const mtg::WaypointParams, const mtg::TmemLaunch, const CUtensorMap);  // + TMEM state, TMA stores
  int stage_bytes_per_warp;
  void (*fn_tmem_fused)(const mtg::WaypointParams, const mtg::TmemLaunch, const CUtensorMap);  // + fused Nfabian
  void (*fn_chunked)(const mtg::WaypointParams, const mtg::ChunkedLaunch, const CUtensorMap);  // any K (K3)
};
#define MTG_WP(N_, R_, D_)                                                                   \
  {                                                                                          \
    N_, R_, D_, mtg::waypoint_state_slots<N_, D_>(), mtg::waypoint_solve_kernel<N_, R_, D_>, \
        mtg::twisted_solve_kernel<N_, R_, D_>, mtg::twisted_tmem_kernel<N_, R_, D_>,         \
        mtg::tmem_stage_bytes_per_warp<N_, D_>(), mtg::twisted_tmem_kernel<N_, R_, D_, true>, \
        mtg::twisted_chunked_kernel<N_, R_, D_, 3>                                           \
  }
// v1 (thread per trajectory) is kept for the headline shapes only (cross-check / profiles)
#define MTG_WP2(N_, R_, D_)                                                                           \
  {                                                                                                   \
    N_, R_, D_, mtg::waypoint_state_slots<N_, D_>(), nullptr, mtg::twisted_solve_kernel<N_, R_, D_>,  \
        mtg::twisted_tmem_kernel<N_, R_, D_>, mtg::tmem_stage_bytes_per_warp<N_, D_>(),               \
        mtg::twisted_tmem_kernel<N_, R_, D_, true>, mtg::twisted_chunked_kernel<N_, R_, D_, 3>        \
  }
const WaypointEntry kWaypointKernels[] = {
    MTG_WP(10, 4, 3),  MTG_WP(10, 4, 1),  MTG_WP2(10, 4, 2), MTG_WP2(10, 4, 4),   // min snap, N = 10
    MTG_WP(10, 3, 3),  MTG_WP2(10, 3, 1), MTG_WP(10, 2, 3),  MTG_WP2(10, 2, 1),   // jerk / acceleration on N = 10
    MTG_WP(8, 3, 3),   MTG_WP(8, 3, 1),   MTG_WP2(8, 3, 2),  MTG_WP2(8, 3, 4),    // min jerk, N = 8
    MTG_WP(12, 5, 3),  MTG_WP2(12, 5, 1), MTG_WP2(12, 5, 4),                      // N = 12 (feasibility tests)
    MTG_WP2(6, 2, 3),  MTG_WP2(6, 2, 1),                                          // min acceleration, N = 6
};

// ---- cost-only kernels (computeCost of the solution without writing coefficients; Mellinger expansion on the fly)
typedef void (*TmemKernel)(const mtg::WaypointParams, const mtg::TmemLaunch, const CUtensorMap);
struct CostEntry {
  int N, R, D;
  TmemKernel fn;
};
#define MTG_COST(N_, R_, D_) {N_, R_, D_, mtg::twisted_tmem_kernel<N_, R_, D_, false, true>}
const CostEntry kCostKernels[] = {MTG_COST(10, 4, 3), MTG_COST(10, 4, 1), MTG_COST(10, 4, 4), MTG_COST(10, 3, 3),
                                  MTG_COST(10, 2, 3), MTG_COST(8, 3, 3),  MTG_COST(12, 5, 3)};
const CostEntry* find_cost(const mtg_problem* p) {
  for (const auto& e : kCostKernels)
    if (e.N == p->N && e.R == p->r && e.D == p->D) return &e;
  return nullptr;
}

// ---- v4 (persistent, deep input prefetch) kernels: the default for short trajectories (K <= 8), where the per-tile
// prologue of the per-tile kernel is a large share of a tile (profiles/r02_k1_variants.json: C2 +11 %, C4 +18 %;
// at K = 16 the per-tile kernel is 5 % faster and stays the default)
typedef void (*V4Kernel)(const mtg::WaypointParams, const mtg::TmemLaunchV4, const CUtensorMap);
struct V4Entry {
  int N, R, D;
  V4Kernel fn, fn_fused;
};
#define MTG_V4(N_, R_, D_, MB_)                                                                    \
  {                                                                                                \
    N_, R_, D_, mtg::twisted_tmem_v4_kernel<N_, R_, D_, false, 3, MB_>,                           \
        mtg::twisted_tmem_v4_kernel<N_, R_, D_, true, 3, MB_>                                      \
  }
const V4Entry kV4Kernels[] = {MTG_V4(10, 4, 3, 2), MTG_V4(8, 3, 3, 3), MTG_V4(10, 4, 1, 2), MTG_V4(10, 3, 3, 2),
                              MTG_V4(10, 2, 3, 2), MTG_V4(12, 5, 3, 2)};
constexpr int kV4MaxK = 8;

// ---- v5: v4 with the inputs moved by TMA bulk copies (whole 16-trajectory tiles, double buffered); K <= 8
typedef void (*V5Kernel)(const mtg::WaypointParams, const mtg::TmemLaunchV5, const CUtensorMap);
using mtg::kV5Early;
struct V5Entry {
  int N, R, D;
  V5Kernel fn, fn_fused;
  V5Kernel fn_early, fn_fused_early;  // the EARLY = kV5Early instantiations
};
#define MTG_V5(N_, R_, D_, MB_)                                                                                       \
  {N_, R_, D_, mtg::twisted_tmem_v5_kernel<N_, R_, D_, MB_, false>, mtg::twisted_tmem_v5_kernel<N_, R_, D_, MB_, true>, \
   mtg::twisted_tmem_v5_kernel<N_, R_, D_, MB_, false, kV5Early>, mtg::twisted_tmem_v5_kernel<N_, R_, D_, MB_, true, kV5Early>}
const V5Entry kV5Kernels[] = {MTG_V5(10, 4, 3, 2), MTG_V5(8, 3, 3, 3),  MTG_V5(10, 4, 1, 2),
                              MTG_V5(10, 3, 3, 2), MTG_V5(10, 2, 3, 2), MTG_V5(12, 5, 3, 2)};
const V5Entry* find_v5(const mtg_problem* p) {
  for (const auto& e : kV5Kernels)
    if (e.N == p->N && e.R == p->r && e.D == p->D) return &e;
  return nullptr;
}
// compile-time-shape instantiations (KC = K) of the v5 kernel, each built for the layout v5_static_layout() gives it
struct V5StaticEntry {
  int N, R, D, K;
  V5Kernel fn;
  mtg::V5Layout layout;
  int early;
};
#define MTG_V5K(N_, R_, D_, MB_, K_)                                                                               \
  {N_, R_, D_, K_,                                                                                                 \
   mtg::twisted_tmem_v5_kernel<N_, R_, D_, MB_, false,                                                           \
                               mtg::v5_static_layout<N_, D_, MB_, K_>().early_fits ? kV5Early : 0, K_>,          \
   mtg::v5_static_layout<N_, D_, MB_, K_>(), mtg::v5_static_layout<N_, D_, MB_, K_>().early_fits ? kV5Early : 0}
const V5StaticEntry kV5StaticKernels[] = {MTG_V5K(10, 4, 3, 2, 16), MTG_V5K(10, 4, 3, 2, 8), MTG_V5K(8, 3, 3, 3, 4)};
const V5StaticEntry* find_v5_static(const mtg_problem* p) {
  for (const auto& e : kV5StaticKernels)
    if (e.N == p->N && e.R == p->r && e.D == p->D && e.K == p->K) return &e;
  return nullptr;
}

const V4Entry* find_v4(const mtg_problem* p) {
  for (const auto& e : kV4Kernels)
    if (e.N == p->N && e.R == p->r && e.D == p->D) return &e;
  return nullptr;
}

const WaypointEntry* find_waypoint(const mtg_handle* h, const mtg_problem* p, const Layout& L) {
  if (!L.waypoint) return nullptr;
  for (const auto& e : kWaypointKernels)
    if (e.N == p->N && e.R == p->r && e.D == p->D) return &e;  // any K: the chunked kernel has a fixed footprint
  (void)h;
  return nullptr;
}

int route(const mtg_handle* h, const mtg_problem* p, const Layout& L) {
  if (L.n_free == 0) return MTG_KERNEL_NOFREE;
  if (find_waypoint(h, p, L)) return MTG_KERNEL_WAYPOINT;
  return MTG_KERNEL_GENERIC;
}

CachedTopology* get_topology(mtg_handle* h, const mtg_problem* p) {
  std::vector<uint8_t> mask = canonical_mask(p);
  for (auto& t : h->topologies)
    if (t.N == p->N && t.K == p->K && t.mask == mask) return &t;
  CachedTopology t;
  t.N = p->N;
  t.K = p->K;
  t.mask = mask;
  compute_layout(p->N, p->K, mask, &t.layout);
  if (set_err(h, "cudaMalloc(slot_col)", cudaMalloc(&t.d_slot_col, sizeof(int32_t) * t.layout.slot_col.size())))
    return nullptr;
  if (set_err(h, "cudaMemcpy(slot_col)",
              cudaMemcpy(t.d_slot_col, t.layout.slot_col.data(), sizeof(int32_t) * t.layout.slot_col.size(),
                         cudaMemcpyHostToDevice)))
    return nullptr;
  if (set_err(h, "cudaMalloc(vcol)", cudaMalloc(&t.d_vcol, sizeof(int32_t) * t.layout.vcol.size()))) return nullptr;
  if (set_err(h, "cudaMemcpy(vcol)", cudaMemcpy(t.d_vcol, t.layout.vcol.data(), sizeof(int32_t) * t.layout.vcol.size(),
                                                cudaMemcpyHostToDevice)))
    return nullptr;
  if (h->topologies.size() >= 64) {  // bound the cache
    cudaFree(h->topologies.front().d_vcol);
    cudaFree(h->topologies.front().d_slot_col);
    h->topologies.erase(h->topologies.begin());
  }
  h->topologies.push_back(std::move(t));
  return &h->topologies.back();
}

// Grow-only arena.  acquire(): make the arena usable by a kernel about to be launched on `stream` (orders it
// after the previous user when that one ran on another stream); release(): note the new last user.
int arena_acquire(mtg_handle* h, mtg_handle::Arena& a, size_t bytes, cudaStream_t stream) {
  if (bytes > a.bytes) {
    if (a.p) {
      MTG_CUDA(h, cudaDeviceSynchronize());
      cudaFree(a.p);
      a.p = nullptr;
      a.bytes = 0;
    }
    MTG_CUDA(h, cudaMalloc(&a.p, bytes));
    a.bytes = bytes;
    a.used = false;
  }
  if (a.used && a.last != stream) MTG_CUDA(h, cudaStreamWaitEvent(stream, a.ev, 0));
  return MTG_OK;
}
int arena_release(mtg_handle* h, mtg_handle::Arena& a, cudaStream_t stream) {
  if (!a.ev) MTG_CUDA(h, cudaEventCreateWithFlags(&a.ev, cudaEventDisableTiming));
  MTG_CUDA(h, cudaEventRecord(a.ev, stream));
  a.last = stream;
  a.used = true;
  return MTG_OK;
}

// zeroed dynamic-tile counter of pipeline slot `slot`, ordered after the previous launch that used it
int tile_counter_acquire(mtg_handle* h, int slot, cudaStream_t stream, unsigned long long** out) {
  mtg_handle::Arena& a = h->counters[slot];
  const int rc = arena_acquire(h, a, 256, stream);
  if (rc != MTG_OK) return rc;
  *out = reinterpret_cast<unsigned long long*>(a.p);
  MTG_CUDA(h, cudaMemsetAsync(*out, 0, sizeof(unsigned long long), stream));
  return MTG_OK;
}

// Make sure `fn` may be launched with `bytes` of dynamic shared memory (raises the function attribute when needed).
int ensure_dyn_smem(mtg_handle* h, const void* fn, size_t bytes) {
  for (auto& kv : h->smem_set)
    if (kv.first == fn) {
      if (kv.second >= bytes) return MTG_OK;
      MTG_CUDA(h, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
      kv.second = bytes;
      return MTG_OK;
    }
  MTG_CUDA(h, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  h->smem_set.emplace_back(fn, bytes);
  return MTG_OK;
}

// registers per thread of a kernel (cached: a B = 1 solveLinear() call must not pay an attribute query)
int kernel_regs(mtg_handle* h, const void* fn, int* out) {
  for (auto& kv : h->regs_of)
    if (kv.first == fn) {
      *out = kv.second;
      return MTG_OK;
    }
  cudaFuncAttributes attr;
  MTG_CUDA(h, cudaFuncGetAttributes(&attr, fn));
  h->regs_of.emplace_back(fn, attr.numRegs);
  *out = attr.numRegs;
  return MTG_OK;
}

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

// coeffs as a 2-D fp64 tensor [B][K*D*N] for the TMA stores (box = 16 trajectories x one segment)
int encode_coeff_tmap(mtg_handle* h, CUtensorMap* out, double* coeffs, int64_t B, const mtg_problem* p,
                      int box_inner = 0) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                               const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                               CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  // function-local static with a lambda initialiser: initialised exactly once, thread-safe (C++11)
  static const EncodeFn encode = []() -> EncodeFn {
    void* fp = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fp, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return nullptr;
    return reinterpret_cast<EncodeFn>(fp);
  }();
  if (!encode) {
    h->error = "cuTensorMapEncodeTiled is not available from the driver";
    return MTG_ERR_CUDA;
  }
  const cuuint64_t row = cuuint64_t(p->K) * p->D * p->N;
  const cuuint64_t dims[2] = {row, cuuint64_t(B)};
  const cuuint64_t strides[1] = {row * sizeof(double)};
  const cuuint32_t box[2] = {cuuint32_t(box_inner > 0 ? box_inner : p->D * p->N), 16u};
  const cuuint32_t estr[2] = {1u, 1u};
  const CUresult cr = encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, coeffs, dims, strides, box, estr,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                             CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) {
    h->error = "cuTensorMapEncodeTiled failed (" + std::to_string(int(cr)) + ")";
    return MTG_ERR_CUDA;
  }
  return MTG_OK;
}

struct FusedInput {
  const double* positions;
  double v_max, a_max, magic;
  double* times_out;
};

// K3: the chunked (checkpoint + recompute) twisted kernel -- any K, fixed on-chip footprint.
int launch_chunked(mtg_handle* h, const mtg_problem* p, const WaypointEntry* e, const mtg::WaypointParams& prm,
                   double* coeffs, int64_t B, cudaStream_t stream, int slot) {
  const int hh = p->N / 2, mm = hh - 1, D = p->D, rd = 3;
  const int kslots = mm * (mm + 1) / 2 + mm * D + D, kck = mm * mm + mm * D;
  const int nmax = (p->K + 1) / 2 - 1;
  int n_regs = 0;
  {
    const int rc_regs = kernel_regs(h, (const void*)e->fn_chunked, &n_regs);
    if (rc_regs != MTG_OK) return rc_regs;
  }
  const int by_regs = std::max(1, 65536 / (std::max(n_regs, 1) * mtg::kTmemThreads));
  auto smem_of = [&](int C, int ntm) {
    return size_t(mtg::kTmemHeaderBytes) + size_t(4) * e->stage_bytes_per_warp +
           size_t(rd * (1 + D) + (C + 1) + (D + 1) + (1 + 2 * D) + (C - ntm) * kslots) * mtg::kTmemThreads * 8;
  };
  int best_ctas = 0, best_C = 0, best_cols = 0, best_ntm = 0;
  size_t best_smem = 0;
  const int cmax = std::max(1, std::min(nmax, 24));
  const int col_options[] = {256, 512, 128, 64, 0};
  for (int cols : col_options)
    for (int C = cmax; C >= 1; --C) {
      if (h->chunk_blocks > 0 && C != std::min(h->chunk_blocks, cmax)) continue;
      const int ntm = cols ? std::min(C, cols / (2 * kslots)) : 0;
      const size_t smem = smem_of(C, ntm);
      if (smem > h->smem_optin) continue;
      int ctas = std::min<int>(by_regs, int((228 * 1024) / (smem + 1024)));
      if (cols) ctas = std::min(ctas, 512 / cols);
      ctas = std::min(ctas, 8);
      // More resident CTAs first.  Then: when the sweep needs several rounds anyway, the chunk that fits tensor memory
      // entirely (no shared-memory blocks: 60 KB per CTA instead of 114 KB leaves ~100 KB of L1 for the re-read
      // inputs and checkpoints -- measured at K = 50: 0.376 of the HBM roofline with C = 4 vs 0.255 with C = 7);
      // a single round (C >= nmax) always wins over recomputation.
      const bool single = C >= nmax, best_single = best_C >= nmax && best_C > 0;
      const bool all_tmem = ntm == C, best_all_tmem = best_ntm == best_C;
      bool better = ctas > best_ctas;
      if (ctas == best_ctas && ctas > 0) {
        if (single != best_single) better = single;
        else if (!single && all_tmem != best_all_tmem) better = all_tmem;
        else better = C > best_C;
      }
      if (better) {
        best_ctas = ctas;
        best_C = C;
        best_cols = cols;
        best_ntm = ntm;
        best_smem = smem;
      }
    }
  if (best_ctas == 0) {
    h->error = "chunked kernel: no launch configuration fits";
    return MTG_ERR_ALLOC;
  }
  const int64_t ctiles = (B + 63) / 64;
  const int64_t blocks = std::min<int64_t>(ctiles, int64_t(best_ctas) * h->sm_count);
  const int nc = nmax > 0 ? (nmax + best_C - 1) / best_C : 1;
  mtg::ChunkedLaunch cl;
  cl.chunk = best_C;
  cl.n_tmem_blocks = best_ntm;
  cl.tmem_cols = best_cols;
  cl.ckpt = nullptr;
  mtg_handle::Arena& ar = h->scratch[slot];
  if (nc > 1) {
    const size_t bytes = size_t(nc - 1) * kck * size_t(blocks) * mtg::kTmemThreads * sizeof(double);
    const int rc = arena_acquire(h, ar, bytes, stream);
    if (rc != MTG_OK) return rc;
    cl.ckpt = ar.p;
  }
  {
        const int rc_smem = ensure_dyn_smem(h, (const void*)e->fn_chunked, size_t(best_smem));
        if (rc_smem != MTG_OK) return rc_smem;
      }
  CUtensorMap tmap;
  {
    const int rc = encode_coeff_tmap(h, &tmap, coeffs, B, p);
    if (rc != MTG_OK) return rc;
  }
  e->fn_chunked<<<(unsigned)blocks, mtg::kTmemThreads, best_smem, stream>>>(prm, cl, tmap);
  MTG_CUDA(h, cudaGetLastError());
  h->launches++;
  if (nc > 1) return arena_release(h, ar, stream);
  return MTG_OK;
}

// ---- K4: masked block-tridiagonal kernel, any mask; N in {2..12}, dimension groups of 1..4
typedef void (*MaskedKernel)(const mtg::MaskedParams, const CUtensorMap);
#define MTG_MASKED_ROW(N_)                                                                                  \
  {                                                                                                         \
    mtg::masked_block_kernel<N_, 1>, mtg::masked_block_kernel<N_, 2>, mtg::masked_block_kernel<N_, 3>,     \
        mtg::masked_block_kernel<N_, 4>                                                                     \
  }
const MaskedKernel kMaskedKernels[6][4] = {MTG_MASKED_ROW(2), MTG_MASKED_ROW(4),  MTG_MASKED_ROW(6),
                                           MTG_MASKED_ROW(8), MTG_MASKED_ROW(10), MTG_MASKED_ROW(12)};

int launch_masked(mtg_handle* h, const mtg_problem* p, CachedTopology* topo, int64_t B, const double* times,
                  const double* dfix, double* coeffs, double* dfree, int32_t* status, cudaStream_t stream, int slot) {
  const Layout& L = topo->layout;
  const int hh = p->N / 2;
  mtg::MaskedParams prm;
  prm.N = p->N;
  prm.r = p->r;
  prm.K = p->K;
  prm.D = p->D;
  prm.n_fixed = L.n_fixed;
  prm.n_free = L.n_free;
  prm.B = B;
  prm.vcol = topo->d_vcol;
  prm.times = times;
  prm.dfix = dfix;
  prm.coeffs = coeffs;
  prm.dfree = dfree;
  prm.status = status;
  mtg_handle::Arena& ar = h->scratch[slot];
  for (int d0 = 0; d0 < p->D;) {
    const int rem = p->D - d0;
    const int dg = rem > 4 ? (rem == 5 ? 3 : 4) : rem;  // 5 = 3 + 2 rather than 4 + 1
    MaskedKernel fn = kMaskedKernels[p->N / 2 - 1][dg - 1];
    const int kslots = hh * (hh + 1) / 2 + hh * dg;
    const size_t smem = size_t(4) * 32 * dg * p->N * sizeof(double);  // staging tiles of the four warps
    {
        const int rc_smem = ensure_dyn_smem(h, (const void*)fn, size_t(smem));
        if (rc_smem != MTG_OK) return rc_smem;
      }
    int per_sm = 0;
    MTG_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)fn, 128, smem));
    per_sm = std::max(per_sm, 1);
    const int64_t blocks = std::min<int64_t>((B + 127) / 128, int64_t(per_sm) * h->sm_count);
    const size_t bytes = size_t(p->K + 1) * kslots * size_t(blocks) * 128 * sizeof(double);
    int rc = arena_acquire(h, ar, bytes, stream);
    if (rc != MTG_OK) return rc;
    prm.lifo = ar.p;
    prm.d0 = d0;
    CUtensorMap tmap;
    rc = encode_coeff_tmap(h, &tmap, coeffs, B, p, dg * p->N);
    if (rc != MTG_OK) return rc;
    fn<<<(unsigned)blocks, 128, smem, stream>>>(prm, tmap);
    MTG_CUDA(h, cudaGetLastError());
    h->launches++;
    rc = arena_release(h, ar, stream);
    if (rc != MTG_OK) return rc;
    d0 += dg;
  }
  return MTG_OK;
}

// Fused cost-only solve (SURVEY.md 8f-2): nx problems -> cost_x[nx].  With mel_k1 > 0 the nx = B * mel_k1 problems
// are the Mellinger expansion of the B trajectories in (times, dfix), generated inside the kernel.
// Returns MTG_ERR_ALLOC when no fused kernel / launch configuration exists (caller falls back).
int launch_cost_fused(mtg_handle* h, const mtg_problem* p, CachedTopology* topo, int64_t nx, const double* times,
                      const double* dfix, double* cost_x, int mel_k1, double inc, double lower, cudaStream_t stream) {
  const Layout& L = topo->layout;
  const CostEntry* ce = find_cost(p);
  const WaypointEntry* e = L.waypoint ? find_waypoint(h, p, L) : nullptr;
  if (!ce || !e || L.n_free == 0) return MTG_ERR_ALLOC;
  const int nmax = (p->K + 1) / 2 - 1;
  int n_regs = 0;
  {
    const int rc_regs = kernel_regs(h, (const void*)ce->fn, &n_regs);
    if (rc_regs != MTG_OK) return rc_regs;
  }
  const int by_regs = std::max(1, 65536 / (std::max(n_regs, 1) * mtg::kTmemThreads));
  int best_ctas = 0, best_cols = 0, best_ntm = 0;
  size_t best_smem = 0;
  const int col_options[] = {512, 256, 128, 64, 32, 0};
  for (int cols : col_options) {
    const int tslots = e->slots + e->D;
    const int ntm = cols ? std::min(nmax, cols / (2 * tslots)) : 0;
    if (cols && ntm == 0) continue;
    const size_t smem = mtg::kTmemHeaderBytes + size_t(4) * e->stage_bytes_per_warp +
                        size_t(2) * (1 + p->D) * mtg::kTmemThreads * 8 + size_t(nmax + 1) * mtg::kTmemThreads * 8 +
                        size_t(nmax - ntm) * tslots * mtg::kTmemThreads * sizeof(double);
    if (smem > h->smem_optin) continue;
    int ctas = std::min<int>(by_regs, int((228 * 1024) / (smem + 1024)));
    ctas = std::min(ctas, 16);
    if (cols) ctas = std::min(ctas, 512 / cols);
    if (ctas > best_ctas || (ctas == best_ctas && smem < best_smem)) {
      best_ctas = ctas;
      best_cols = cols;
      best_ntm = ntm;
      best_smem = smem;
    }
  }
  if (best_ctas < 2) return MTG_ERR_ALLOC;  // large K: unfused path (chunked kernel + cost kernel)
  mtg::WaypointParams prm;
  prm.K = p->K;
  prm.n_fixed = L.n_fixed;
  prm.B = nx;
  prm.times = times;
  prm.dfix = dfix;
  prm.coeffs = nullptr;
  prm.dfree = nullptr;
  prm.status = nullptr;
  prm.positions = nullptr;
  prm.v_max = prm.a_max = prm.magic = 0.0;
  prm.times_out = nullptr;
  prm.cost = cost_x;
  prm.mel_k1 = mel_k1;
  prm.mel_inc = inc;
  prm.mel_lower = lower;
  mtg::TmemLaunch tl;
  tl.n_tmem_blocks = best_ntm;
  tl.tmem_cols = best_cols;
  {
        const int rc_smem = ensure_dyn_smem(h, (const void*)ce->fn, size_t(best_smem));
        if (rc_smem != MTG_OK) return rc_smem;
      }
  CUtensorMap tmap;
  std::memset(&tmap, 0, sizeof(tmap));  // unused by the cost-only instantiation
  ce->fn<<<(unsigned)((nx + 63) / 64), mtg::kTmemThreads, best_smem, stream>>>(prm, tl, tmap);
  MTG_CUDA(h, cudaGetLastError());
  h->launches++;
  return MTG_OK;
}

int launch_solve(mtg_handle* h, const mtg_problem* p, CachedTopology* topo, int64_t B, const double* times,
                 const double* dfix, const double* dfree_in, double* coeffs, double* dfree, int32_t* status,
                 cudaStream_t stream, bool backsub_only, const FusedInput* fused = nullptr,
                 int slot = mtg_handle::kPipe) {
  const Layout& L = topo->layout;
  if (B == 0) return MTG_OK;
  // clear a stale (non-sticky) error another library of the process may have left behind: the
  // cudaGetLastError() after our launches must report OUR launch only
  (void)cudaGetLastError();
  int kind = backsub_only ? MTG_KERNEL_NOFREE : route(h, p, L);
  // Every specialised kernel stores coefficients in 16-byte units (TMA tensor stores / double2): an output that
  // is only 8-byte aligned (e.g. a tensor slice) takes the banded generic kernel, which stores scalar doubles.
  const bool out_aligned = (reinterpret_cast<uintptr_t>(coeffs) & 15u) == 0;
  if (kind == MTG_KERNEL_WAYPOINT && !fused && !out_aligned) kind = MTG_KERNEL_GENERIC;
  if (kind == MTG_KERNEL_WAYPOINT) {
    const WaypointEntry* e = find_waypoint(h, p, L);
    mtg::WaypointParams prm;
    prm.K = p->K;
    prm.n_fixed = L.n_fixed;
    prm.B = B;
    prm.times = times;
    prm.dfix = dfix;
    prm.coeffs = coeffs;
    prm.dfree = dfree;
    prm.status = status;
    prm.positions = fused ? fused->positions : nullptr;
    prm.v_max = fused ? fused->v_max : 0.0;
    prm.a_max = fused ? fused->a_max : 0.0;
    prm.magic = fused ? fused->magic : 0.0;
    prm.times_out = fused ? fused->times_out : nullptr;
    prm.cost = nullptr;
    prm.mel_k1 = 0;
    prm.mel_inc = prm.mel_lower = 0.0;
    const size_t smem_v1 = size_t(p->K - 1) * e->slots * 32 * sizeof(double);
    const bool use_v1 = h->waypoint_variant == 1 && e->fn != nullptr && smem_v1 <= h->smem_optin;
    // The TMA tensor stores need a 16-byte aligned output (cuTensorMapEncodeTiled); an 8-byte aligned
    // caller buffer (e.g. a tensor slice) takes the shared-memory twisted kernel instead of failing.
    const bool coeffs_aligned = (reinterpret_cast<uintptr_t>(coeffs) & 15u) == 0;
    if (h->waypoint_variant == 5 && coeffs_aligned && !fused)
      return launch_chunked(h, p, e, prm, coeffs, B, stream, slot);
    const bool v5_eligible =
        coeffs_aligned && (B % 16) == 0 &&
        (fused ? (reinterpret_cast<uintptr_t>(fused->positions) & 15u) == 0
               : ((reinterpret_cast<uintptr_t>(times) | reinterpret_cast<uintptr_t>(dfix)) & 15u) == 0);
    if ((h->waypoint_variant == 6 || (h->waypoint_variant == 0 && h->tma_inputs)) && v5_eligible) {
      const V5Entry* e5 = find_v5(p);
      if (e5) {
        const V5Kernel fn5 = fused ? e5->fn_fused : e5->fn;
        int n_regs = 0;
        {
          const int rc_regs = kernel_regs(h, (const void*)fn5, &n_regs);
          if (rc_regs != MTG_OK) return rc_regs;
        }
        const int by_regs = std::max(1, 65536 / (std::max(n_regs, 1) * mtg::kTmemThreads));
        const mtg::V5Layout lay = mtg::v5_layout(p->N, p->D, p->K, L.n_fixed, fused != nullptr, h->smem_optin, by_regs);
        const int best_ctas = lay.ctas, best_cols = lay.cols, best_nbuf = lay.nbuf;
        const size_t best_smem = lay.smem;
        const bool take = best_ctas >= 2 && (h->waypoint_variant == 6 || best_nbuf == 2 || h->tma_inputs == 2);
        if (take) {
          mtg::TmemLaunchV5 tl;
          tl.tmem_slots = best_cols / 2;
          tl.tmem_cols = best_cols;
          tl.n_buffers = best_nbuf;
          tl.tile_counter = nullptr;
          V5Kernel launch_fn = fn5;
          int early = 0;
          if (h->early_steps >= 0 && lay.early_fits) {  // early refill of the single tile buffer (EARLY instantiation)
            const V5Kernel fe = fused ? e5->fn_fused_early : e5->fn_early;
            if (fe != nullptr) {
              int regs_e = 0;
              const int rc_regs = kernel_regs(h, (const void*)fe, &regs_e);
              if (rc_regs != MTG_OK) return rc_regs;
              if (65536 / (std::max(regs_e, 1) * mtg::kTmemThreads) >= best_ctas) {
                launch_fn = fe;
                early = kV5Early;
              }
            }
          }
          // the compile-time-shape instantiation of this K, when it was built for exactly this layout
          const V5StaticEntry* es = (h->v5_static_shape >= 0 && !fused) ? find_v5_static(p) : nullptr;
          if (es != nullptr && es->layout.cols == best_cols && es->layout.nbuf == best_nbuf && es->early == early &&
              L.n_fixed == p->K + p->N - 1) {
            int regs_s = 0;
            const int rc_regs = kernel_regs(h, (const void*)es->fn, &regs_s);
            if (rc_regs != MTG_OK) return rc_regs;
            if (65536 / (std::max(regs_s, 1) * mtg::kTmemThreads) >= best_ctas) launch_fn = es->fn;
          }
          const int64_t blocks = std::min<int64_t>((B + 63) / 64, int64_t(best_ctas) * h->sm_count);
          // dynamic tile counter for long tiles with several tiles per warp (balances the tail: C3 0.618 vs 0.605,
          // C5 on one GPU 0.655 vs 0.630); static round-robin for short trajectories, where the atomic's round trip is
          // not small against a tile (C2 0.581 vs 0.529, C4 0.812 vs 0.797)  [profiles/r02_k1_variants.json]
          const int64_t tiles_per_warp = (B / 16) / std::max<int64_t>(1, blocks * 4);
          if (h->dynamic_tiles == 1 || (h->dynamic_tiles == 0 && tiles_per_warp >= 8 && p->K > kV4MaxK)) {
            const int rc_ctr = tile_counter_acquire(h, slot, stream, &tl.tile_counter);
            if (rc_ctr != MTG_OK) return rc_ctr;
          }
          {
            const int rc_smem = ensure_dyn_smem(h, (const void*)launch_fn, best_smem);
            if (rc_smem != MTG_OK) return rc_smem;
          }
          CUtensorMap tmap;
          {
            const int rc = encode_coeff_tmap(h, &tmap, coeffs, B, p);
            if (rc != MTG_OK) return rc;
          }
          launch_fn<<<(unsigned)blocks, mtg::kTmemThreads, best_smem, stream>>>(prm, tl, tmap);
          MTG_CUDA(h, cudaGetLastError());
          h->launches++;
          if (tl.tile_counter != nullptr) return arena_release(h, h->counters[slot], stream);
          return MTG_OK;
        }
      }
    }
    if ((h->waypoint_variant == 4 || (h->waypoint_variant == 0 && p->K <= kV4MaxK)) && coeffs_aligned) {
      const V4Entry* e4 = find_v4(p);
      if (e4) {
        V4Kernel fn = fused ? e4->fn_fused : e4->fn;
        const int rd = 3;
        const int hh = p->N / 2, mm = hh - 1;
        const int kslots = mm * (mm + 1) / 2 + mm * p->D + p->D, kpro = 2 * p->D + mm * p->D + 1;
        const int nmax = (p->K + 1) / 2 - 1;
        int n_regs = 0;
        {
          const int rc_regs = kernel_regs(h, (const void*)fn, &n_regs);
          if (rc_regs != MTG_OK) return rc_regs;
        }
        const int by_regs = std::max(1, 65536 / (std::max(n_regs, 1) * mtg::kTmemThreads));
        int best_ctas = 0, best_cols = 0, best_ntm = 0;
        size_t best_smem = 0;
        const int col_options[] = {512, 256, 128, 64, 32, 0};
        for (int cols : col_options) {
          const int ntm = cols ? std::min(nmax, cols / (2 * kslots)) : 0;
          if (cols && ntm == 0 && nmax > 0) continue;
          const int spill = std::max(0, nmax - ntm) * kslots;
          const size_t smem = mtg::kTmemHeaderBytes + size_t(4) * e->stage_bytes_per_warp +
                              size_t(rd * (1 + p->D) + (nmax + 1) + p->D + std::max(spill, kpro)) * mtg::kTmemThreads * 8;
          if (smem > h->smem_optin) continue;
          int ctas = std::min<int>(by_regs, int((228 * 1024) / (smem + 1024)));
          if (cols) ctas = std::min(ctas, 512 / cols);
          ctas = std::min(ctas, 8);
          if (ctas > best_ctas || (ctas == best_ctas && smem < best_smem)) {
            best_ctas = ctas;
            best_cols = cols;
            best_ntm = ntm;
            best_smem = smem;
          }
        }
        if (best_ctas > 0) {
          const bool per_tile = h->ctas_per_sm == 9;
          if (h->ctas_per_sm > 0 && !per_tile) best_ctas = std::min(best_ctas, h->ctas_per_sm);
          mtg::TmemLaunchV4 tl;
          tl.n_tmem_blocks = best_ntm;
          tl.tmem_cols = best_cols;
          tl.region_slots = 0;
          tl.tile_counter = nullptr;
          // dynamic tile counter when every warp has many tiles to draw (balances the tail); static round-robin for
          // small batches, where the first draw's round trip to L2 is not amortised (measured: C2 static, C4 dynamic)
          const int64_t tiles_per_warp = ((B + 15) / 16) / std::max<int64_t>(1, int64_t(best_ctas) * h->sm_count * 4);
          const bool dyn = h->dynamic_tiles == 1 || (h->dynamic_tiles == 0 && tiles_per_warp >= 16);
          if (dyn && !per_tile) {
            const int rc_ctr = tile_counter_acquire(h, slot, stream, &tl.tile_counter);
            if (rc_ctr != MTG_OK) return rc_ctr;
          }
          {
        const int rc_smem = ensure_dyn_smem(h, (const void*)fn, size_t(best_smem));
        if (rc_smem != MTG_OK) return rc_smem;
      }
          CUtensorMap tmap;
          {
            const int rc = encode_coeff_tmap(h, &tmap, coeffs, B, p);
            if (rc != MTG_OK) return rc;
          }
          const int64_t ctiles = (B + 63) / 64;
          const int64_t blocks = per_tile ? ctiles : std::min<int64_t>(ctiles, int64_t(best_ctas) * h->sm_count);
          fn<<<(unsigned)blocks, mtg::kTmemThreads, best_smem, stream>>>(prm, tl, tmap);
          MTG_CUDA(h, cudaGetLastError());
          h->launches++;
          if (tl.tile_counter != nullptr) return arena_release(h, h->counters[slot], stream);
          return MTG_OK;
        }
      }
    }
    const bool twisted_fits = size_t((p->K + 1) / 2 - 1) * e->slots * 32 * sizeof(double) <= h->smem_optin;
    const bool want_default = h->waypoint_variant == 0 || h->waypoint_variant >= 3 || fused ||
                              (h->waypoint_variant == 2 && !twisted_fits) || (h->waypoint_variant == 1 && !use_v1 && !twisted_fits);
    if (want_default && (coeffs_aligned || fused)) {
      if (!coeffs_aligned) return MTG_ERR_ALLOC;  // fused entry: caller falls back to pack + solve
      const int nmax = (p->K + 1) / 2 - 1;
      // ---- launch plan (TMEM column count / spill split maximising resident CTAs per SM): computed and
      // the function attributes set ONCE per (kernel, K); a B = 1 solveLinear() call pays none of it again.
      mtg_handle::TmemPlan* plan = nullptr;
      for (auto& pl : h->plans)
        if (pl.entry == (const void*)e && pl.K == p->K) plan = &pl;
      if (!plan) {
        int n_regs = 0;
        {
          const int rc_regs = kernel_regs(h, (const void*)e->fn_tmem, &n_regs);
          if (rc_regs != MTG_OK) return rc_regs;
        }
        const int by_regs = std::max(1, 65536 / (std::max(n_regs, 1) * mtg::kTmemThreads));
        mtg_handle::TmemPlan np;
        np.entry = (const void*)e;
        np.K = p->K;
        const int col_options[] = {512, 256, 128, 64, 32, 0};
        for (int cols : col_options) {
          const int tslots = e->slots + e->D;  // TMEM kernel also keeps the vertex position in the state block
          const int ntm = cols ? std::min(nmax, cols / (2 * tslots)) : 0;
          if (cols && ntm == 0) continue;
          const size_t smem = mtg::kTmemHeaderBytes + size_t(4) * e->stage_bytes_per_warp +
                              size_t(2) * (1 + p->D) * mtg::kTmemThreads * 8 + size_t(nmax + 1) * mtg::kTmemThreads * 8 +
                              size_t(nmax - ntm) * tslots * mtg::kTmemThreads * sizeof(double);
          if (smem > h->smem_optin) continue;
          int ctas = std::min<int>(by_regs, int((228 * 1024) / (smem + 1024)));
          ctas = std::min(ctas, 16);
          if (cols) ctas = std::min(ctas, 512 / cols);
          if (ctas > np.ctas || (ctas == np.ctas && smem < np.smem)) {
            np.ctas = ctas;
            np.cols = cols;
            np.ntm = ntm;
            np.smem = smem;
          }
        }
        h->plans.push_back(np);
        plan = &h->plans.back();
      }
      if (plan->ctas < 2 && fused) return MTG_ERR_ALLOC;  // caller falls back to pack + solve
      if (plan->ctas < 2)  // the whole factor does not fit on chip at two CTAs per SM: checkpoint + recompute (K3)
        return launch_chunked(h, p, e, prm, coeffs, B, stream, slot);
      mtg::TmemLaunch tl;
      tl.n_tmem_blocks = plan->ntm;
      tl.tmem_cols = plan->cols;
      const int64_t blocks = (B + 63) / 64;
      auto fn = fused ? e->fn_tmem_fused : e->fn_tmem;
      {
        const int rc_smem = ensure_dyn_smem(h, (const void*)fn, plan->smem);
        if (rc_smem != MTG_OK) return rc_smem;
      }
      // coeffs as a 2-D fp64 tensor [B][K*D*N] for the TMA stores (box = 16 trajectories x one segment);
      // the encoded map is cached for repeated calls on the same output buffer
      if (!(h->tmap_key.base == coeffs && h->tmap_key.B == B && h->tmap_key.K == p->K && h->tmap_key.D == p->D &&
            h->tmap_key.N == p->N)) {
        const int rc = encode_coeff_tmap(h, &h->tmap_cached, coeffs, B, p);
        if (rc != MTG_OK) {
          h->tmap_key.base = nullptr;
          return rc;
        }
        h->tmap_key.base = coeffs;
        h->tmap_key.B = B;
        h->tmap_key.K = p->K;
        h->tmap_key.D = p->D;
        h->tmap_key.N = p->N;
      }
      fn<<<(unsigned)blocks, mtg::kTmemThreads, plan->smem, stream>>>(prm, tl, h->tmap_cached);
    } else if (use_v1) {
      {
        const int rc_smem = ensure_dyn_smem(h, (const void*)e->fn, size_t(smem_v1));
        if (rc_smem != MTG_OK) return rc_smem;
      }
      const int64_t blocks = (B + 31) / 32;
      e->fn<<<(unsigned)blocks, 32, smem_v1, stream>>>(prm);
    } else {
      const size_t smem = size_t((p->K + 1) / 2 - 1) * e->slots * 32 * sizeof(double);
      {
        const int rc_smem = ensure_dyn_smem(h, (const void*)e->fn_twisted, size_t(smem));
        if (rc_smem != MTG_OK) return rc_smem;
      }
      const int64_t blocks = (B + 15) / 16;
      e->fn_twisted<<<(unsigned)blocks, 32, smem, stream>>>(prm);
    }
    MTG_CUDA(h, cudaGetLastError());
    h->launches++;
    return MTG_OK;
  }
  if (kind == MTG_KERNEL_GENERIC && out_aligned && h->generic_variant == 0)
    return launch_masked(h, p, topo, B, times, dfix, coeffs, dfree, status, stream, slot);
  mtg::GenericParams prm;
  prm.N = p->N;
  prm.r = p->r;
  prm.K = p->K;
  prm.D = p->D;
  prm.n_fixed = L.n_fixed;
  prm.n_free = L.n_free;
  prm.bw = L.bw;
  prm.B = B;
  prm.slot_col = topo->d_slot_col;
  prm.times = times;
  prm.dfix = dfix;
  prm.dfree_in = dfree_in;
  prm.coeffs = coeffs;
  prm.dfree = dfree;
  prm.status = status;
  prm.scratch = nullptr;
  prm.scratch_stride = 0;
  const int threads = 128;
  int64_t blocks = (B + threads - 1) / threads;
  const int64_t max_blocks = int64_t(h->sm_count) * 8;
  if (blocks > max_blocks) blocks = max_blocks;
  if (kind == MTG_KERNEL_NOFREE) {
    if (L.n_free > 0 && dfree_in == nullptr) {
      h->error = "d_free is required for back-substitution of a problem with free constraints";
      return MTG_ERR_BAD_ARG;
    }
    mtg::backsub_kernel<<<(unsigned)blocks, threads, 0, stream>>>(prm);
  } else {
    const size_t per_thread = size_t(L.n_free) * (L.bw + 1 + p->D);
    const size_t bytes = per_thread * size_t(blocks) * threads * sizeof(double);
    mtg_handle::Arena& ar = h->scratch[slot];
    int rc = arena_acquire(h, ar, bytes, stream);
    if (rc != MTG_OK) return rc;
    prm.scratch = ar.p;
    prm.scratch_stride = blocks * threads;
    mtg::generic_solve_kernel<<<(unsigned)blocks, threads, 0, stream>>>(prm);
    MTG_CUDA(h, cudaGetLastError());
    rc = arena_release(h, ar, stream);
    if (rc != MTG_OK) return rc;
  }
  MTG_CUDA(h, cudaGetLastError());
  h->launches++;
  return MTG_OK;
}

int ensure_pipe(mtg_handle* h, int i, size_t bytes) {
  if (!h->streams[i]) MTG_CUDA(h, cudaStreamCreateWithFlags(&h->streams[i], cudaStreamNonBlocking));
  if (bytes > h->dev_buf_bytes[i]) {
    if (h->dev_buf[i]) {
      MTG_CUDA(h, cudaStreamSynchronize(h->streams[i]));
      cudaFree(h->dev_buf[i]);
      h->dev_buf[i] = nullptr;
      h->dev_buf_bytes[i] = 0;
    }
    MTG_CUDA(h, cudaMalloc(&h->dev_buf[i], bytes));
    h->dev_buf_bytes[i] = bytes;
  }
  return MTG_OK;
}

size_t align_up(size_t x) { return (x + 255) & ~size_t(255); }
// element counts of sub-buffers carved out of one allocation: keep every sub-buffer 256-byte aligned
// (the TMA tensor map of the coefficient buffer needs >= 16 bytes)
size_t align_doubles(size_t n) { return (n + 31) & ~size_t(31); }

}  // namespace

extern "C" {

int mtg_version(void) { return 100; }

int mtg_create(int device, mtg_handle** out) {
  if (!out) return MTG_ERR_BAD_ARG;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0) {
    g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e);
    return MTG_ERR_NO_DEVICE;
  }
  if (device < 0 || device >= count) {
    g_create_error = "device index out of range";
    return MTG_ERR_BAD_ARG;
  }
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) {
    g_create_error = std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e);
    return MTG_ERR_CUDA;
  }
  if (prop.major != 10) {
    g_create_error = "this library contains sm_100a code only; device is sm_" + std::to_string(prop.major) +
                     std::to_string(prop.minor);
    return MTG_ERR_NO_DEVICE;
  }
  mtg_handle* h = new (std::nothrow) mtg_handle();
  if (!h) return MTG_ERR_ALLOC;
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  h->cc_major = prop.major;
  h->smem_optin = prop.sharedMemPerBlockOptin;
  *out = h;
  return MTG_OK;
}

void mtg_destroy(mtg_handle* h) {
  if (!h) return;
  DeviceGuard g(h->device);
  cudaDeviceSynchronize();
  for (auto& t : h->topologies) {
    cudaFree(t.d_slot_col);
    cudaFree(t.d_vcol);
  }
  for (int i = 0; i <= mtg_handle::kPipe; ++i) {
    for (mtg_handle::Arena* a : {&h->scratch[i], &h->pack[i], &h->counters[i]}) {
      if (a->p) cudaFree(a->p);
      if (a->ev) cudaEventDestroy(a->ev);
    }
  }
  for (int i = 0; i < mtg_handle::kPipe; ++i) {
    if (h->dev_buf[i]) cudaFree(h->dev_buf[i]);
    if (h->streams[i]) cudaStreamDestroy(h->streams[i]);
  }
  delete h;
}

const char* mtg_last_error(const mtg_handle* h) { return h ? h->error.c_str() : g_create_error.c_str(); }

int64_t mtg_launch_count(const mtg_handle* h) { return h ? h->launches : 0; }

int mtg_device_is_sm100(const mtg_handle* h) { return h && h->cc_major == 10; }

int mtg_set_option(mtg_handle* h, int key, int value) {
  if (!h) return MTG_ERR_BAD_ARG;
  if (key == MTG_OPT_MELLINGER_UNFUSED && (value == 0 || value == 1)) {
    h->mellinger_unfused = value;
    return MTG_OK;
  }
  if (key == MTG_OPT_GENERIC_VARIANT && (value == 0 || value == 1)) {
    h->generic_variant = value;
    return MTG_OK;
  }
  if (key == MTG_OPT_CHUNK_BLOCKS && value >= 0 && value <= 64) {
    h->chunk_blocks = value;
    return MTG_OK;
  }
  if (key == MTG_OPT_TMA_INPUTS && value >= 0 && value <= 2) {
    h->tma_inputs = value;
    return MTG_OK;
  }
  if (key == MTG_OPT_WAYPOINT_VARIANT && value >= 0 && value <= 6) {
    h->waypoint_variant = value;
    return MTG_OK;
  }
  if (key == MTG_OPT_EARLY_REFILL && value >= -1 && value <= 0) {
    h->early_steps = value;
    return MTG_OK;
  }
  if (key == MTG_OPT_V5_STATIC_SHAPE && value >= -1 && value <= 0) {
    h->v5_static_shape = value;
    return MTG_OK;
  }
  if (key == MTG_OPT_RING_DEPTH && value >= 2 && value <= 4) {
    h->ring_depth = value;
    return MTG_OK;
  }
  if (key == MTG_OPT_CTAS_PER_SM && value >= 0 && value <= 9) {
    h->ctas_per_sm = value;
    return MTG_OK;
  }
  if (key == MTG_OPT_STAGGER_US && value >= 0 && value <= 1000) {
    h->stagger_us = value;
    return MTG_OK;
  }
  if (key == MTG_OPT_DYNAMIC_TILES && value >= 0 && value <= 2) {  // 0 = auto, 1 = always, 2 = never
    h->dynamic_tiles = value;
    return MTG_OK;
  }
  h->error = "unknown option";
  return MTG_ERR_BAD_ARG;
}

int mtg_problem_layout(const mtg_problem* p, mtg_layout* out, int32_t* slot_col) {
  if (!valid_problem(p) || !out) return MTG_ERR_BAD_ARG;
  Layout L;
  compute_layout(p->N, p->K, canonical_mask(p), &L);
  out->n_all = L.n_all;
  out->n_fixed = L.n_fixed;
  out->n_free = L.n_free;
  // routing without a device: assume the B200 opt-in shared memory limit (227 KB)
  mtg_handle fake;
  fake.smem_optin = 227 * 1024;
  out->kernel = route(&fake, p, L);
  if (slot_col) std::memcpy(slot_col, L.slot_col.data(), sizeof(int32_t) * L.slot_col.size());
  return MTG_OK;
}

int mtg_solve_linear_batch_f64(mtg_handle* h, const mtg_problem* p, int64_t B, const double* seg_times,
                               const double* d_fixed, double* coeffs, double* d_free, int32_t* status,
                               void* stream) {
  if (!h) return MTG_ERR_BAD_ARG;
  if (!valid_problem(p) || B < 0 || (B > 0 && (!seg_times || !d_fixed || !coeffs))) {
    h->error = "bad argument";
    return MTG_ERR_BAD_ARG;
  }
  DeviceGuard g(h->device);
  CachedTopology* topo = get_topology(h, p);
  if (!topo) return MTG_ERR_CUDA;
  return launch_solve(h, p, topo, B, seg_times, d_fixed, nullptr, coeffs, d_free, status, (cudaStream_t)stream,
                      false);
}

static int nfabian_device(mtg_handle* h, int32_t N, int32_t r, int32_t K, int32_t D, int64_t B,
                          const double* positions, double v_max, double a_max, double magic, double* coeffs,
                          double* seg_times_out, int32_t* status, cudaStream_t s, int slot) {
  if (!h) return MTG_ERR_BAD_ARG;
  mtg_problem p = {N, r, K, D, nullptr};
  if (!valid_problem(&p) || B < 0 || !(v_max > 0.0) || !(a_max > 0.0) || (B > 0 && (!positions || !coeffs))) {
    h->error = "bad argument";
    return MTG_ERR_BAD_ARG;
  }
  if (B == 0) return MTG_OK;
  DeviceGuard g(h->device);
  CachedTopology* topo = get_topology(h, &p);
  if (!topo) return MTG_ERR_CUDA;
  const Layout& L = topo->layout;
  if (route(h, &p, L) == MTG_KERNEL_WAYPOINT) {
    FusedInput f = {positions, v_max, a_max, magic, seg_times_out};
    const int rc = launch_solve(h, &p, topo, B, nullptr, nullptr, nullptr, coeffs, nullptr, status, s, false, &f, slot);
    if (rc != MTG_ERR_ALLOC) return rc;
  }
  // no fused specialisation: pack (times, d_fixed) with a small kernel, then the regular path
  const size_t n_t = align_doubles(size_t(B) * K), n_f = size_t(B) * D * L.n_fixed;
  mtg_handle::Arena& ar = h->pack[slot];
  int rc = arena_acquire(h, ar, (n_t + n_f) * 8, s);
  if (rc != MTG_OK) return rc;
  double* t_buf = seg_times_out ? seg_times_out : ar.p;
  double* f_buf = ar.p + n_t;
  mtg::PackParams pk;
  pk.N = N;
  pk.K = K;
  pk.D = D;
  pk.n_fixed = L.n_fixed;
  pk.B = B;
  pk.positions = positions;
  pk.v_max = v_max;
  pk.a_max = a_max;
  pk.magic = magic;
  pk.times = t_buf;
  pk.dfix = f_buf;
  const int threads = 128;
  const int64_t blocks = std::min<int64_t>((B + threads - 1) / threads, int64_t(h->sm_count) * 16);
  mtg::nfabian_pack_kernel<<<(unsigned)blocks, threads, 0, s>>>(pk);
  MTG_CUDA(h, cudaGetLastError());
  h->launches++;
  rc = launch_solve(h, &p, topo, B, t_buf, f_buf, nullptr, coeffs, nullptr, status, s, false, nullptr, slot);
  if (rc != MTG_OK) return rc;
  return arena_release(h, ar, s);  // the solve was the last reader of the packed inputs
}

int mtg_solve_waypoints_nfabian_batch_f64(mtg_handle* h, int32_t N, int32_t r, int32_t K, int32_t D, int64_t B,
                                          const double* positions, double v_max, double a_max, double magic,
                                          double* coeffs, double* seg_times_out, int32_t* status, void* stream) {
  return nfabian_device(h, N, r, K, D, B, positions, v_max, a_max, magic, coeffs, seg_times_out, status,
                        (cudaStream_t)stream, mtg_handle::kPipe);
}

int mtg_coeffs_from_constraints_batch_f64(mtg_handle* h, const mtg_problem* p, int64_t B,
                                          const double* seg_times, const double* d_fixed,
                                          const double* d_free, double* coeffs, void* stream) {
  if (!h) return MTG_ERR_BAD_ARG;
  if (!valid_problem(p) || B < 0 || (B > 0 && (!seg_times || !d_fixed || !coeffs))) {
    h->error = "bad argument";
    return MTG_ERR_BAD_ARG;
  }
  DeviceGuard g(h->device);
  CachedTopology* topo = get_topology(h, p);
  if (!topo) return MTG_ERR_CUDA;
  return launch_solve(h, p, topo, B, seg_times, d_fixed, d_free, coeffs, nullptr, nullptr, (cudaStream_t)stream,
                      true);
}

int mtg_compute_cost_batch_f64(mtg_handle* h, const mtg_problem* p, int64_t B, const double* seg_times,
                               const double* coeffs, double* cost, void* stream) {
  if (!h) return MTG_ERR_BAD_ARG;
  if (!valid_problem(p) || B < 0 || (B > 0 && (!seg_times || !coeffs || !cost))) {
    h->error = "bad argument";
    return MTG_ERR_BAD_ARG;
  }
  if (B == 0) return MTG_OK;
  DeviceGuard g(h->device);
  mtg::CostParams prm;
  prm.N = p->N;
  prm.r = p->r;
  prm.K = p->K;
  prm.D = p->D;
  prm.B = B;
  prm.times = seg_times;
  prm.coeffs = coeffs;
  prm.cost = cost;
  const int threads = 256;
  const int KD = p->K * p->D;
  const int tpb = std::max(1, threads / KD);
  const size_t smem = (size_t(36) + size_t(tpb) * KD) * sizeof(double);
  if (smem > h->smem_optin) {
    h->error = "mtg_compute_cost_batch_f64: K * D too large";
    return MTG_ERR_BAD_ARG;
  }
  typedef void (*CostFn)(const mtg::CostParams, const int);
  struct CostEntry {
    int N, r;
    CostFn fn;
  };
  static const CostEntry kCost[] = {{10, 4, mtg::cost_kernel<10, 4>}, {10, 3, mtg::cost_kernel<10, 3>},
                                    {10, 2, mtg::cost_kernel<10, 2>}, {8, 3, mtg::cost_kernel<8, 3>},
                                    {12, 5, mtg::cost_kernel<12, 5>}, {12, 4, mtg::cost_kernel<12, 4>},
                                    {6, 2, mtg::cost_kernel<6, 2>},   {4, 1, mtg::cost_kernel<4, 1>}};
  CostFn fn = mtg::cost_kernel<0, 0>;
  for (const auto& e : kCost)
    if (e.N == p->N && e.r == p->r) fn = e.fn;
  {
    const int rc_smem = ensure_dyn_smem(h, (const void*)fn, smem);
    if (rc_smem != MTG_OK) return rc_smem;
  }
  int64_t blocks = std::min<int64_t>((B + tpb - 1) / tpb, int64_t(h->sm_count) * 16);
  fn<<<(unsigned)blocks, threads, smem, (cudaStream_t)stream>>>(prm, tpb);
  MTG_CUDA(h, cudaGetLastError());
  h->launches++;
  return MTG_OK;
}

int mtg_evaluate_batch_f64(mtg_handle* h, int32_t N, int32_t K, int32_t D, int64_t B, const double* seg_times,
                           const double* coeffs, int32_t derivative, double t_start, double dt, int32_t n_samples,
                           double* out, void* stream) {
  if (!h) return MTG_ERR_BAD_ARG;
  if (N < 1 || N > MTG_MAX_N || K < 1 || D < 1 || B < 0 || derivative < 0 || n_samples < 0 ||
      (B > 0 && n_samples > 0 && (!seg_times || !coeffs || !out))) {
    h->error = "bad argument";
    return MTG_ERR_BAD_ARG;
  }
  if (B == 0 || n_samples == 0) return MTG_OK;
  DeviceGuard g(h->device);
  mtg::EvalParams ep;
  ep.N = N;
  ep.K = K;
  ep.D = D;
  ep.derivative = derivative;
  ep.n_samples = n_samples;
  ep.B = B;
  ep.t_start = t_start;
  ep.dt = dt;
  ep.times = seg_times;
  ep.coeffs = coeffs;
  ep.out = out;
  if (size_t(32) * D * 8 > size_t(160) * 1024) {
    h->error = "mtg_evaluate_batch_f64: D too large for the output tile";
    return MTG_ERR_BAD_ARG;
  }
  const int threads = std::max(32, std::min(256, int((40 * 1024) / (D * 8)) / 32 * 32));
  const size_t smem = size_t(threads) * D * sizeof(double);
  typedef void (*EvalFn)(const mtg::EvalParams);
  static const EvalFn kEval[MTG_MAX_N] = {
      mtg::evaluate_kernel<1>, mtg::evaluate_kernel<2>,  mtg::evaluate_kernel<3>,  mtg::evaluate_kernel<4>,
      mtg::evaluate_kernel<5>, mtg::evaluate_kernel<6>,  mtg::evaluate_kernel<7>,  mtg::evaluate_kernel<8>,
      mtg::evaluate_kernel<9>, mtg::evaluate_kernel<10>, mtg::evaluate_kernel<11>, mtg::evaluate_kernel<12>};
  const EvalFn fn = kEval[N - 1];
  {
    const int rc_smem = ensure_dyn_smem(h, (const void*)fn, smem);
    if (rc_smem != MTG_OK) return rc_smem;
  }
  const int64_t total = B * int64_t(n_samples);
  const int64_t blocks = std::min<int64_t>((total + threads - 1) / threads, int64_t(h->sm_count) * 32);
  fn<<<(unsigned)blocks, threads, smem, (cudaStream_t)stream>>>(ep);
  MTG_CUDA(h, cudaGetLastError());
  h->launches++;
  return MTG_OK;
}

int mtg_evaluate_range_batch_f64(mtg_handle* h, int32_t N, int32_t K, int32_t D, int64_t B, const double* seg_times,
                                 const double* coeffs, double t_start, double t_end, double dt, int32_t n_derivs,
                                 const int32_t* derivs, int32_t max_samples, double* out, int32_t* n_samples,
                                 double* sampling_times, void* stream) {
  if (!h) return MTG_ERR_BAD_ARG;
  if (N < 1 || N > MTG_MAX_N || K < 1 || D < 1 || B < 0 || n_derivs < 1 || n_derivs > 8 || !derivs || max_samples < 0 ||
      !(dt > 0.0) || (B > 0 && (!seg_times || !coeffs || !n_samples || (max_samples > 0 && !out)))) {
    h->error = "bad argument";
    return MTG_ERR_BAD_ARG;
  }
  for (int q = 0; q < n_derivs; ++q)
    if (derivs[q] < 0) {
      h->error = "bad argument";
      return MTG_ERR_BAD_ARG;
    }
  if (B == 0) return MTG_OK;
  DeviceGuard g(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t ns = size_t(B) * size_t(std::max(max_samples, 1));
  mtg_handle::Arena& ar = h->pack[mtg_handle::kPipe];
  const size_t o_idx = align_doubles(ns);  // t_local first (doubles), then seg_idx (int32)
  int rc = arena_acquire(h, ar, (o_idx + align_doubles((ns + 1) / 2)) * 8, s);
  if (rc != MTG_OK) return rc;
  mtg::RangeParams rp;
  rp.N = N;
  rp.K = K;
  rp.D = D;
  rp.n_derivs = n_derivs;
  rp.max_samples = max_samples;
  for (int q = 0; q < 8; ++q) rp.derivs[q] = q < n_derivs ? derivs[q] : 0;
  rp.B = B;
  rp.t_start = t_start;
  rp.t_end = t_end;
  rp.dt = dt;
  rp.times = seg_times;
  rp.coeffs = coeffs;
  rp.t_local = ar.p;
  rp.seg_idx = reinterpret_cast<int*>(ar.p + o_idx);
  rp.n_samples = n_samples;
  rp.sampling_times = sampling_times;
  rp.out = out;
  {
    const int threads = 128;
    const int64_t blocks = std::min<int64_t>((B + threads - 1) / threads, int64_t(h->sm_count) * 16);
    mtg::range_walk_kernel<<<(unsigned)blocks, threads, 0, s>>>(rp);
    MTG_CUDA(h, cudaGetLastError());
    h->launches++;
  }
  if (max_samples > 0) {
    // block size: the output tile (threads * n_derivs * D doubles) stays under 40 KB of shared memory
    const int rec = n_derivs * D;
    if (size_t(32) * rec * 8 > size_t(160) * 1024) {
      h->error = "mtg_evaluate_range_batch_f64: n_derivs * D too large for the output tile";
      arena_release(h, ar, s);
      return MTG_ERR_BAD_ARG;
    }
    const int threads = std::max(32, std::min(256, int((40 * 1024) / (rec * 8)) / 32 * 32));
    const size_t smem = size_t(threads) * rec * sizeof(double);
    typedef void (*RangeEval)(const mtg::RangeParams);
    static const RangeEval kRangeEval[MTG_MAX_N] = {
        mtg::range_eval_kernel<1>, mtg::range_eval_kernel<2>,  mtg::range_eval_kernel<3>,  mtg::range_eval_kernel<4>,
        mtg::range_eval_kernel<5>, mtg::range_eval_kernel<6>,  mtg::range_eval_kernel<7>,  mtg::range_eval_kernel<8>,
        mtg::range_eval_kernel<9>, mtg::range_eval_kernel<10>, mtg::range_eval_kernel<11>, mtg::range_eval_kernel<12>};
    const RangeEval fn = kRangeEval[N - 1];
    {
      const int rc_smem = ensure_dyn_smem(h, (const void*)fn, smem);
      if (rc_smem != MTG_OK) return rc_smem;
    }
    const int64_t total = B * int64_t(max_samples);
    const int64_t blocks = std::min<int64_t>((total + threads - 1) / threads, int64_t(h->sm_count) * 32);
    fn<<<(unsigned)blocks, threads, smem, s>>>(rp);
    MTG_CUDA(h, cudaGetLastError());
    h->launches++;
  }
  return arena_release(h, ar, s);
}

int mtg_cost_gradient_mellinger_batch_f64(mtg_handle* h, const mtg_problem* p, int64_t B, const double* seg_times,
                                          const double* d_fixed, double* cost, double* grad, void* stream) {
  if (!h) return MTG_ERR_BAD_ARG;
  if (!valid_problem(p) || B < 0 || (B > 0 && (!seg_times || !d_fixed || !grad))) {
    h->error = "bad argument";
    return MTG_ERR_BAD_ARG;
  }
  if (B == 0) return MTG_OK;
  DeviceGuard g(h->device);
  CachedTopology* topo = get_topology(h, p);
  if (!topo) return MTG_ERR_CUDA;
  const Layout& L = topo->layout;
  cudaStream_t s = (cudaStream_t)stream;
  const size_t K = p->K, D = p->D, N = p->N, nf = L.n_fixed;
  if (p->K > 1 && h->mellinger_unfused == 0) {
    // fused path: one cost-only launch over the B*(K+1) expanded problems (expansion generated in the kernel, no
    // perturbed inputs or coefficients ever written), then the finite differences
    mtg_handle::Arena& arf = h->pack[mtg_handle::kPipe];
    int rc = arena_acquire(h, arf, size_t(B) * (K + 1) * 8, s);
    if (rc != MTG_OK) return rc;
    rc = launch_cost_fused(h, p, topo, B * int64_t(K + 1), seg_times, d_fixed, arf.p, int(K + 1), 0.1, 0.1, s);
    if (rc == MTG_OK) {
      const int threads = 128;
      const int64_t gb = std::min<int64_t>((B + threads - 1) / threads, int64_t(h->sm_count) * 16);
      mtg::mellinger_gradient_kernel<<<(unsigned)gb, threads, 0, s>>>(B, p->K, arf.p, cost, grad, 0.1);
      MTG_CUDA(h, cudaGetLastError());
      h->launches++;
      return arena_release(h, arf, s);
    }
    if (rc != MTG_ERR_ALLOC) return rc;
  }
  const size_t per_x = (K + D * nf + K * D * N + 1) * 8;  // times + d_fixed + coeffs + cost of one expanded problem
  int64_t chunk = std::max<int64_t>(1, int64_t((size_t(384) << 20) / (per_x * (K + 1))));
  chunk = std::min<int64_t>(chunk, B);
  const size_t nx_max = size_t(chunk) * (K + 1);
  const size_t o_f = align_doubles(nx_max * K), o_c = o_f + align_doubles(nx_max * D * nf),
               o_j = o_c + align_doubles(nx_max * K * D * N), need = (o_j + align_doubles(nx_max)) * 8;
  mtg_handle::Arena& ar = h->pack[mtg_handle::kPipe];
  {
    const int rc = arena_acquire(h, ar, need, s);
    if (rc != MTG_OK) return rc;
  }
  for (int64_t b0 = 0; b0 < B; b0 += chunk) {
    const int64_t nb = std::min<int64_t>(chunk, B - b0), nx = nb * int64_t(K + 1);
    double* t_x = ar.p;
    double* f_x = ar.p + o_f;
    double* c_x = ar.p + o_c;
    double* j_x = ar.p + o_j;
    mtg::MellingerParams mp;
    mp.K = p->K;
    mp.D = p->D;
    mp.n_fixed = L.n_fixed;
    mp.B = nb;
    mp.times = seg_times + b0 * K;
    mp.dfix = d_fixed + b0 * D * nf;
    mp.times_x = t_x;
    mp.dfix_x = f_x;
    mp.increment = 0.1;  // reference: increment_time (nonlinear_impl.h:310)
    mp.lower = 0.1;      // kOptimizationTimeLowerBound (polynomial_optimization_nonlinear.h:31)
    const int threads = 128;
    const int64_t blocks = std::min<int64_t>((nx + threads - 1) / threads, int64_t(h->sm_count) * 16);
    mtg::mellinger_expand_kernel<<<(unsigned)blocks, threads, 0, s>>>(mp);
    MTG_CUDA(h, cudaGetLastError());
    h->launches++;
    int rc = launch_solve(h, p, topo, nx, t_x, f_x, nullptr, c_x, nullptr, nullptr, s, false);
    if (rc != MTG_OK) return rc;
    rc = mtg_compute_cost_batch_f64(h, p, nx, t_x, c_x, j_x, s);
    if (rc != MTG_OK) return rc;
    const int64_t gb = std::min<int64_t>((nb + threads - 1) / threads, int64_t(h->sm_count) * 16);
    mtg::mellinger_gradient_kernel<<<(unsigned)gb, threads, 0, s>>>(nb, p->K, j_x, cost ? cost + b0 : nullptr,
                                                                  grad + b0 * K, mp.increment);
    MTG_CUDA(h, cudaGetLastError());
    h->launches++;
  }
  return arena_release(h, ar, s);
}

// ---- host-pointer variants: chunked H2D -> kernel -> D2H over kPipe streams ---------------
// Every exit of a host-pointer entry point -- error returns included -- waits for all pipeline streams:
// copies into caller-owned (possibly pinned) buffers must not be in flight when the caller gets control back.
struct PipeSyncGuard {
  mtg_handle* h;
  ~PipeSyncGuard() {
    for (int i = 0; i < mtg_handle::kPipe; ++i)
      if (h->streams[i]) cudaStreamSynchronize(h->streams[i]);
  }
};

static int host_pipeline(mtg_handle* h, const mtg_problem* p, int64_t B, const double* seg_times,
                         const double* d_fixed, const double* d_free_in, double* coeffs, double* d_free_out,
                         int32_t* status, bool backsub_only) {
  if (!h) return MTG_ERR_BAD_ARG;
  if (!valid_problem(p) || B < 0 || (B > 0 && (!seg_times || !d_fixed || !coeffs))) {
    h->error = "bad argument";
    return MTG_ERR_BAD_ARG;
  }
  if (B == 0) return MTG_OK;
  DeviceGuard g(h->device);
  CachedTopology* topo = get_topology(h, p);
  if (!topo) return MTG_ERR_CUDA;
  const Layout& L = topo->layout;
  const size_t K = p->K, D = p->D, N = p->N;
  const size_t b_times = K * 8, b_fix = D * L.n_fixed * 8, b_free = D * size_t(L.n_free) * 8,
               b_coef = K * D * N * 8;
  const bool need_free_in = backsub_only && L.n_free > 0;
  if (need_free_in && !d_free_in) {
    h->error = "d_free is required";
    return MTG_ERR_BAD_ARG;
  }
  // chunk so that the pipeline has work for every stream but stays in a few tens of MB
  int64_t chunk = std::max<int64_t>(1, std::min<int64_t>((B + mtg_handle::kPipe - 1) / mtg_handle::kPipe, 32768));
  if (B <= 4096) chunk = B;
  int rc = MTG_OK;
  int slot = 0;
  PipeSyncGuard sync_on_exit{h};
  for (int64_t b0 = 0; b0 < B; b0 += chunk, slot = (slot + 1) % mtg_handle::kPipe) {
    const int64_t nb = std::min<int64_t>(chunk, B - b0);
    const size_t o_times = 0;
    const size_t o_fix = align_up(o_times + b_times * nb);
    const size_t o_freein = align_up(o_fix + b_fix * nb);
    const size_t o_coef = align_up(o_freein + (need_free_in ? b_free * nb : 0));
    const size_t o_free = align_up(o_coef + b_coef * nb);
    const size_t o_stat = align_up(o_free + (d_free_out ? b_free * nb : 0));
    const size_t total = align_up(o_stat + (status ? 4 * nb : 0));
    rc = ensure_pipe(h, slot, total);
    if (rc != MTG_OK) return rc;
    cudaStream_t s = h->streams[slot];
    char* base = static_cast<char*>(h->dev_buf[slot]);
    MTG_CUDA(h, cudaMemcpyAsync(base + o_times, seg_times + b0 * K, b_times * nb, cudaMemcpyHostToDevice, s));
    MTG_CUDA(h, cudaMemcpyAsync(base + o_fix, d_fixed + b0 * D * L.n_fixed, b_fix * nb, cudaMemcpyHostToDevice, s));
    if (need_free_in)
      MTG_CUDA(h, cudaMemcpyAsync(base + o_freein, d_free_in + b0 * D * L.n_free, b_free * nb,
                                  cudaMemcpyHostToDevice, s));
    rc = launch_solve(h, p, topo, nb, reinterpret_cast<double*>(base + o_times),
                      reinterpret_cast<double*>(base + o_fix),
                      need_free_in ? reinterpret_cast<double*>(base + o_freein) : nullptr,
                      reinterpret_cast<double*>(base + o_coef),
                      d_free_out ? reinterpret_cast<double*>(base + o_free) : nullptr,
                      status ? reinterpret_cast<int32_t*>(base + o_stat) : nullptr, s, backsub_only, nullptr, slot);
    if (rc != MTG_OK) return rc;
    MTG_CUDA(h, cudaMemcpyAsync(coeffs + b0 * K * D * N, base + o_coef, b_coef * nb, cudaMemcpyDeviceToHost, s));
    if (d_free_out && L.n_free > 0)
      MTG_CUDA(h, cudaMemcpyAsync(d_free_out + b0 * D * L.n_free, base + o_free, b_free * nb,
                                  cudaMemcpyDeviceToHost, s));
    if (status) MTG_CUDA(h, cudaMemcpyAsync(status + b0, base + o_stat, 4 * nb, cudaMemcpyDeviceToHost, s));
    // the buffer of this slot is reused kPipe chunks later: wait for it then
    const int next = (slot + 1) % mtg_handle::kPipe;
    if (b0 + chunk < B && h->streams[next]) MTG_CUDA(h, cudaStreamSynchronize(h->streams[next]));
  }
  for (int i = 0; i < mtg_handle::kPipe; ++i)
    if (h->streams[i]) MTG_CUDA(h, cudaStreamSynchronize(h->streams[i]));
  return MTG_OK;
}

int mtg_solve_linear_batch_host_f64(mtg_handle* h, const mtg_problem* p, int64_t B, const double* seg_times,
                                    const double* d_fixed, double* coeffs, double* d_free, int32_t* status) {
  return host_pipeline(h, p, B, seg_times, d_fixed, nullptr, coeffs, d_free, status, false);
}

int mtg_solve_waypoints_nfabian_batch_host_f64(mtg_handle* h, int32_t N, int32_t r, int32_t K, int32_t D, int64_t B,
                                               const double* positions, double v_max, double a_max, double magic,
                                               double* coeffs, double* seg_times_out, int32_t* status) {
  if (!h) return MTG_ERR_BAD_ARG;
  mtg_problem p = {N, r, K, D, nullptr};
  if (!valid_problem(&p) || B < 0 || (B > 0 && (!positions || !coeffs))) {
    h->error = "bad argument";
    return MTG_ERR_BAD_ARG;
  }
  if (B == 0) return MTG_OK;
  DeviceGuard g(h->device);
  const size_t b_pos = size_t(K + 1) * D * 8, b_coef = size_t(K) * D * N * 8, b_t = size_t(K) * 8;
  int64_t chunk = std::max<int64_t>(1, std::min<int64_t>((B + mtg_handle::kPipe - 1) / mtg_handle::kPipe, 32768));
  if (B <= 4096) chunk = B;
  int slot = 0;
  PipeSyncGuard sync_on_exit{h};
  for (int64_t b0 = 0; b0 < B; b0 += chunk, slot = (slot + 1) % mtg_handle::kPipe) {
    const int64_t nb = std::min<int64_t>(chunk, B - b0);
    const size_t o_coef = align_up(b_pos * nb), o_t = align_up(o_coef + b_coef * nb), o_stat = align_up(o_t + b_t * nb);
    int rc = ensure_pipe(h, slot, align_up(o_stat + 4 * nb));
    if (rc != MTG_OK) return rc;
    cudaStream_t s = h->streams[slot];
    char* base = static_cast<char*>(h->dev_buf[slot]);
    MTG_CUDA(h, cudaMemcpyAsync(base, positions + b0 * (K + 1) * D, b_pos * nb, cudaMemcpyHostToDevice, s));
    rc = nfabian_device(h, N, r, K, D, nb, reinterpret_cast<double*>(base), v_max, a_max, magic,
                        reinterpret_cast<double*>(base + o_coef), reinterpret_cast<double*>(base + o_t),
                        reinterpret_cast<int32_t*>(base + o_stat), s, slot);
    if (rc != MTG_OK) return rc;
    MTG_CUDA(h, cudaMemcpyAsync(coeffs + b0 * K * D * N, base + o_coef, b_coef * nb, cudaMemcpyDeviceToHost, s));
    if (seg_times_out)
      MTG_CUDA(h, cudaMemcpyAsync(seg_times_out + b0 * K, base + o_t, b_t * nb, cudaMemcpyDeviceToHost, s));
    if (status) MTG_CUDA(h, cudaMemcpyAsync(status + b0, base + o_stat, 4 * nb, cudaMemcpyDeviceToHost, s));
    const int next = (slot + 1) % mtg_handle::kPipe;
    if (b0 + chunk < B && h->streams[next]) MTG_CUDA(h, cudaStreamSynchronize(h->streams[next]));
  }
  for (int i = 0; i < mtg_handle::kPipe; ++i)
    if (h->streams[i]) MTG_CUDA(h, cudaStreamSynchronize(h->streams[i]));
  return MTG_OK;
}

int mtg_coeffs_from_constraints_batch_host_f64(mtg_handle* h, const mtg_problem* p, int64_t B,
                                               const double* seg_times, const double* d_fixed,
                                               const double* d_free, double* coeffs) {
  return host_pipeline(h, p, B, seg_times, d_fixed, d_free, coeffs, nullptr, nullptr, true);
}

int mtg_compute_cost_batch_host_f64(mtg_handle* h, const mtg_problem* p, int64_t B, const double* seg_times,
                                    const double* coeffs, double* cost) {
  if (!h) return MTG_ERR_BAD_ARG;
  if (!valid_problem(p) || B < 0 || (B > 0 && (!seg_times || !coeffs || !cost))) {
    h->error = "bad argument";
    return MTG_ERR_BAD_ARG;
  }
  if (B == 0) return MTG_OK;
  DeviceGuard g(h->device);
  const size_t K = p->K, D = p->D, N = p->N;
  const size_t o_coef = align_up(K * 8 * B), o_cost = align_up(o_coef + K * D * N * 8 * B);
  int rc = ensure_pipe(h, 0, o_cost + 8 * B);
  if (rc != MTG_OK) return rc;
  cudaStream_t s = h->streams[0];
  char* base = static_cast<char*>(h->dev_buf[0]);
  MTG_CUDA(h, cudaMemcpyAsync(base, seg_times, K * 8 * B, cudaMemcpyHostToDevice, s));
  MTG_CUDA(h, cudaMemcpyAsync(base + o_coef, coeffs, K * D * N * 8 * B, cudaMemcpyHostToDevice, s));
  rc = mtg_compute_cost_batch_f64(h, p, B, reinterpret_cast<double*>(base), reinterpret_cast<double*>(base + o_coef),
                                  reinterpret_cast<double*>(base + o_cost), s);
  if (rc != MTG_OK) return rc;
  MTG_CUDA(h, cudaMemcpyAsync(cost, base + o_cost, 8 * B, cudaMemcpyDeviceToHost, s));
  MTG_CUDA(h, cudaStreamSynchronize(s));
  return MTG_OK;
}

int mtg_cost_gradient_mellinger_batch_host_f64(mtg_handle* h, const mtg_problem* p, int64_t B, const double* seg_times,
                                               const double* d_fixed, double* cost, double* grad) {
  if (!h) return MTG_ERR_BAD_ARG;
  if (!valid_problem(p) || B < 0 || (B > 0 && (!seg_times || !d_fixed || !grad))) {
    h->error = "bad argument";
    return MTG_ERR_BAD_ARG;
  }
  if (B == 0) return MTG_OK;
  DeviceGuard g(h->device);
  CachedTopology* topo = get_topology(h, p);
  if (!topo) return MTG_ERR_CUDA;
  const size_t K = p->K, D = p->D, nf = topo->layout.n_fixed;
  const size_t o_f = align_up(K * 8 * B), o_c = align_up(o_f + D * nf * 8 * B), o_g = align_up(o_c + 8 * B);
  int rc = ensure_pipe(h, 0, o_g + K * 8 * B);
  if (rc != MTG_OK) return rc;
  cudaStream_t s = h->streams[0];
  char* base = static_cast<char*>(h->dev_buf[0]);
  PipeSyncGuard sync_on_exit{h};
  MTG_CUDA(h, cudaMemcpyAsync(base, seg_times, K * 8 * B, cudaMemcpyHostToDevice, s));
  MTG_CUDA(h, cudaMemcpyAsync(base + o_f, d_fixed, D * nf * 8 * B, cudaMemcpyHostToDevice, s));
  rc = mtg_cost_gradient_mellinger_batch_f64(h, p, B, reinterpret_cast<double*>(base), reinterpret_cast<double*>(base + o_f),
                                             reinterpret_cast<double*>(base + o_c), reinterpret_cast<double*>(base + o_g), s);
  if (rc != MTG_OK) return rc;
  if (cost) MTG_CUDA(h, cudaMemcpyAsync(cost, base + o_c, 8 * B, cudaMemcpyDeviceToHost, s));
  MTG_CUDA(h, cudaMemcpyAsync(grad, base + o_g, K * 8 * B, cudaMemcpyDeviceToHost, s));
  MTG_CUDA(h, cudaStreamSynchronize(s));
  return MTG_OK;
}

int mtg_evaluate_range_batch_host_f64(mtg_handle* h, int32_t N, int32_t K, int32_t D, int64_t B, const double* seg_times,
                                      const double* coeffs, double t_start, double t_end, double dt, int32_t n_derivs,
                                      const int32_t* derivs, int32_t max_samples, double* out, int32_t* n_samples,
                                      double* sampling_times) {
  if (!h) return MTG_ERR_BAD_ARG;
  if (N < 1 || N > MTG_MAX_N || K < 1 || D < 1 || B < 0 || n_derivs < 1 || n_derivs > 8 || max_samples < 0 ||
      (B > 0 && (!seg_times || !coeffs || !n_samples || (max_samples > 0 && !out)))) {
    h->error = "bad argument";
    return MTG_ERR_BAD_ARG;
  }
  if (B == 0) return MTG_OK;
  DeviceGuard g(h->device);
  const size_t b_t = size_t(K) * 8 * B, b_c = size_t(K) * D * N * 8 * B, b_o = size_t(max_samples) * n_derivs * D * 8 * B,
               b_n = 4 * size_t(B), b_s = size_t(max_samples) * 8 * B;
  const size_t o_c = align_up(b_t), o_o = align_up(o_c + b_c), o_n = align_up(o_o + b_o), o_s = align_up(o_n + b_n);
  int rc = ensure_pipe(h, 0, o_s + b_s);
  if (rc != MTG_OK) return rc;
  cudaStream_t s = h->streams[0];
  char* base = static_cast<char*>(h->dev_buf[0]);
  PipeSyncGuard sync_on_exit{h};
  MTG_CUDA(h, cudaMemcpyAsync(base, seg_times, b_t, cudaMemcpyHostToDevice, s));
  MTG_CUDA(h, cudaMemcpyAsync(base + o_c, coeffs, b_c, cudaMemcpyHostToDevice, s));
  rc = mtg_evaluate_range_batch_f64(h, N, K, D, B, reinterpret_cast<double*>(base), reinterpret_cast<double*>(base + o_c),
                                    t_start, t_end, dt, n_derivs, derivs, max_samples, reinterpret_cast<double*>(base + o_o),
                                    reinterpret_cast<int32_t*>(base + o_n),
                                    sampling_times ? reinterpret_cast<double*>(base + o_s) : nullptr, s);
  if (rc != MTG_OK) return rc;
  if (max_samples > 0) MTG_CUDA(h, cudaMemcpyAsync(out, base + o_o, b_o, cudaMemcpyDeviceToHost, s));
  MTG_CUDA(h, cudaMemcpyAsync(n_samples, base + o_n, b_n, cudaMemcpyDeviceToHost, s));
  if (sampling_times && max_samples > 0)
    MTG_CUDA(h, cudaMemcpyAsync(sampling_times, base + o_s, b_s, cudaMemcpyDeviceToHost, s));
  MTG_CUDA(h, cudaStreamSynchronize(s));
  return MTG_OK;
}

void* mtg_host_alloc(mtg_handle* h, uint64_t bytes) {
  void* p = nullptr;
  if (!h) return nullptr;
  DeviceGuard g(h->device);
  if (set_err(h, "cudaMallocHost", cudaMallocHost(&p, bytes ? bytes : 1))) return nullptr;
  return p;
}
void mtg_host_free(mtg_handle* h, void* ptr) {
  if (h && ptr) {
    DeviceGuard g(h->device);
    cudaFreeHost(ptr);
  }
}
void* mtg_device_alloc(mtg_handle* h, uint64_t bytes) {
  void* p = nullptr;
  if (!h) return nullptr;
  DeviceGuard g(h->device);
  if (set_err(h, "cudaMalloc", cudaMalloc(&p, bytes ? bytes : 1))) return nullptr;
  return p;
}
void mtg_device_free(mtg_handle* h, void* ptr) {
  if (h && ptr) {
    DeviceGuard g(h->device);
    cudaFree(ptr);
  }
}
int mtg_memcpy_h2d(mtg_handle* h, void* dst, const void* src, uint64_t bytes, void* stream) {
  if (!h) return MTG_ERR_BAD_ARG;
  DeviceGuard g(h->device);
  MTG_CUDA(h, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
  return MTG_OK;
}
int mtg_memcpy_d2h(mtg_handle* h, void* dst, const void* src, uint64_t bytes, void* stream) {
  if (!h) return MTG_ERR_BAD_ARG;
  DeviceGuard g(h->device);
  MTG_CUDA(h, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  return MTG_OK;
}
int mtg_memcpy_d2d(mtg_handle* h, void* dst, const void* src, uint64_t bytes, void* stream) {
  if (!h) return MTG_ERR_BAD_ARG;
  DeviceGuard g(h->device);
  MTG_CUDA(h, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, (cudaStream_t)stream));
  return MTG_OK;
}

// ---- peer memory (NVLink): export / import a device allocation between the one-process-per-GPU ranks ----------
int mtg_ipc_export(mtg_handle* h, const void* ptr, uint8_t handle_out[64], uint64_t* offset_out) {
  if (!h || !ptr || !handle_out || !offset_out) return MTG_ERR_BAD_ARG;
  DeviceGuard g(h->device);
  typedef CUresult (*RangeFn)(CUdeviceptr*, size_t*, CUdeviceptr);
  static const RangeFn range = []() -> RangeFn {
    void* fp = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &fp, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return nullptr;
    return reinterpret_cast<RangeFn>(fp);
  }();
  if (!range) {
    h->error = "cuMemGetAddressRange is not available from the driver";
    return MTG_ERR_CUDA;
  }
  CUdeviceptr base = 0;
  size_t size = 0;
  if (range(&base, &size, reinterpret_cast<CUdeviceptr>(ptr)) != CUDA_SUCCESS) {
    h->error = "cuMemGetAddressRange failed";
    return MTG_ERR_CUDA;
  }
  cudaIpcMemHandle_t hd;
  MTG_CUDA(h, cudaIpcGetMemHandle(&hd, reinterpret_cast<void*>(base)));
  static_assert(sizeof(hd) == 64, "cudaIpcMemHandle_t is 64 bytes");
  std::memcpy(handle_out, &hd, 64);
  *offset_out = uint64_t(reinterpret_cast<CUdeviceptr>(ptr) - base);
  return MTG_OK;
}

int mtg_ipc_import(mtg_handle* h, const uint8_t handle[64], uint64_t offset, void** ptr_out, void** base_out) {
  if (!h || !handle || !ptr_out || !base_out) return MTG_ERR_BAD_ARG;
  DeviceGuard g(h->device);  // opened with THIS handle's device current: peer access to the owner is enabled lazily
  cudaIpcMemHandle_t hd;
  std::memcpy(&hd, handle, 64);
  void* base = nullptr;
  MTG_CUDA(h, cudaIpcOpenMemHandle(&base, hd, cudaIpcMemLazyEnablePeerAccess));
  *base_out = base;
  *ptr_out = static_cast<char*>(base) + offset;
  return MTG_OK;
}

int mtg_ipc_close(mtg_handle* h, void* base) {
  if (!h || !base) return MTG_ERR_BAD_ARG;
  DeviceGuard g(h->device);
  MTG_CUDA(h, cudaIpcCloseMemHandle(base));
  return MTG_OK;
}

int mtg_stream_synchronize(mtg_handle* h, void* stream) {
  if (!h) return MTG_ERR_BAD_ARG;
  DeviceGuard g(h->device);
  MTG_CUDA(h, cudaStreamSynchronize((cudaStream_t)stream));
  return MTG_OK;
}

}  // extern "C"

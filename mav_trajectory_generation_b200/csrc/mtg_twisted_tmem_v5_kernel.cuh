// mtg_twisted_tmem_v5_kernel.cuh -- K1 (v5): the persistent twisted TMEM kernel with its INPUTS MOVED BY THE TMA.
//
// The whole input record of a 16-trajectory warp tile -- seg_times[16][K] and d_fixed[16][D][n_fixed], two
// contiguous spans of global memory -- is brought into shared memory by one elected lane with two cp.async.bulk
// copies completing on an mbarrier, and every lane then reads its segment times, waypoints and end derivatives
// from shared memory.  For short trajectories (K <= 8) two tiles fit next to the coefficient staging tile and the
// NEXT tile is fetched a whole tile ahead; for longer ones (K = 16: 11.6 KB per tile) one tile fits beside the part
// of the sweep state that overflows tensor memory, and the refill is issued while the last segment of the current
// tile is emitted.  The waypoints are no longer copied into the sweep state (the tile stays resident), which
// shrinks the state to 22 doubles per vertex, and the state is split between TMEM and shared memory slot by slot
// instead of block by block (K = 16: 128 of 154 doubles per lane in TMEM, 26 in shared memory).  Compared with v4 this removes every per-lane global
// load (LDG / LDGSTS: 16 distinct 128-byte lines per warp instruction), the cp.async ring, the time history, the
// prologue prefetch region and their address arithmetic; what is left on the LSU are shared-memory accesses and
// the TMA descriptors.  Requirements (checked by the host, which otherwise launches v4): B a multiple of 16 and
// 16-byte aligned seg_times / d_fixed, so that every tile is a whole, aligned bulk copy.
// Arithmetic per trajectory is the v3/v4 sequence: results are bitwise identical.
#pragma once

#include "mtg_twisted_tmem_v4_kernel.cuh"

namespace mtg {

struct TmemLaunchV5 {
  int tmem_slots;   // sweep-state doubles per lane held in tensor memory (= tmem_cols / 2); the state is split at SLOT
                    // granularity: state double number s (block * 22 + slot at N = 10, D = 3) lives in TMEM when
                    // s < tmem_slots, in shared memory otherwise
  int tmem_cols;
  int n_buffers;    // input tiles per warp: 2 = next tile fetched a whole tile ahead (K <= 12 at N = 10, D = 3), 1 = the
                    // state of longer trajectories leaves room for one tile only: refilled during the outward sweep
                    // (EARLY template parameter) or while the last segment is emitted
  unsigned long long* tile_counter;  // non-null: dynamic tile assignment
};

// sweep state per eliminated vertex: L (strictly lower) + inverse pivots + y  (positions come from the input tile)
__host__ __device__ constexpr int v5_state_slots(int N, int D) {
  return (N / 2 - 1) * (N / 2) / 2 + (N / 2 - 1) * D;
}
// dynamic shared memory: [holder 128][staging x 4 warps][mbarriers 128][input tiles: 4 warps x nbuf x tile][spill]
// [FUSED: segment-time history]; a tile is 16*(K + D*nf) doubles (FUSED: the waypoints, 16*(K+1)*D)
__host__ __device__ constexpr size_t v5_smem_bytes(int N, int D, int K, int nf, int tmem_slots, int nbuf, bool fused) {
  const int nmax = (K + 1) / 2 - 1;
  const int total = nmax * v5_state_slots(N, D);
  const int spill = total > tmem_slots ? total - tmem_slots : 0;
  const size_t tile_doubles = fused ? size_t(16) * (K + 1) * D : size_t(16) * (K + D * nf);
  const size_t stage_bytes_per_warp = size_t(32) * D * (N / 2) * 16;  // tmem_stage_bytes_per_warp<N, D>()
  return size_t(kTmemHeaderBytes) + size_t(kTmemThreads / 32) * stage_bytes_per_warp + 128 +
         size_t(kTmemThreads / 32) * nbuf * tile_doubles * 8 + size_t(spill + (fused ? nmax + 1 : 0)) * kTmemThreads * 8;
}

namespace bulk {
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
// global -> shared bulk copy (bytes a multiple of 16, both addresses 16-byte aligned), completion on `bar`
__device__ __forceinline__ void copy_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
}  // namespace bulk

// EARLY = E > 0 (single tile buffer only): when the outward sweep reaches own vertex E, what its last E steps and the
// closing step still read from the tile ((D+1)*E + D + m*D + 1 doubles per lane) is parked in tensor-memory slots of
// state blocks that are already popped (blocks >= E), and the tile buffer is refilled with the next tile there and
// then: E back-substitution + emission steps of lead for the fetch instead of one.  The host launches this
// instantiation only when n_buffers == 1, both lanes own >= E vertices, and the parking area lies inside tensor memory.
__host__ __device__ constexpr int v5_early_stash_slots(int N, int D, int E) {
  return (D + 1) * E + D + (N / 2 - 1) * D + 1;
}
// lead (outward-sweep steps) of the single-buffer tile refill: measured on C3 / C5-on-one-GPU / K = 14 with E = off, 1, 2, 3,
// 4 -> 0.625 / 0.638 / 0.646 / 0.641 / 0.639 (C3), 0.657 / 0.679 / 0.690 / 0.671 / 0.663 (C5x1)  [tools/early_refill_sweep.py]
constexpr int kV5Early = 2;

// Launch layout of the v5 kernel for one shape: tensor-memory columns, input tile buffers, dynamic shared memory and
// resident CTAs per SM, and whether the early refill's parking area fits (single buffer only).  The host searches it at
// run time (smem_optin of the device, by_regs = CTAs per SM the kernel's registers allow); the compile-time-shape
// instantiations (KC > 0) are compiled for the result of the same search at the B200's budget.
struct V5Layout {
  int ctas = 0, cols = 0, nbuf = 0;
  size_t smem = 0;
  bool early_fits = false;
};
__host__ __device__ constexpr V5Layout v5_layout(int N, int D, int K, int nf, bool fused, size_t smem_optin, int by_regs) {
  const int nmax = (K + 1) / 2 - 1;
  V5Layout best{};
  const int col_options[] = {256, 128, 64, 32, 512};
  for (int nbuf = 2; nbuf >= 1; --nbuf)
    for (int cols : col_options) {
      const size_t smem = v5_smem_bytes(N, D, K, nf, cols / 2, nbuf, fused);
      if (smem > smem_optin) continue;
      int ctas = int((228 * 1024) / (smem + 1024));
      ctas = by_regs < ctas ? by_regs : ctas;
      ctas = 512 / cols < ctas ? 512 / cols : ctas;
      ctas = ctas < 8 ? ctas : 8;
      // more resident CTAs first; then double buffering; then less shared memory
      if (ctas > best.ctas ||
          (ctas == best.ctas && ctas > 0 && (nbuf > best.nbuf || (nbuf == best.nbuf && smem < best.smem)))) {
        best.ctas = ctas;
        best.cols = cols;
        best.nbuf = nbuf;
        best.smem = smem;
      }
    }
  // early refill: both lanes must own >= E vertices and the parking area must lie in tensor memory behind the state
  // blocks still needed
  const int own_min = K - (K + 1) / 2 - 1;
  best.early_fits = best.nbuf == 1 && kV5Early <= own_min && kV5Early <= nmax &&
                    kV5Early * v5_state_slots(N, D) + v5_early_stash_slots(N, D, kV5Early) <= best.cols / 2;
  return best;
}
// the layout a compile-time-shape instantiation is built for: waypoint constraints (n_fixed = K + N - 1), the B200's
// 227 KB of opt-in shared memory per block, and the CTAs per SM its __launch_bounds__ guarantee
constexpr size_t kV5StaticSmemOptin = 227 * 1024;
template <int N, int D, int MINB, int KC>
__host__ __device__ constexpr V5Layout v5_static_layout() {
  return v5_layout(N, D, KC, KC + N - 1, false, kV5StaticSmemOptin, MINB);
}

// KC > 0: the instantiation for K = KC segments (waypoint constraints, no FUSED) and the launch layout
// v5_static_layout<N, D, MINB, KC>(), which the host launches only when its run-time layout is that one.  Every shape
// quantity is then a compile-time constant: loop trip counts, tile offsets, the TMEM / shared-memory split test of each
// state slot, and the warp-uniform `v <= nh` tests, which vanish (K even: both lanes own K/2 - 1 vertices).
// The arithmetic is the same expressions in the same order: results are bitwise identical to KC = 0.
template <int N, int R, int D, int MINB, bool FUSED = false, int EARLY = 0, int KC = 0>
__global__ void __launch_bounds__(kTmemThreads, MINB)
    twisted_tmem_v5_kernel(const WaypointParams prm, const TmemLaunchV5 tl, const __grid_constant__ CUtensorMap tmap) {
  static_assert(KC == 0 || (!FUSED && KC % 2 == 0 && KC >= 4), "compile-time shapes: waypoint inputs, even K >= 4");
  constexpr V5Layout kS = KC > 0 ? v5_static_layout<N, D, MINB, KC>() : V5Layout{};
  static_assert(KC == 0 || (kS.ctas >= 2 && EARLY == (kS.early_fits ? kV5Early : 0)),
                "compile-time shape without a v5 layout, or EARLY differs from the layout's");
  constexpr int h = N / 2;
  constexpr int m = h - 1;
  constexpr int kL = m * (m + 1) / 2;
  constexpr int kSlots = kL + m * D;  // no positions in the state: the input tile stays resident for the whole tile
  constexpr int kWords = 2 * kSlots;
  constexpr unsigned kFull = 0xffffffffu;
  constexpr int kWarps = kTmemThreads / 32;
  constexpr double kTiny = 0x1p-600, kHuge = 0x1p+600;
  using G = H1Imm<N, R>;
  using AI = A1InvImm<N>;

  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int half = lane & 1;
  const int K = KC > 0 ? KC : prm.K;
  const int nf = KC > 0 ? KC + N - 1 : prm.n_fixed;
  const int M = (K + 1) >> 1;
  const int nh = half ? K - M - 1 : M - 1;
  const int nmax = M - 1;
  const int tslots = KC > 0 ? kS.cols / 2 : tl.tmem_slots;
  const int tcols = KC > 0 ? kS.cols : tl.tmem_cols;
  const int nbuf = KC > 0 ? kS.nbuf : tl.n_buffers;

  uint32_t* holder = reinterpret_cast<uint32_t*>(smem_raw);
  double2* stage = reinterpret_cast<double2*>(smem_raw + kTmemHeaderBytes) + size_t(warp) * 32 * (D * h);
  unsigned char* after_stage = smem_raw + kTmemHeaderBytes + size_t(kWarps) * tmem_stage_bytes_per_warp<N, D>();
  const uint32_t bar0 = tmem::smem_u32(after_stage) + uint32_t(warp) * 16;  // two 8-byte mbarriers per warp
  // FUSED (SURVEY.md 8f-1): the tile is the waypoint record positions[16][K+1][D]; segment times are computed from it
  // (estimateSegmentTimesNfabian) and kept in a small per-thread history for the outward sweep
  const int tile_t = FUSED ? 0 : 16 * K, tile_f = FUSED ? 16 * (K + 1) * D : 16 * D * nf, tile_doubles = tile_t + tile_f;
  double* tiles = reinterpret_cast<double*>(after_stage + 128) + size_t(warp) * nbuf * tile_doubles;
  double* spill = reinterpret_cast<double*>(after_stage + 128) + size_t(kWarps) * nbuf * tile_doubles + threadIdx.x;
  double* thist = nullptr;  // FUSED only: behind the spilled state
  if constexpr (FUSED) {
    const int total_state = nmax * kSlots;
    thist = spill + size_t(total_state > tslots ? total_state - tslots : 0) * kTmemThreads;
  }
  auto TH = [&](int j) -> double& { return thist[size_t(j) * kTmemThreads]; };
  auto SPG = [&](int s_global) -> double& { return spill[size_t(s_global - tslots) * kTmemThreads]; };

  uint32_t tbase = 0;
  if (tcols > 0) {
    if (warp == 0) tmem::alloc(tmem::smem_u32(holder), (uint32_t)tcols);
    tmem::fence_before_sync();
    __syncthreads();
    tmem::fence_after_sync();
    tbase = *holder + (uint32_t(warp * 32) << 16);
  }
  // State block `blk` occupies state doubles [blk*kSlots, (blk+1)*kSlots): entirely in TMEM, entirely in shared
  // memory, or -- for the one block that straddles tmem_slots -- split slot by slot (all tests are warp-uniform).
  auto put_state = [&](int blk, const double (&sv)[kSlots]) {
    const int s0 = blk * kSlots;
    if (s0 + kSlots <= tslots) {
#pragma unroll
      for (int i = 0; i < kSlots; ++i) {
        const uint32_t w[2] = {(uint32_t)__double2loint(sv[i]), (uint32_t)__double2hiint(sv[i])};
        tmem::st<2>(tbase + uint32_t(2 * (s0 + i)), w);
      }
    } else if (s0 >= tslots) {
#pragma unroll
      for (int i = 0; i < kSlots; ++i) SPG(s0 + i) = sv[i];
    } else {
#pragma unroll
      for (int i = 0; i < kSlots; ++i) {
        if (s0 + i < tslots) {
          const uint32_t w[2] = {(uint32_t)__double2loint(sv[i]), (uint32_t)__double2hiint(sv[i])};
          tmem::st<2>(tbase + uint32_t(2 * (s0 + i)), w);
        } else {
          SPG(s0 + i) = sv[i];
        }
      }
    }
  };
  auto get_state = [&](int blk, double (&sv)[kSlots]) {
    const int s0 = blk * kSlots;
    if (s0 + kSlots <= tslots) {
      uint32_t w[kWords];
      tmem::ld_words<kWords>(tbase + uint32_t(2 * s0), w);
      tmem::wait_ld();
#pragma unroll
      for (int i = 0; i < kSlots; ++i) sv[i] = __hiloint2double((int)w[2 * i + 1], (int)w[2 * i]);
    } else if (s0 >= tslots) {
#pragma unroll
      for (int i = 0; i < kSlots; ++i) sv[i] = SPG(s0 + i);
    } else {
      uint32_t w[kWords];
#pragma unroll
      for (int i = 0; i < kSlots; ++i)
        if (s0 + i < tslots) tmem::ld<2>(tbase + uint32_t(2 * (s0 + i)), &w[2 * i]);
      tmem::wait_ld();
#pragma unroll
      for (int i = 0; i < kSlots; ++i)
        sv[i] = (s0 + i < tslots) ? __hiloint2double((int)w[2 * i + 1], (int)w[2 * i]) : SPG(s0 + i);
    }
  };

  auto seg = [&](int j) -> int { return half ? K - 1 - j : j; };
  auto pidx = [&](int v) -> int {
    const int o = half ? K - v : v;
    return o == 0 ? 0 : (o < K ? h + o - 1 : h + K - 1);
  };
  auto sgn = [&](int idx) -> double { return (half && !(idx & 1)) ? -1.0 : 1.0; };
  const int e0 = half ? h + K : 1;

  const long long n_wtiles = prm.B >> 4;  // B is a multiple of 16 (host-checked)
  const long long wt_stride = (long long)gridDim.x * kWarps;
  const bool dyn = tl.tile_counter != nullptr;
  // Dynamic assignment: the FIRST tile of every warp is its static one (no atomic in front of the first fetch); the
  // counter hands out the tiles after those, and is always drawn one tile ahead of its use so that the atomic's
  // round trip to L2 never sits in front of a fetch.
  // (inline PTX: the compiler turns atomicAdd() under `lane == 0` into its warp-aggregated form, ATOMG followed at once
  // by a SHFL of the result -- which puts the round trip back in front of the warp: 2.4 % of all stall samples)
  auto draw_tile = [&]() -> long long {
    unsigned long long old = 0;
    if (lane == 0) asm volatile("atom.global.add.u64 %0, [%1], 1;" : "=l"(old) : "l"(tl.tile_counter) : "memory");
    return (long long)old + wt_stride;
  };
  long long wt = (long long)blockIdx.x * kWarps + warp;
  long long pending = dyn ? draw_tile() : 0;  // lane 0 holds the tile after `wt`

  // one elected lane moves a whole tile: seg_times[16][K] and d_fixed[16][D][nf] are contiguous in global memory
  if (lane == 0) {
    bulk::mbar_init(bar0, 1);
    bulk::mbar_init(bar0 + 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  auto fetch_tile = [&](long long w, int buf) {
    if (lane == 0) {
      const uint32_t bar = bar0 + 8u * buf;
      double* dst = tiles + size_t(buf) * tile_doubles;
      bulk::mbar_expect_tx(bar, uint32_t(tile_doubles) * 8u);
      if constexpr (FUSED) {
        bulk::copy_g2s(tmem::smem_u32(dst), prm.positions + w * 16 * (long long)(K + 1) * D, uint32_t(tile_f) * 8u, bar);
      } else {
        bulk::copy_g2s(tmem::smem_u32(dst), prm.times + w * 16 * K, uint32_t(tile_t) * 8u, bar);
        bulk::copy_g2s(tmem::smem_u32(dst + tile_t), prm.dfix + w * 16 * (long long)D * nf, uint32_t(tile_f) * 8u, bar);
      }
    }
  };
  if (wt < n_wtiles) fetch_tile(wt, 0);

  double2* my_row = stage + ((lane & 1) * 16 + (lane >> 1)) * (D * h);
  const int nhF = M - 1, nhB = K - M - 1;
  const int tl_row = lane >> 1;  // this lane's trajectory inside the tile

  for (int it = 0; wt < n_wtiles; ++it) {
    const int buf = nbuf == 2 ? (it & 1) : 0;
    long long wt_next = dyn ? __shfl_sync(kFull, pending, 0) : wt + wt_stride;
    if (dyn) pending = draw_tile();
    if (nbuf == 2) {
      // fetch the next tile into the other buffer now: a whole tile of lead.  That buffer was read (generic proxy) by
      // the previous tile; order those reads before the asynchronous-proxy write.
      fence_proxy_async();
      __syncwarp();
      if (wt_next < n_wtiles) fetch_tile(wt_next, buf ^ 1);
    }
    bulk::mbar_wait(bar0 + 8u * buf, nbuf == 2 ? (uint32_t(it >> 1) & 1u) : (uint32_t(it) & 1u));

    const double* __restrict__ tT = tiles + size_t(buf) * tile_doubles + tl_row * K;
    const double* __restrict__ tF =
        tiles + size_t(buf) * tile_doubles + tile_t + tl_row * (FUSED ? (K + 1) * D : D * nf);
    // KC > 0: own segment j and own interior vertex v (1 <= v <= K - 1) are at a per-lane base pointer plus a +-1 stride
    // (the mirrored lane walks the tile backwards) instead of a mirrored index selected at every read
    const int dir = half ? -1 : 1;
    const double* tTj = tT + (half ? K - 1 : 0);
    const double* tXv = tF + (half ? h + K - 1 : h - 1);
    const double* tX0 = tF + (half ? h + K - 1 : 0);
    // time of own segment j: from the tile, or (FUSED) from the history filled by the inward sweep
    auto in_T = [&](int j) -> double {
      if constexpr (FUSED) return TH(j);
      if constexpr (KC > 0) return tTj[dir * j];
      return tT[seg(j)];
    };
    auto in_x = [&](int v, int d) -> double {
      if constexpr (FUSED) return tF[(half ? K - v : v) * D + d];
      if constexpr (KC > 0) return v == 0 ? tX0[d * nf] : tXv[d * nf + dir * v];
      return tF[d * nf + pidx(v)];
    };
    auto in_u0 = [&](int b, int d) -> double {  // fixed end derivative b+1 of own vertex 0, own-frame sign
      if constexpr (FUSED) return 0.0;
      return sgn(b) * tF[d * nf + e0 + b];
    };
    const long long traj0 = wt * 16;
    const long long traj = traj0 + tl_row;

    // emit own-frame segment j for every lane of the warp at once (convergent)
    auto emit_all = [&](int j, int v_step, double T, double iT, const double (&sd)[h][D], const double (&ed)[h][D]) {
      double tp[h], itp[h];
      const double Ts = half ? -T : T;
      tp[0] = 1.0;
#pragma unroll
      for (int k = 1; k < h; ++k) tp[k] = tp[k - 1] * Ts;
      itp[0] = pow_int<h>(iT);
#pragma unroll
      for (int k = 1; k < h; ++k) itp[k] = itp[k - 1] * iT;
#pragma unroll
      for (int d = 0; d < D; ++d) {
        double c[N], ss[h], se[h];
#pragma unroll
        for (int k = 0; k < h; ++k) {
          const double s0 = half ? ed[k][d] : sd[k][d];
          const double e0v = half ? sd[k][d] : ed[k][d];
          c[k] = s0 * ((half && (k & 1)) ? -AI::at(k, k) : AI::at(k, k));
          ss[k] = tp[k] * s0;
          se[k] = tp[k] * e0v;
        }
        double ee[h];
#pragma unroll
        for (int k = 0; k < h; ++k) {
          double acc = se[k] - ss[k];
#pragma unroll
          for (int j2 = k + 1; j2 < h; ++j2) {
            constexpr double kInvFact[6] = {1.0, 1.0, 0.5, 1.0 / 6.0, 1.0 / 24.0, 1.0 / 120.0};
            acc = (j2 - k == 1) ? acc - ss[j2] : fma(-kInvFact[j2 - k], ss[j2], acc);
          }
          ee[k] = acc;
        }
#pragma unroll
        for (int q = 0; q < h; ++q) {
          double acc = AI::at(h + q, h) * ee[0];
#pragma unroll
          for (int k = 1; k < h; ++k) acc = fma(AI::at(h + q, h + k), ee[k], acc);
          c[h + q] = acc * itp[q];
        }
        if (d == 0) {  // the TMA must have finished reading the previous segment's tile
          if (lane == 0) bulk_wait_read();
          __syncwarp();
        }
#pragma unroll
        for (int q = 0; q < h; ++q) my_row[d * h + q] = make_double2(c[2 * q], c[2 * q + 1]);
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        if (v_step <= nhF) tma_store_box(&tmap, stage, j * (D * N), (int)traj0);
        if (v_step <= nhB) tma_store_box(&tmap, stage + 16 * (D * h), (K - 1 - j) * (D * N), (int)traj0);
        bulk_commit();
      }
    };


    int stat = 0;
    double Wp[m][m], yp[m][D], Cee[m][m], cps[m], cpe[m], xm[D], xc[D];
    {
#pragma unroll
      for (int d = 0; d < D; ++d) {
        xm[d] = in_x(0, d);
        xc[d] = in_x(1, d);
      }
      double T0;
      if constexpr (FUSED) {
        T0 = nfabian_time<D>(xm, xc, prm.v_max, prm.a_max, prm.magic);
        TH(0) = T0;
      } else {
        T0 = in_T(0);
      }
      if (!(T0 > 0.0)) stat |= kStatusBadTime;
      const double iT0 = fast_rcp(T0);
      double pw[N - 1];
      segment_powers<N, R>(T0, iT0, pw);
#pragma unroll
      for (int a = 0; a < m; ++a) {
#pragma unroll
        for (int b = 0; b < m; ++b) {
          Cee[a][b] = pw[a + b + 2] * G::at(h + 1 + a, h + 1 + b);
          Wp[a][b] = (a == b) ? kTiny : 0.0;
        }
        cps[a] = pw[a + 1] * G::at(h + 1 + a, 0);
        cpe[a] = pw[a + 1] * G::at(h + 1 + a, h);
      }
#pragma unroll
      for (int d = 0; d < D; ++d) {
        double u0[m];
#pragma unroll
        for (int b = 0; b < m; ++b) u0[b] = in_u0(b, d);
#pragma unroll
        for (int a = 0; a < m; ++a) {
          double acc = 0.0;
#pragma unroll
          for (int b = 0; b < m; ++b) acc = fma(pw[a + b + 2] * G::at(h + 1 + a, 1 + b), u0[b], acc);
          yp[a][d] = acc * kHuge;
        }
      }
    }

    // ---------------------------------------------------------------- sweep towards the middle
    // The vertex loops stay rolled also at a compile-time trip count (KC > 0): on C5 the KC = 16 kernel gains 15 % over
    // the run-time kernel rolled (2 250 instructions), 7 % unrolled by two (4 080) and 4 % unrolled fully (7 300)
    // (profiles/r03_v5_static_shape_variants.log): the unrolled code no longer fits the instruction caches.
#pragma unroll 1
    for (int v = 1; v <= nmax; ++v) {
      double sv[kSlots];
      if (v <= nh) {
        double xn[D];
#pragma unroll
        for (int d = 0; d < D; ++d) xn[d] = in_x(v + 1, d);
        double T;
        if constexpr (FUSED) {
          T = nfabian_time<D>(xc, xn, prm.v_max, prm.a_max, prm.magic);
          TH(v) = T;
        } else {
          T = in_T(v);
        }
        if (!(T > 0.0)) stat |= kStatusBadTime;
        const double iT = fast_rcp(T);
        double pw[N - 1];
        segment_powers<N, R>(T, iT, pw);

        double Dp[m][m], E[m][m], bb[m][D];
#pragma unroll
        for (int a = 0; a < m; ++a) {
#pragma unroll
          for (int b = 0; b <= a; ++b) {
            double s = fma(pw[a + b + 2], G::at(1 + a, 1 + b), Cee[a][b]);
#pragma unroll
            for (int k = 0; k < m; ++k) s = fma(-Wp[k][a], Wp[k][b], s);
            Dp[a][b] = s;
          }
#pragma unroll
          for (int b = 0; b < m; ++b) E[a][b] = pw[a + b + 2] * G::at(1 + a, h + 1 + b);
          const double gmid = fma(pw[a + 1], G::at(1 + a, 0), cpe[a]);
          const double gnext = pw[a + 1] * G::at(1 + a, h);
#pragma unroll
          for (int d = 0; d < D; ++d) {
            double s = -cps[a] * xm[d];
            s = fma(-gmid, xc[d], s);
            s = fma(-gnext, xn[d], s);
#pragma unroll
            for (int k = 0; k < m; ++k) s = fma(-Wp[k][a], yp[k][d], s);
            bb[a][d] = s;
          }
        }
        double L[m][m], inv[m];
#pragma unroll
        for (int j = 0; j < m; ++j) {
          double s = Dp[j][j];
#pragma unroll
          for (int k = 0; k < j; ++k) s = fma(-L[j][k], L[j][k], s);
          if (!(s > 0.0)) stat |= kStatusNotSpd;
          inv[j] = fast_rsqrt(s);
#pragma unroll
          for (int i = j + 1; i < m; ++i) {
            double t = Dp[i][j];
#pragma unroll
            for (int k = 0; k < j; ++k) t = fma(-L[i][k], L[j][k], t);
            L[i][j] = t * inv[j];
          }
        }
#pragma unroll
        for (int d = 0; d < D; ++d) {
#pragma unroll
          for (int j = 0; j < m; ++j) {
            double s = bb[j][d];
#pragma unroll
            for (int k = 0; k < j; ++k) s = fma(-L[j][k], yp[k][d], s);
            yp[j][d] = s * inv[j];
          }
        }
#pragma unroll
        for (int c = 0; c < m; ++c) {
#pragma unroll
          for (int j = 0; j < m; ++j) {
            double s = E[j][c];
#pragma unroll
            for (int k = 0; k < j; ++k) s = fma(-L[j][k], Wp[k][c], s);
            Wp[j][c] = s * inv[j];
          }
        }
        {
          int slot = 0;
#pragma unroll
          for (int i = 1; i < m; ++i)
#pragma unroll
            for (int j = 0; j < i; ++j) sv[slot++] = L[i][j];
#pragma unroll
          for (int j = 0; j < m; ++j) sv[slot++] = inv[j];
#pragma unroll
          for (int j = 0; j < m; ++j)
#pragma unroll
            for (int d = 0; d < D; ++d) sv[slot++] = yp[j][d];
        }
#pragma unroll
        for (int a = 0; a < m; ++a) {
#pragma unroll
          for (int b = 0; b <= a; ++b) Cee[a][b] = pw[a + b + 2] * G::at(h + 1 + a, h + 1 + b);
          cps[a] = pw[a + 1] * G::at(h + 1 + a, 0);
          cpe[a] = pw[a + 1] * G::at(h + 1 + a, h);
        }
#pragma unroll
        for (int d = 0; d < D; ++d) {
          xm[d] = xc[d];
          xc[d] = xn[d];
        }
      }
      __syncwarp();
      put_state(v - 1, sv);
    }
    __syncwarp();
    if (tslots > 0) tmem::wait_st();

    // ---------------------------------------------------------------- middle vertex
    double um[m][D];
    {
      double Dl[m][m], bl[m][D];
#pragma unroll
      for (int a = 0; a < m; ++a) {
#pragma unroll
        for (int b = 0; b <= a; ++b) {
          double s = Cee[a][b];
#pragma unroll
          for (int k = 0; k < m; ++k) s = fma(-Wp[k][a], Wp[k][b], s);
          Dl[a][b] = s;
        }
#pragma unroll
        for (int d = 0; d < D; ++d) {
          double s = -cps[a] * xm[d];
          s = fma(-cpe[a], xc[d], s);
#pragma unroll
          for (int k = 0; k < m; ++k) s = fma(-Wp[k][a], yp[k][d], s);
          bl[a][d] = s;
        }
      }
#pragma unroll
      for (int a = 0; a < m; ++a) {
#pragma unroll
        for (int b = 0; b <= a; ++b) {
          const double o = __shfl_xor_sync(kFull, Dl[a][b], 1);
          Dl[a][b] += ((a + b) & 1) ? -o : o;
        }
#pragma unroll
        for (int d = 0; d < D; ++d) {
          const double o = __shfl_xor_sync(kFull, bl[a][d], 1);
          bl[a][d] += (a & 1) ? o : -o;
        }
      }
      stat |= __shfl_xor_sync(kFull, stat, 1);
      double L[m][m], inv[m];
#pragma unroll
      for (int j = 0; j < m; ++j) {
        double s = Dl[j][j];
#pragma unroll
        for (int k = 0; k < j; ++k) s = fma(-L[j][k], L[j][k], s);
        if (!(s > 0.0)) stat |= kStatusNotSpd;
        inv[j] = fast_rsqrt(s);
#pragma unroll
        for (int i = j + 1; i < m; ++i) {
          double t = Dl[i][j];
#pragma unroll
          for (int k = 0; k < j; ++k) t = fma(-L[i][k], L[j][k], t);
          L[i][j] = t * inv[j];
        }
      }
#pragma unroll
      for (int d = 0; d < D; ++d) {
        double y[m];
#pragma unroll
        for (int j = 0; j < m; ++j) {
          double s = bl[j][d];
#pragma unroll
          for (int k = 0; k < j; ++k) s = fma(-L[j][k], y[k], s);
          y[j] = s * inv[j];
        }
#pragma unroll
        for (int j = m - 1; j >= 0; --j) {
          double s = y[j];
#pragma unroll
          for (int k = j + 1; k < m; ++k) s = fma(-L[k][j], um[k][d], s);
          um[j][d] = s * inv[j];
        }
      }
    }
    if (half == 0 && prm.status != nullptr) prm.status[traj] = stat;

    // ---------------------------------------------------------------- outward back-substitution
    const int np = (K - 1) * m;
    double* __restrict__ df = prm.dfree != nullptr ? prm.dfree + traj * (long long)D * np : nullptr;
    auto store_free = [&](int v_own, const double (&u)[h][D]) {
      if (df != nullptr) {
        const int vo = half ? K - v_own : v_own;
#pragma unroll
        for (int d = 0; d < D; ++d)
#pragma unroll
          for (int j = 0; j < m; ++j) df[d * np + (vo - 1) * m + j] = sgn(j) * u[1 + j][d];
      }
    };

    double ed[h][D];
#pragma unroll
    for (int d = 0; d < D; ++d) {
      ed[0][d] = xc[d];
#pragma unroll
      for (int j = 0; j < m; ++j) ed[1 + j][d] = um[j][d];
    }
    if (half == 0) store_free(nh + 1, ed);

    constexpr int kStash0 = EARLY * kSlots;  // state slots of the blocks >= EARLY: popped when the sweep reaches vertex EARLY
    auto park = [&](int slot, double val) {
      const uint32_t w[2] = {(uint32_t)__double2loint(val), (uint32_t)__double2hiint(val)};
      tmem::st<2>(tbase + uint32_t(2 * (kStash0 + slot)), w);
    };
#pragma unroll 1
    for (int v = nmax; v >= 1; --v) {
      if constexpr (EARLY > 0) {
        if (v == EARLY) {
          // park what steps EARLY..1 and the closing step read from the tile, then refill the tile buffer now
#pragma unroll
          for (int u = EARLY; u >= 1; --u) {
#pragma unroll
            for (int d = 0; d < D; ++d) park((EARLY - u) * (D + 1) + d, in_x(u, d));
            park((EARLY - u) * (D + 1) + D, in_T(u));
          }
#pragma unroll
          for (int d = 0; d < D; ++d) park(EARLY * (D + 1) + d, in_x(0, d));
#pragma unroll
          for (int d = 0; d < D; ++d)
#pragma unroll
            for (int b = 0; b < m; ++b) park(EARLY * (D + 1) + D + d * m + b, in_u0(b, d));
          park(EARLY * (D + 1) + D + m * D, in_T(0));
          tmem::wait_st();
          fence_proxy_async();
          __syncwarp();
          if (wt_next < n_wtiles) fetch_tile(wt_next, 0);
        }
      }
      double sv[kSlots];
      get_state(v - 1, sv);
      const bool act = v <= nh;
      double T = 1.0, iT = 1.0;
      double sd[h][D];
      if (act) {
        double xv[D];
        if (EARLY > 0 && v <= EARLY) {
          uint32_t w[2 * (D + 1)];
          tmem::ld_words<2 * (D + 1)>(tbase + uint32_t(2 * (kStash0 + (EARLY - v) * (D + 1))), w);
          tmem::wait_ld();
#pragma unroll
          for (int d = 0; d < D; ++d) xv[d] = __hiloint2double((int)w[2 * d + 1], (int)w[2 * d]);
          T = __hiloint2double((int)w[2 * D + 1], (int)w[2 * D]);
        } else {
#pragma unroll
          for (int d = 0; d < D; ++d) xv[d] = in_x(v, d);
          T = in_T(v);
        }
        if constexpr (FUSED) {
          if (prm.times_out != nullptr) prm.times_out[traj * K + seg(v)] = T;
        }
        iT = fast_rcp(T);
        double pw[N - 1];
        segment_powers<N, R>(T, iT, pw);
        double tE[m][D];
#pragma unroll
        for (int d = 0; d < D; ++d)
#pragma unroll
          for (int a = 0; a < m; ++a) {
            double s = 0.0;
#pragma unroll
            for (int b = 0; b < m; ++b) s = fma(pw[a + b + 2] * G::at(1 + a, h + 1 + b), ed[1 + b][d], s);
            tE[a][d] = s;
          }
        double L[m][m], inv[m], rhs[m][D];
        {
          int slot = 0;
#pragma unroll
          for (int i = 1; i < m; ++i)
#pragma unroll
            for (int j = 0; j < i; ++j) L[i][j] = sv[slot++];
#pragma unroll
          for (int j = 0; j < m; ++j) inv[j] = sv[slot++];
#pragma unroll
          for (int j = 0; j < m; ++j)
#pragma unroll
            for (int d = 0; d < D; ++d) rhs[j][d] = sv[slot++];
        }
#pragma unroll
        for (int d = 0; d < D; ++d) {
          double t[m];
#pragma unroll
          for (int j = 0; j < m; ++j) {
            double s = tE[j][d];
#pragma unroll
            for (int k = 0; k < j; ++k) s = fma(-L[j][k], t[k], s);
            t[j] = s * inv[j];
            rhs[j][d] -= t[j];
          }
        }
#pragma unroll
        for (int d = 0; d < D; ++d) {
#pragma unroll
          for (int j = m - 1; j >= 0; --j) {
            double s = rhs[j][d];
#pragma unroll
            for (int k = j + 1; k < m; ++k) s = fma(-L[k][j], sd[1 + k][d], s);
            sd[1 + j][d] = s * inv[j];
          }
          sd[0][d] = xv[d];
        }
        store_free(v, sd);
      }
      __syncwarp();
      emit_all(v, v, T, iT, sd, ed);
      if (act) {
#pragma unroll
        for (int d = 0; d < D; ++d)
#pragma unroll
          for (int k = 0; k < h; ++k) ed[k][d] = sd[k][d];
      }
    }
    {
      double sd[h][D];
      double T;
      if constexpr (EARLY > 0) {
        constexpr int kClose = D + m * D + 1;
        uint32_t w[2 * kClose];
        tmem::ld_words<2 * kClose>(tbase + uint32_t(2 * (kStash0 + EARLY * (D + 1))), w);
        tmem::wait_ld();
#pragma unroll
        for (int d = 0; d < D; ++d) {
          sd[0][d] = __hiloint2double((int)w[2 * d + 1], (int)w[2 * d]);
#pragma unroll
          for (int b = 0; b < m; ++b)
            sd[1 + b][d] = __hiloint2double((int)w[2 * (D + d * m + b) + 1], (int)w[2 * (D + d * m + b)]);
        }
        T = __hiloint2double((int)w[2 * (kClose - 1) + 1], (int)w[2 * (kClose - 1)]);
      } else {
#pragma unroll
        for (int d = 0; d < D; ++d) {
          sd[0][d] = in_x(0, d);
#pragma unroll
          for (int b = 0; b < m; ++b) sd[1 + b][d] = in_u0(b, d);
        }
        T = in_T(0);
      }
      if constexpr (FUSED) {
        if (prm.times_out != nullptr) prm.times_out[traj * K + seg(0)] = T;
      }
      const double iT = fast_rcp(T);
      if (EARLY == 0 && nbuf == 1) {
        // single buffer: every input of this tile is in registers now -- refill it with the next tile while the last
        // segment is emitted
        fence_proxy_async();
        __syncwarp();
        if (wt_next < n_wtiles) fetch_tile(wt_next, 0);
      }
      __syncwarp();
      emit_all(0, 0, T, iT, sd, ed);
    }
    wt = wt_next;
  }

  if (lane == 0) bulk_wait_all();
  if (tcols > 0) {
    tmem::fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem::dealloc(*holder, (uint32_t)tcols);
  }
}

}  // namespace mtg

// engine.cuh -- what the translation units of libecdna_b200.so share: the context, the launch planner
// and the launch templates.  The kernel is instantiated per tile width in its own .cu file (ssa_l1.cu ..
// ssa_l32.cu, ssa_hbm.cu) so that the widths compile in parallel; capi.cu holds the C ABI.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "ssa_kernel.cuh"

namespace ecdna {

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes, bool zero_new = false) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) return e;
    cap = bytes;
    if (zero_new) e = cudaMemset(p, 0, bytes);
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

// the per-run result columns, in the order of ecdna_b200_results_t
enum Col {
  C_STOP, C_NMINUS, C_NPLUS, C_TIME, C_NEVENTS, C_KMAX, C_MEAN, C_FREQ, C_ENT, C_VAR, C_ABCD, C_ABCA, C_HASH,
  C_CHAIN, C_HIST, C_SNAPCOUNT, C_SNAPCELLS, C_SNAPTIME, C_SNAPHIST, C_DYNCOUNT, C_DYN, C_SUMK, C_NDIV, C_NDEATH,
  C_SUBHIST, C_COUNT
};

// layout of the 128-byte counter block in HBM
constexpr size_t kTotalsOffset = 16;  // 8 x u64 (SsaArgs::totals)
constexpr int kTotalsCount = 8;
constexpr size_t kRingCtrOffset = 96;  // 4 x u32 (SsaArgs::ts_ctr)

}  // namespace ecdna

struct ecdna_b200_comm;  // abc_gather.cu

struct ecdna_b200_ctx {
  int device = 0;
  ecdna_b200_comm* comm = nullptr;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev_begin = nullptr, ev_k0 = nullptr, ev_k1 = nullptr, ev_end = nullptr;
  bool have_total = false;
  uint64_t expect_finished = 0;  // replicates the last run must have finished (checked in get_timing / run)
  std::string err;
  ecdna::DevBuf init_k, init_c, snap, rates, replay, replay_off, abc_cdf, arena, counters, scratch, park_list, park_rec,
      park_list2, park_rec2, order, order_hist, cells, zig, ts_ring, ts_rec, sub_sizes, hist_tmp, pack_idx, pack_out, pack_cnt,
      sp_desc, sp_len, sp_bsum, sp_arena, smc_prev, smc_cum, smc_new, smc_parent, smc_tiles, smc_sum, smc_cov,
      cols[ecdna::C_COUNT];
  // the packed batch the last ecdna_b200_run_sparse left on the device (sparse.cuh)
  struct {
    bool valid = false, packed = false;
    uint64_t n_runs = 0, n_snap = 0, n_sub = 0, rows = 0, words = 0;
    uint32_t stride = 0;
  } sp;
  size_t arena_words = 0, arena_kcap = 0;
  ecdna_b200_timing_t timing{};
};

// several GPUs of one process (multi.cu); the ABC-SMC driver (abc_smc.cu) runs its proposals on the first one
struct ecdna_b200_multi {
  std::vector<ecdna_b200_ctx*> ctx;
  std::vector<uint64_t> last_begin, last_count;
  std::vector<uint64_t> sp_words;  // arena words of every GPU's block of the last sparse run
  uint64_t sp_snap = 0, sp_sub = 0;
  bool sp_valid = false;
  std::string err;
};

namespace ecdna {

inline int fail(ecdna_b200_ctx* ctx, int code, const std::string& msg) {
  if (ctx) ctx->err = msg;
  return code;
}
#define CU(call)                                                                                  \
  do {                                                                                            \
    cudaError_t e__ = (call);                                                                     \
    if (e__ != cudaSuccess)                                                                       \
      return fail(ctx, ECDNA_B200_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); \
  } while (0)

// bytes per replicate of result column c, and the column's pointer inside the results struct
inline size_t col_bytes(int c, const ecdna_b200_params_t* p, uint32_t stride) {
  switch (c) {
    case C_STOP: case C_KMAX: case C_SNAPCOUNT: case C_DYNCOUNT: case C_NDIV: case C_NDEATH: return 4;
    case C_NMINUS: case C_NPLUS: case C_NEVENTS: case C_HASH: case C_CHAIN: case C_SUMK: return 8;
    case C_TIME: case C_MEAN: case C_FREQ: case C_ENT: case C_VAR: return 4;
    case C_ABCD: return 16;
    case C_ABCA: return 1;
    case C_HIST: return (size_t)stride * 4;
    case C_SNAPCELLS: return (size_t)p->n_snapshots * 8;
    case C_SNAPTIME: return (size_t)p->n_snapshots * 4;
    case C_SNAPHIST: return (size_t)p->n_snapshots * stride * 4;
    case C_DYN: return (size_t)p->dyn_points * 5 * 4;
    case C_SUBHIST: return (size_t)p->n_subsamples * stride * 4;
  }
  return 0;
}
inline void** col_slot(ecdna_b200_results_t* r, int c) {
  switch (c) {
    case C_STOP: return (void**)&r->stop_reason;
    case C_NMINUS: return (void**)&r->nminus;
    case C_NPLUS: return (void**)&r->nplus;
    case C_TIME: return (void**)&r->time;
    case C_NEVENTS: return (void**)&r->n_events;
    case C_KMAX: return (void**)&r->kmax;
    case C_MEAN: return (void**)&r->mean;
    case C_FREQ: return (void**)&r->frequency;
    case C_ENT: return (void**)&r->entropy;
    case C_VAR: return (void**)&r->variance;
    case C_ABCD: return (void**)&r->abc_distance;
    case C_ABCA: return (void**)&r->abc_accept;
    case C_HASH: return (void**)&r->hash;
    case C_CHAIN: return (void**)&r->chain;
    case C_HIST: return (void**)&r->hist;
    case C_SNAPCOUNT: return (void**)&r->snap_count;
    case C_SNAPCELLS: return (void**)&r->snap_cells;
    case C_SNAPTIME: return (void**)&r->snap_time;
    case C_SNAPHIST: return (void**)&r->snap_hist;
    case C_DYNCOUNT: return (void**)&r->dyn_count;
    case C_DYN: return (void**)&r->dyn;
    case C_SUMK: return (void**)&r->sum_k;
    case C_NDIV: return (void**)&r->n_div;
    case C_NDEATH: return (void**)&r->n_death;
    case C_SUBHIST: return (void**)&r->sub_hist;
  }
  return nullptr;
}

// Relative duration of one event of every resident replicate with w blocks per SM, measured on B200 with
// the shared-memory kernel (profiles/): up to one warp per scheduler an event costs the latency of its
// dependent chain, from about three on the warps share the issue slots.
inline double round_cost(int w, int lanes) {
  static const double c4[] = {0.0, 1.00, 1.47, 2.05, 2.72, 3.31};  // 4-lane tiles (and wider), 4 warps per block
  static const double c2[] = {0.0, 1.00, 1.43, 2.02, 2.65, 3.30};  // 2-lane tiles (3 blocks per SM fit)
  static const double c1[] = {0.0, 1.00, 1.00, 1.22, 1.22, 1.60};  // 1-lane tiles, 2 warps per block (3 blocks fit)
  const double* c = lanes == 1 ? c1 : (lanes == 2 ? c2 : c4);
  return w <= 5 ? c[w] : c[5] + 0.6 * (w - 5);
}

// The default tile width.  Up to one warp per scheduler (4 x sm_count warps) an event takes the latency of
// its dependent chain whatever the width, so take the widest tile that keeps the batch within that; beyond,
// fewer lanes per replicate mean fewer instructions per event.  1-lane tiles (a lane owns a replicate: no
// shuffles at all, a third of the instructions of 2-lane tiles) need a 256-bin window to fit six warps per
// SM, so they are only taken when `lane_ok` (native stream, small initial copy numbers, no forced window).
inline uint32_t default_tile_width(uint64_t n_runs, int sm_count, bool native, bool lane_ok) {
  const uint64_t one_per_scheduler = 4ull * (uint64_t)sm_count;
  if (n_runs <= one_per_scheduler) return 32u;
  if (n_runs <= 2 * one_per_scheduler) return 16u;
  if (n_runs <= 4 * one_per_scheduler) return 8u;
  if (!native) return 4u;
  if (lane_ok && n_runs > 8 * one_per_scheduler) return 1u;
  return n_runs <= 8 * one_per_scheduler * 13 / 10 ? 4u : 2u;
}

// How many blocks per SM to launch and whether to time-slice.  Without slicing a batch of equal-length
// replicates (the unfavourable but common case: C1, C2, C5 are pure-birth runs of identical length) runs
// as full waves plus a last wave at the occupancy its size gives; with slicing n / slots "waves" run on
// a launch that holds fewer replicates than the batch.
inline void plan_launch(uint64_t n, int sm, int bps, int tiles_per_block, uint32_t slice_events, int lanes, int* w_out,
                        bool* sliced) {
  const bool prefer_four = lanes == 4;
  *w_out = bps;
  *sliced = false;
  const uint64_t per_w = (uint64_t)sm * tiles_per_block;  // replicates one block per SM holds
  const bool forced = slice_events != 0 && slice_events != 0xFFFFFFFFu && lanes != 1;
  if (slice_events == 0xFFFFFFFFu || lanes == 1 || (!forced && n >= 4 * per_w * bps)) {  // many waves: the queue balances them
    // (the 4-lane kernel at 4 blocks per SM and 128 registers is ~4 % ahead of 5 blocks at 96)
    if (slice_events != 0xFFFFFFFFu && prefer_four && bps > 4) *w_out = 4;
    return;
  }
  double best = 1e300;
  for (int w = 1; w <= bps; ++w) {
    const uint64_t slots = per_w * w;
    const uint64_t rem = n % slots;
    const double direct = (double)(n / slots) * round_cost(w, lanes) + (rem ? round_cost((int)((rem + per_w - 1) / per_w), lanes) : 0.0);
    if (!forced && direct < best) { best = direct; *w_out = w; *sliced = false; }
    if (n > slots) {
      const double sl = (double)n / (double)slots * round_cost(w, lanes) * 1.03;
      if (sl < best) { best = sl; *w_out = w; *sliced = true; }
    }
  }
  if (forced && !*sliced) *w_out = bps;  // the batch fits one launch at the lowest occupancy: nothing to slice
}

// one launch of ssa_kernel<L, GLOBAL, REPLAY>; returns the grid used through *grid_out
template <int L, bool GLOBAL, bool REPLAY, int KG, int SPEC = 0>
int launch_kernel(ecdna_b200_ctx* ctx, SsaArgs& a, cudaStream_t st, uint64_t max_items, uint32_t* grid_out,
                  uint32_t* bps_out, uint32_t slice_events) {
  auto kern = ssa_kernel<L, GLOBAL, REPLAY, KG, ECDNA_MIN_BLOCKS_L4, SPEC>;
  constexpr int BT = block_threads<L>();
  const int warps = BT / 32;
  const int tiles_per_block = BT / L;
  const size_t smem = GLOBAL ? 0 : (size_t)warps * Tile<L, GLOBAL>::window_words(a.kcap_s) * sizeof(uint32_t);
  if (smem > 220 * 1024) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "smem_bins too large for this tile width");
  CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int bps = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, BT, smem));
  if (bps < 1) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "kernel does not fit on an SM");
  if (GLOBAL && bps > 8) bps = 8;  // bounds the arena: one (32 + kcap_g)-word window per resident warp
  const uint64_t need = (max_items + tiles_per_block - 1) / tiles_per_block;
  int w = bps;
  bool sliced = false;
  if (!GLOBAL && !REPLAY) plan_launch(max_items, ctx->sm_count, bps, tiles_per_block, slice_events, L, &w, &sliced);
  uint64_t grid = (uint64_t)ctx->sm_count * w;
  if (need < grid) grid = need;
  if (grid == 0) grid = 1;
  // the build of the kernel that matches the blocks per SM of this launch (see ssa_kernel)
  constexpr bool HAS_BUILDS = L == 4 && !GLOBAL && !REPLAY;
  int minb = ECDNA_MIN_BLOCKS_L4;
  if constexpr (HAS_BUILDS) {
    const uint64_t per_sm = (grid + ctx->sm_count - 1) / ctx->sm_count;
    auto fits = [&](auto k, int blocks) -> bool {
      if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return false;
      int b = 0;
      return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, k, BT, smem) == cudaSuccess && b >= blocks;
    };
    if (per_sm <= 3 && fits(ssa_kernel<L, GLOBAL, REPLAY, KG, 3>, (int)per_sm)) minb = 3;
    else if (per_sm <= 4 && fits(ssa_kernel<L, GLOBAL, REPLAY, KG, 4>, (int)per_sm)) minb = 4;
  }
  a.ts_quantum = 0;
  if (sliced) {
    uint32_t q = slice_events ? slice_events : 1024u;
    uint32_t q2 = 64;
    while (q2 < q && q2 < (1u << 30)) q2 <<= 1;
    uint64_t cap = 1024;
    while (cap < 2 * max_items) cap <<= 1;
    const size_t rec_words = (size_t)max_items * (kParkHdr + 32u + a.kcap_s);
    CU(ctx->ts_ring.ensure(cap * 8));
    CU(ctx->ts_rec.ensure(rec_words * 4));
    CU(cudaMemsetAsync(ctx->ts_ring.p, 0, cap * 8, st));
    a.ts_quantum = q2;
    a.ts_slots = (uint32_t)(grid * tiles_per_block);
    a.ts_mask = (uint32_t)(cap - 1);
    a.ts_ring = (unsigned long long*)ctx->ts_ring.p;
    a.ts_rec = (uint32_t*)ctx->ts_rec.p;
    a.ts_ctr = (uint32_t*)((char*)ctx->counters.p + kRingCtrOffset);
    ctx->timing.slice_events = q2;
  }
  if (GLOBAL) {
    const size_t words = (size_t)grid * warps * Tile<32, true>::window_words(a.kcap_g);
    if (words > ctx->arena_words) {
      CU(ctx->arena.ensure(words * sizeof(uint32_t)));
      ctx->arena_words = words;
      CU(cudaMemsetAsync(ctx->arena.p, 0, words * sizeof(uint32_t), st));
    } else if (a.kcap_g != ctx->arena_kcap) {
      CU(cudaMemsetAsync(ctx->arena.p, 0, ctx->arena_words * sizeof(uint32_t), st));
    }
    ctx->arena_kcap = a.kcap_g;
    a.arena = (uint32_t*)ctx->arena.p;
  }
  if constexpr (HAS_BUILDS) {
    if (minb == 3) ssa_kernel<L, GLOBAL, REPLAY, KG, 3><<<(unsigned)grid, BT, smem, st>>>(a);
    else if (minb == 4) ssa_kernel<L, GLOBAL, REPLAY, KG, 4><<<(unsigned)grid, BT, smem, st>>>(a);
    else kern<<<(unsigned)grid, BT, smem, st>>>(a);
  } else if constexpr (L == 1 && !GLOBAL && !REPLAY && KG == 2) {
    // more than one warp per scheduler: issue slots bound the launch, take the build with the event loop unrolled once
    // (measured on one box, no-unroll / unroll: 125 000 birth-death draws 285.9 / 278.4 ms; 10^4 birth-death replicates
    // with dynamics 87.5 / 86.4 ms; 10^4 pure-birth replicates - C2 - 70.4 / 72.9 ms: the pure-birth build only when full)
    auto kern2 = ssa_kernel<L, GLOBAL, REPLAY, KG, ECDNA_MIN_BLOCKS_L4, SPEC, 2>;
    bool unrolled = grid * (uint64_t)warps > 4ull * (uint64_t)ctx->sm_count || SPEC == 2;
    if (const char* e = getenv("ECDNA_B200_UNROLL")) unrolled = e[0] == '1';  // (A/B measurements)
    if (unrolled) {
      int b2 = 0;
      unrolled = cudaFuncSetAttribute(kern2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess &&
                 cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b2, kern2, BT, smem) == cudaSuccess && b2 >= w;
    }
    if (getenv("ECDNA_B200_TRACE")) fprintf(stderr, "[ecdna_b200] 1-lane launch: grid %llu x %d warps, %d blocks/SM, loop unrolled: %d\n", (unsigned long long)grid, warps, w, (int)unrolled);
    if (unrolled) kern2<<<(unsigned)grid, BT, smem, st>>>(a);
    else kern<<<(unsigned)grid, BT, smem, st>>>(a);
  } else {
    kern<<<(unsigned)grid, BT, smem, st>>>(a);
  }
  CU(cudaGetLastError());
  *grid_out = (uint32_t)grid;
  *bps_out = (uint32_t)bps;
  return ECDNA_B200_OK;
}

// sparse return (capi.cu): the batch is simulated, measured and laid out on the device (*words = arena words it
// needs); sparse_fetch packs it and copies descriptors and arena to the host, the arena at word `base` of the
// caller's arena and the offsets shifted by `base` (blocks of a multi-GPU batch follow each other)
int sparse_prepare(ecdna_b200_ctx* ctx, const ecdna_b200_params_t* p, uint64_t idx_begin, uint64_t n_runs,
                   const ecdna_b200_results_t* results, uint64_t* words);
int sparse_fetch(ecdna_b200_ctx* ctx, ecdna_b200_dist_t* final_dist, ecdna_b200_dist_t* snap_dist,
                 ecdna_b200_dist_t* sub_dist, uint32_t* arena, uint64_t base);

// the launch with the histogram in the HBM arena (ssa_hbm.cu): every replicate of the batch, or, when
// a.park_list is set, the replicates the shared-memory launch parked
int launch_hbm(ecdna_b200_ctx* ctx, SsaArgs& a, cudaStream_t st, bool replay, uint32_t* grid_out, uint32_t* bps_out);

// the shared-memory launch for tiles of L lanes (ssa_l<L>.cu)
template <int L>
int launch_smem(ecdna_b200_ctx* ctx, SsaArgs& a, cudaStream_t st, bool replay, uint32_t slice_events, uint32_t* grid_out,
                uint32_t* bps_out);

template <int L, bool REPLAY>
int launch_smem_impl(ecdna_b200_ctx* ctx, SsaArgs& a, cudaStream_t st, uint32_t slice_events, uint32_t* grid,
                     uint32_t* bps) {
  // the walk over the shared window is unrolled for the common window sizes
  if constexpr (L == 1 && !REPLAY) {
    if (a.kcap_s == 128) return launch_kernel<L, false, REPLAY, 1>(ctx, a, st, a.n_runs, grid, bps, slice_events);
    // the reference's default process (pure birth, binomial segregation) has its own build of the kernel
    if (a.kcap_s == 256 && a.pure_birth_binomial) return launch_kernel<L, false, REPLAY, 2, 1>(ctx, a, st, a.n_runs, grid, bps, slice_events);
    if (a.kcap_s == 256 && a.binomial_only) return launch_kernel<L, false, REPLAY, 2, 2>(ctx, a, st, a.n_runs, grid, bps, slice_events);
  }
  if (!REPLAY && a.kcap_s == 256) return launch_kernel<L, false, REPLAY, 2>(ctx, a, st, a.n_runs, grid, bps, slice_events);
  if constexpr ((L == 16 || L == 32) && !REPLAY) {  // (the tiles of small batches: C1, C5)
    if (a.kcap_s == 512 && a.pure_birth_binomial) return launch_kernel<L, false, REPLAY, 4, 1>(ctx, a, st, a.n_runs, grid, bps, slice_events);
  }
  if (!REPLAY && a.kcap_s == 512) return launch_kernel<L, false, REPLAY, 4>(ctx, a, st, a.n_runs, grid, bps, slice_events);
  return launch_kernel<L, false, REPLAY, 0>(ctx, a, st, a.n_runs, grid, bps, slice_events);
}

#define ECDNA_DEFINE_LAUNCH_SMEM(L_)                                                                             \
  namespace ecdna {                                                                                              \
  template <>                                                                                                    \
  int launch_smem<L_>(ecdna_b200_ctx * ctx, SsaArgs & a, cudaStream_t st, bool replay, uint32_t slice_events,    \
                      uint32_t* grid_out, uint32_t* bps_out) {                                                   \
    if constexpr (L_ <= 2) {                                                                                     \
      if (replay) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "1- and 2-lane tiles exist for the native random source only"); \
      return launch_smem_impl<L_, false>(ctx, a, st, slice_events, grid_out, bps_out);                           \
    } else {                                                                                                     \
      return replay ? launch_smem_impl<L_, true>(ctx, a, st, slice_events, grid_out, bps_out)                    \
                    : launch_smem_impl<L_, false>(ctx, a, st, slice_events, grid_out, bps_out);                  \
    }                                                                                                            \
  }                                                                                                              \
  }

}  // namespace ecdna

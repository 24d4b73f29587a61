// capi.cu -- the C ABI of libecdna_b200.so (include/ecdna_b200.h) over the SSA kernel.
//
// One context = one GPU, one stream, grow-only device buffers.  There is no CPU path: without an
// sm_100 device every entry point fails with ECDNA_B200_ERR_NO_DEVICE / ECDNA_B200_ERR_CUDA.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "engine.cuh"
#include "sparse.cuh"
#include "subsample.cuh"
#include "uniform_replay.cuh"

using namespace ecdna;

namespace {

// ---- longest-expected-first order of a batch with per-run rates (ABC prior draws) ----
// The replicates of such a batch differ several-fold in length: a draw with net growth rate r = b - d of its
// dominant cell type takes about min(N, e^(rT)) (b + d) / r events to reach N cells or the time limit T.  A
// launch that hands out the longest first ends with the short ones, which cuts the under-occupied tail of the
// batch (decisive when 1e6 draws are spread over 8 GPUs).  Results do not depend on the order.
constexpr uint32_t kLptBuckets = 1024;
__device__ __forceinline__ uint32_t lpt_bucket(const float* r, float max_cells, float max_time) {
  const float rp = r[1] - r[3], rm = r[0] - r[2];
  const bool plus = rp >= rm;
  const float net = plus ? rp : rm, tot = plus ? r[1] + r[3] : r[0] + r[2];
  float cost = 1.0f;
  if (net > 0.02f) cost = fminf(max_cells, __expf(fminf(net * max_time, 80.f))) * tot / net;
  const int b = (int)(__log2f(fmaxf(cost, 1.0f)) * 24.0f);  // ~3 % steps
  return kLptBuckets - 1u - (uint32_t)min(max(b, 0), (int)kLptBuckets - 1);  // bucket 0 = the longest
}
__global__ void lpt_count(const float* rates, uint32_t n, float max_cells, float max_time, uint32_t* hist) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) atomicAdd(hist + lpt_bucket(rates + 4 * (size_t)i, max_cells, max_time), 1u);
}
__global__ void lpt_scan(uint32_t* hist) {  // one block of kLptBuckets threads: exclusive scan in place
  __shared__ uint32_t sh[kLptBuckets];
  const uint32_t t = threadIdx.x;
  sh[t] = hist[t];
  __syncthreads();
  for (uint32_t o = 1; o < kLptBuckets; o <<= 1) {
    const uint32_t v = t >= o ? sh[t - o] : 0u;
    __syncthreads();
    sh[t] += v;
    __syncthreads();
  }
  hist[t] = sh[t] - hist[t];
}
__global__ void lpt_scatter(const float* rates, uint32_t n, float max_cells, float max_time, uint32_t* cursor, uint32_t* order) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) order[atomicAdd(cursor + lpt_bucket(rates + 4 * (size_t)i, max_cells, max_time), 1u)] = i;
}

// phase 1: histogram in shared memory, tiles of L lanes; a replicate that outgrows its window is parked with
// its state and continued by the next launch of the cascade: (1-lane tiles with a 128-bin window only) a second
// shared-memory launch with 256 bins, then the launch with the histogram in HBM
int launch_all(ecdna_b200_ctx* ctx, SsaArgs& a, cudaStream_t st, const ecdna_b200_params_t* p, uint32_t L, bool replay) {
  uint32_t grid = 0, bps = 0;
  ecdna_b200_timing_t& tm = ctx->timing;
  uint32_t* const ctr = (uint32_t*)ctx->counters.p;  // [0] [1] [28]: queues of the three launches; [2] [3]: park counts
  CU(cudaEventRecord(ctx->ev_k0, st));
  a.resume_count = nullptr;
  a.work_counter = ctr;
  if (p->state_mode == ECDNA_B200_STATE_HBM) {
    a.park_list = nullptr;
    a.allow_park = 0;
    int rc = launch_hbm(ctx, a, st, replay, &grid, &bps);
    if (rc) return rc;
    tm.kernel_launches = 1;
    tm.tile_width = 32;
    tm.block_threads = kBlockThreads;
  } else {
    a.allow_park = p->state_mode == ECDNA_B200_STATE_AUTO ? 1u : 0u;
    int rc;
    switch (L) {
      case 1: rc = launch_smem<1>(ctx, a, st, replay, p->slice_events, &grid, &bps); break;
      case 2: rc = launch_smem<2>(ctx, a, st, replay, p->slice_events, &grid, &bps); break;
      case 4: rc = launch_smem<4>(ctx, a, st, replay, p->slice_events, &grid, &bps); break;
      case 8: rc = launch_smem<8>(ctx, a, st, replay, p->slice_events, &grid, &bps); break;
      case 16: rc = launch_smem<16>(ctx, a, st, replay, p->slice_events, &grid, &bps); break;
      default: rc = launch_smem<32>(ctx, a, st, replay, p->slice_events, &grid, &bps); break;
    }
    if (rc) return rc;
    tm.kernel_launches = 1;
    tm.tile_width = L;
    tm.block_threads = L == 1 ? (uint32_t)block_threads<1>() : (uint32_t)kBlockThreads;
    tm.smem_bins = a.kcap_s;
    if (a.allow_park) {
      // the next launch works through what this one parked
      SsaArgs n = a;
      n.resume_count = a.park_count; n.resume_list = a.park_list; n.resume_rec = a.park_rec;
      n.resume_cap = a.park_cap; n.resume_kcap = a.kcap_s;
      n.work_counter = ctr + 1;
      n.ts_quantum = 0;
      uint32_t g2 = 0, b2 = 0;
      if (L == 1 && a.kcap_s == 128) {
        // 1-lane tiles run ten warps per SM with a 128-bin window (six with 256); the few replicates whose
        // copy numbers pass 127 continue in a 256-bin launch of the same kernel, whose own leftovers go to HBM
        const uint64_t cap2 = a.park_cap;
        CU(ctx->park_list2.ensure((size_t)a.n_runs * 4));
        CU(ctx->park_rec2.ensure((cap2 ? cap2 : 1) * (size_t)(kParkHdr + 32u + 256u) * 4));
        n.kcap_s = 256;
        if (n.kcap_g < n.kcap_s) n.kcap_g = n.kcap_s;
        n.park_count = ctr + 3; n.park_list = (uint32_t*)ctx->park_list2.p; n.park_rec = (uint32_t*)ctx->park_rec2.p;
        n.park_cap = (uint32_t)cap2;
        rc = launch_smem<1>(ctx, n, st, replay, 0xFFFFFFFFu, &g2, &b2);
        if (rc) return rc;
        tm.kernel_launches += 1;
        SsaArgs h = n;
        h.resume_count = n.park_count; h.resume_list = n.park_list; h.resume_rec = n.park_rec;
        h.resume_cap = n.park_cap; h.resume_kcap = n.kcap_s;
        h.work_counter = ctr + 28;
        n = h;
      }
      n.allow_park = 0;
      rc = launch_hbm(ctx, n, st, replay, &g2, &b2);
      if (rc) return rc;
      tm.kernel_launches += 1;
    }
  }
  CU(cudaEventRecord(ctx->ev_k1, st));
  if (p->state_mode == ECDNA_B200_STATE_HBM) tm.smem_bins = a.kcap_s;
  tm.grid_blocks = grid;
  tm.blocks_per_sm = bps;
  return ECDNA_B200_OK;
}

// target statistics for the ABC epilogue, same definitions as the device epilogue
void target_stats(const std::vector<uint64_t>& h, float* mean, float* ent, float* freq, std::vector<float>* cdf) {
  uint64_t n = 0, s1 = 0;
  for (size_t k = 0; k < h.size(); ++k) { n += h[k]; s1 += (uint64_t)k * h[k]; }
  cdf->assign(h.size(), 1.0f);
  *mean = *ent = *freq = 0.f;
  if (n == 0) return;
  const float nf = (float)n;
  *mean = (float)s1 / nf;
  *freq = (float)(n - h[0]) / nf;
  unsigned long long eq = 0;  // (the same fixed-point entropy as the device epilogue: bit-identical)
  uint64_t cum = 0;
  for (size_t k = 0; k < h.size(); ++k) {
    if (h[k]) eq += entropy_term_q40(h[k], n);
    cum += h[k];
    (*cdf)[k] = (float)cum / nf;
  }
  *ent = entropy_from_q40(eq);
}

int validate(ecdna_b200_ctx* ctx, const ecdna_b200_params_t* p, uint64_t n_runs) {
  if (!p) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "params is NULL");
  if (p->abi_version != ECDNA_B200_ABI_VERSION) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "abi_version mismatch");
  if (n_runs == 0 || n_runs >= 0xFFFFFFF0ull) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "n_runs must be in [1, 2^32)");
  const float r[4] = {p->b0, p->b1, p->d0, p->d1};
  for (float v : r)
    if (!(v >= 0.f)) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "rates must be >= 0 (Exp::new panics otherwise)");
  if (p->segregation > 3) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "unknown segregation rule");
  if (p->max_cells == 0 || p->max_cells >= (1ull << 32)) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "max_cells must be in [1, 2^32)");
  if (p->max_iter == 0 || p->max_iter >= (1ull << 32)) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "max_iter must be in [1, 2^32)");
  if (p->n_init == 0 || !p->init_k || !p->init_c) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "empty initial distribution (ensure!(!distribution.is_empty()), process.rs:88)");
  if (p->n_snapshots && !p->snapshot_cells) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "snapshot_cells is NULL");
  if (p->rng_mode > 2) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "unknown rng_mode");
  if (p->rng_mode == ECDNA_B200_RNG_UNIFORMS) {
    if (!p->replay_u64 || !p->replay_offsets) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "uniform replay needs replay_u64 and replay_offsets");
    if (p->n_snapshots || p->dyn_points || p->abc_enabled) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "uniform replay has no snapshots, dynamics or ABC epilogue");
    if (n_runs * (p->max_cells + 2) > (8ull << 30)) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "uniform replay keeps one u16 per cell per replicate: batch too large");
  }
  if (p->rng_mode == ECDNA_B200_RNG_REPLAY && (!p->replay || !p->replay_offsets)) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "replay mode needs replay and replay_offsets");
  if (p->state_mode > 2) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "unknown state_mode");
  if (p->tile_width != 0 && p->tile_width != 1 && p->tile_width != 2 && p->tile_width != 4 && p->tile_width != 8 && p->tile_width != 16 && p->tile_width != 32) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "tile_width must be 1, 2, 4, 8, 16 or 32");
  if ((p->tile_width == 1 || p->tile_width == 2) && p->rng_mode != ECDNA_B200_RNG_PHILOX) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "1- and 2-lane tiles exist for the native random source only");
  if (p->bd_count_mode > 1) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "bd_count_mode must be 0 or 1");
  if (p->bd_count_mode == 1 && p->rates_per_run && !(p->d0 > 0.f || p->d1 > 0.f))
    return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "bd_count_mode 1 with per-run rates: the BASE d0/d1 select the process type (clap_app.rs:165-174); set one of them > 0 for the birth-death process");
  if (p->max_copies > 65535) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "max_copies must be <= 65535 (DNACopy is u16)");
  if (p->abc_enabled && (!p->abc_target_hist || p->abc_target_len == 0)) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "abc_enabled needs a target distribution");
  if (p->dyn_points && !(p->dyn_dt > 0.f)) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "dyn_dt must be > 0");
  if (p->n_subsamples && !p->subsample_cells) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "subsample_cells is NULL");
  if (p->n_subsamples > 65535) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "at most 65535 subsample sizes");
  return ECDNA_B200_OK;
}

// device_io: results and the bulk inputs are device pointers already
int run_common(ecdna_b200_ctx* ctx, const ecdna_b200_params_t* p, uint64_t idx_begin, uint64_t n_runs,
               const ecdna_b200_results_t* results, cudaStream_t st, bool device_io, bool sparse = false) {
  int rc = validate(ctx, p, n_runs);
  if (rc) return rc;
  if (!results) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "results is NULL");
  CU(cudaSetDevice(ctx->device));
  ecdna_b200_timing_t& tm = ctx->timing;
  tm = ecdna_b200_timing_t{};
  ctx->have_total = !device_io;
  ctx->sp.valid = false;

  SsaArgs a{};
  a.rate[0] = p->b0; a.rate[1] = p->b1; a.rate[2] = p->d0; a.rate[3] = p->d1;
  a.segregation = p->segregation;
  const bool birth_death = p->d0 > 0.f || p->d1 > 0.f;  // clap_app.rs:165-174
  a.cells_stop = (uint32_t)((p->bd_count_mode == 1 && birth_death) ? (p->max_cells + 1) / 2 : p->max_cells);
  a.max_iter_m1 = (uint32_t)(p->max_iter - 1);
  a.max_time = p->max_time;
  a.seed_lo = (uint32_t)p->seed; a.seed_hi = (uint32_t)(p->seed >> 32);
  for (uint32_t r = 0; r < 10; ++r) { a.pk[2 * r] = a.seed_lo + r * 0x9E3779B9u; a.pk[2 * r + 1] = a.seed_hi + r * 0xBB67AE85u; }
  a.idx_begin = idx_begin;
  a.n_runs = (uint32_t)n_runs;
  a.dyn_points = p->dyn_points; a.dyn_dt = p->dyn_dt;
  a.flags = p->flags;
  // tile width: up to one warp per scheduler (4 x 148) an event takes the same time whatever the width
  // (the latency of its dependent chain, profiles/r01_j_occupancy.md); beyond that the warps share the
  // issue slots, so take the widest tile that keeps the batch within one warp per scheduler, down to 4
  // lanes (8 replicates per warp, an eighth of the instructions per event)
  // ... and 2 lanes (16 replicates per warp, each lane carrying two of the event's four Philox slots: 27
  // instructions per event against 39) once even 4-lane tiles exceed one warp per scheduler by ~30 %
  // (measured crossover: 4-lane tiles time-sliced on one block per SM against one block of 2-lane tiles)
  const bool native = p->rng_mode == ECDNA_B200_RNG_PHILOX;
  // shared window: 4-, 2- and 1-lane tiles keep 8 / 16 / 32 replicates per warp window, so 256 bins unless the
  // initial copy numbers are large already (they grow to several times the largest initial one)
  uint32_t k0max = 0;
  for (uint32_t i = 0; i < p->n_init; ++i)
    if (p->init_c[i] != 0 && p->init_k[i] > k0max) k0max = p->init_k[i];
  // (1-lane tiles draw 128 segregation bits per event inline and fit six warps per SM with a 256-bin window only)
  const bool lane_ok = native && k0max <= 16u && (p->smem_bins == 0 || p->smem_bins <= 256u) &&
                       p->state_mode != ECDNA_B200_STATE_HBM;
  uint32_t L = p->tile_width ? p->tile_width : default_tile_width(n_runs, ctx->sm_count, native, lane_ok);
  // Large initial copy numbers: the copy numbers of a growing population spread to roughly twice the largest
  // initial one (measured: {2000: 1} reaches ~3100 at 1e5 cells, {10000: 1} ~12000), and a replicate that
  // outgrows its window moves to the HBM launch, which is several times slower.  So the default window holds
  // 2 k0 + 256 bins when that fits a block (4 warps, ~200 KB of shared memory), on wider tiles if need be.
  uint32_t default_bins = (L <= 4 && k0max <= 16u) ? 256u : 512u;
  // (1-lane tiles with smem_bins = 128 run ten warps per SM instead of six and continue the replicates whose
  //  copy numbers pass 127 in a 256-bin launch, see launch_all.  Measured on the C4 shape: +16 % while every SM
  //  is full, +3 % over a whole 1e6-draw batch - the longer tail of a launch that holds more replicates eats
  //  the rest - so it is not the default.)
  if (k0max > 128u && p->smem_bins == 0 && p->state_mode != ECDNA_B200_STATE_HBM) {
    const uint32_t want_bins = (2u * k0max + 256u + 127u) & ~127u;
    auto fits = [](uint32_t lanes) -> uint32_t {  // bins per replicate a 4-warp block holds with tiles of `lanes`
      const uint32_t r = 32u / lanes, sg = (r + 3u) / 4u;
      return ((200u * 1024u / 16u - 128u * sg) / r) & ~127u;
    };
    // (a draw of 2k bits beyond the tile's own 128 (L - 1) needs the complete step, except on full-warp tiles,
    //  whose straight-line step loops over the extra slots: measured 2.4x on {2000: 1})
    if (!p->tile_width)
      while (L < 32u && (fits(L) < want_bins || 128u * (L - 1u) < 4u * k0max)) L *= 2u;
    default_bins = std::max(default_bins, std::min(want_bins, fits(L)));
  }
  a.kcap_s = p->smem_bins ? ((p->smem_bins + 127u) & ~127u) : default_bins;  // bins come in rows of 4 x 32
  a.kcap_g = ((p->max_copies ? p->max_copies : 65535u) + 128u) & ~127u;
  if (a.kcap_g < a.kcap_s) a.kcap_g = a.kcap_s;
  a.hist_stride = p->hist_stride ? p->hist_stride : 512u;
  const uint32_t stride = a.hist_stride;

  if (!device_io) CU(cudaEventRecord(ctx->ev_begin, st));

  // ---- small inputs: initial distribution, snapshot sizes (always host pointers) ----
  std::vector<uint32_t> ik, ic;
  uint64_t nminus0 = 0;
  for (uint32_t i = 0; i < p->n_init; ++i) {
    if (p->init_c[i] == 0) continue;
    if (p->init_c[i] >= (1ull << 32)) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "initial count too large");
    if (p->init_k[i] == 0) { nminus0 += p->init_c[i]; continue; }
    if (p->init_k[i] >= a.kcap_g) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "initial copy number beyond max_copies");
    ik.push_back(p->init_k[i]);
    ic.push_back((uint32_t)p->init_c[i]);
  }
  if (ik.empty() && nminus0 == 0) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "empty initial distribution (ensure!(!distribution.is_empty()), process.rs:88)");
  {
    uint64_t total0 = nminus0;
    for (uint32_t c : ic) total0 += c;
    if (nminus0 >= (1ull << 32) || total0 >= (1ull << 32)) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "initial population must be below 2^32 cells");
    if (p->rng_mode == ECDNA_B200_RNG_UNIFORMS && total0 - nminus0 > p->max_cells + 2)
      return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "uniform replay keeps max_cells + 2 cells per replicate: the initial ecDNA+ population does not fit");
  }
  a.n_init = (uint32_t)ik.size();
  a.init_nminus = (uint32_t)nminus0;
  if (a.n_init) {
    CU(ctx->init_k.ensure(ik.size() * 4));
    CU(ctx->init_c.ensure(ic.size() * 4));
    CU(cudaMemcpyAsync(ctx->init_k.p, ik.data(), ik.size() * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ctx->init_c.p, ic.data(), ic.size() * 4, cudaMemcpyHostToDevice, st));
    tm.h2d_bytes += ik.size() * 8;
  }
  a.init_k = (const uint32_t*)ctx->init_k.p;
  a.init_c = (const uint32_t*)ctx->init_c.p;
  std::vector<uint32_t> snaps;
  for (uint32_t i = 0; i < p->n_snapshots; ++i)
    snaps.push_back(p->snapshot_cells[i] >= (1ull << 32) ? 0xFFFFFFFFu : (uint32_t)p->snapshot_cells[i]);
  a.n_snap = (uint32_t)snaps.size();
  if (a.n_snap) {
    CU(ctx->snap.ensure(snaps.size() * 4));
    CU(cudaMemcpyAsync(ctx->snap.p, snaps.data(), snaps.size() * 4, cudaMemcpyHostToDevice, st));
    tm.h2d_bytes += snaps.size() * 4;
  }
  a.snap_cells = (const uint32_t*)ctx->snap.p;

  // ---- ABC target: statistics and CDF computed once on the host, uploaded ----
  std::vector<float> cdf;
  if (p->abc_enabled) {
    std::vector<uint64_t> th(p->abc_target_len);
    if (device_io) CU(cudaMemcpyAsync(th.data(), p->abc_target_hist, th.size() * 8, cudaMemcpyDeviceToHost, st));
    else std::memcpy(th.data(), p->abc_target_hist, th.size() * 8);
    if (device_io) CU(cudaStreamSynchronize(st));
    target_stats(th, &a.abc_mean, &a.abc_entropy, &a.abc_freq, &cdf);
    CU(ctx->abc_cdf.ensure(cdf.size() * 4));
    CU(cudaMemcpyAsync(ctx->abc_cdf.p, cdf.data(), cdf.size() * 4, cudaMemcpyHostToDevice, st));
    tm.h2d_bytes += cdf.size() * 4;
    a.abc = 1;
    a.abc_cdf = (const float*)ctx->abc_cdf.p;
    a.abc_len = (uint32_t)cdf.size();
    for (int i = 0; i < 4; ++i) a.abc_thr[i] = p->abc_thresholds[i];
  }

  // ---- bulk inputs: per-run rates, replay stream ----
  if (p->rates_per_run) {
    if (device_io) a.rates_per_run = p->rates_per_run;
    else {
      CU(ctx->rates.ensure(n_runs * 16));
      CU(cudaMemcpyAsync(ctx->rates.p, p->rates_per_run, n_runs * 16, cudaMemcpyHostToDevice, st));
      tm.h2d_bytes += n_runs * 16;
      a.rates_per_run = (const float*)ctx->rates.p;
    }
  }
  const bool uniforms = p->rng_mode == ECDNA_B200_RNG_UNIFORMS;
  const bool replay = p->rng_mode == ECDNA_B200_RNG_REPLAY;
  if (replay) {
    if (device_io) { a.replay = p->replay; a.replay_off = p->replay_offsets; }
    else {
      const uint64_t total = p->replay_offsets[n_runs];
      CU(ctx->replay.ensure((size_t)total * sizeof(ecdna_b200_replay_event_t) + 16));
      CU(ctx->replay_off.ensure((n_runs + 1) * 8));
      CU(cudaMemcpyAsync(ctx->replay.p, p->replay, (size_t)total * sizeof(ecdna_b200_replay_event_t), cudaMemcpyHostToDevice, st));
      CU(cudaMemcpyAsync(ctx->replay_off.p, p->replay_offsets, (n_runs + 1) * 8, cudaMemcpyHostToDevice, st));
      tm.h2d_bytes += total * sizeof(ecdna_b200_replay_event_t) + (n_runs + 1) * 8;
      a.replay = (const ecdna_b200_replay_event_t*)ctx->replay.p;
      a.replay_off = (const uint64_t*)ctx->replay_off.p;
    }
  }

  // ---- outputs ----
  ecdna_b200_results_t host = *results, dev = *results;
  if (!device_io) {
    for (int c = 0; c < C_COUNT; ++c) {
      void** hs = col_slot(&host, c);
      void** ds = col_slot(&dev, c);
      // (the sparse return packs the distributions on the device: they exist there whether or not the host wants them)
      const bool for_sparse = sparse && (c == C_HIST || c == C_SNAPHIST || c == C_SUBHIST || c == C_SNAPCOUNT ||
                                         c == C_SNAPTIME || c == C_TIME || c == C_STOP);
      if (!*hs && !for_sparse) continue;
      const size_t bytes = col_bytes(c, p, stride) * n_runs;
      if (bytes == 0) { *ds = nullptr; continue; }
      CU(ctx->cols[c].ensure(bytes));
      *ds = ctx->cols[c].p;
      // (the staging buffers are reused between calls: nothing of an earlier batch may survive)
      CU(cudaMemsetAsync(*ds, 0, bytes, st));
    }
  }
  const bool want_sub = p->n_subsamples != 0 && dev.sub_hist != nullptr;
  if (want_sub && !dev.hist) {  // the samples are drawn from the final distribution: keep one on the device
    CU(ctx->hist_tmp.ensure((size_t)n_runs * stride * 4));
    dev.hist = (uint32_t*)ctx->hist_tmp.p;
  }
  a.out = dev;
  CU(ctx->counters.ensure(128));
  CU(cudaMemsetAsync(ctx->counters.p, 0, 128, st));
  a.work_counter = (uint32_t*)ctx->counters.p;                              // (launch_all assigns the queues)
  a.park_count = (uint32_t*)ctx->counters.p + 2;
  a.totals = (unsigned long long*)((char*)ctx->counters.p + kTotalsOffset);
  ctx->expect_finished = n_runs;
  if (p->state_mode == ECDNA_B200_STATE_AUTO) {
    uint64_t cap = p->spill_records == 0xFFFFFFFFu ? 0 : (p->spill_records ? p->spill_records : 32768u);
    if (cap > n_runs) cap = n_runs;
    CU(ctx->park_list.ensure(n_runs * 4));
    CU(ctx->park_rec.ensure((cap ? cap : 1) * (size_t)(kParkHdr + 32u + a.kcap_s) * 4));
    a.park_list = (uint32_t*)ctx->park_list.p;
    a.park_rec = (uint32_t*)ctx->park_rec.p;
    a.park_cap = (uint32_t)cap;
  }

  a.pure_birth_binomial = (!a.rates_per_run && p->d0 == 0.f && p->d1 == 0.f && p->segregation == ECDNA_B200_SEG_BINOMIAL &&
                           !(p->flags & ECDNA_B200_WANT_DIGEST)) ? 1u : 0u;
  a.binomial_only = (p->segregation == ECDNA_B200_SEG_BINOMIAL && !(p->flags & ECDNA_B200_WANT_DIGEST)) ? 1u : 0u;
  a.order = nullptr;
  // (1-lane tiles only: they never time-slice, and the timetable of a sliced launch is keyed by replicate index)
  if (a.rates_per_run && native && L == 1 && n_runs >= 8192 && !(p->flags & ECDNA_B200_KEEP_ORDER)) {
    const uint32_t n32 = (uint32_t)n_runs;
    CU(ctx->order.ensure((size_t)n_runs * 4));
    CU(ctx->order_hist.ensure(kLptBuckets * 4));
    CU(cudaMemsetAsync(ctx->order_hist.p, 0, kLptBuckets * 4, st));
    lpt_count<<<(n32 + 255) / 256, 256, 0, st>>>(a.rates_per_run, n32, (float)p->max_cells, p->max_time, (uint32_t*)ctx->order_hist.p);
    lpt_scan<<<1, kLptBuckets, 0, st>>>((uint32_t*)ctx->order_hist.p);
    lpt_scatter<<<(n32 + 255) / 256, 256, 0, st>>>(a.rates_per_run, n32, (float)p->max_cells, p->max_time, (uint32_t*)ctx->order_hist.p,
                                                   (uint32_t*)ctx->order.p);
    CU(cudaGetLastError());
    a.order = (const uint32_t*)ctx->order.p;
  }
  if (uniforms) {
    // the reference's own stream on the reference's own state layout: one thread per replicate
    UrArgs u{};
    for (int i = 0; i < 4; ++i) u.rate[i] = a.rate[i];
    u.rates_per_run = a.rates_per_run;
    u.segregation = a.segregation; u.cells_stop = a.cells_stop; u.max_iter_m1 = a.max_iter_m1; u.max_time = a.max_time;
    u.n_runs = a.n_runs; u.n_init = a.n_init; u.init_k = a.init_k; u.init_c = a.init_c; u.init_nminus = a.init_nminus;
    u.hist_stride = a.hist_stride; u.totals = a.totals; u.out = a.out;
    u.cap = p->max_cells + 2;
    CU(ctx->cells.ensure((size_t)n_runs * u.cap * sizeof(uint16_t)));
    u.cells = (uint16_t*)ctx->cells.p;
    if (device_io) { u.stream = p->replay_u64; u.stream_off = p->replay_offsets; }
    else {
      const uint64_t total = p->replay_offsets[n_runs];
      CU(ctx->replay.ensure((size_t)total * 8 + 16));
      CU(ctx->replay_off.ensure((n_runs + 1) * 8));
      CU(cudaMemcpyAsync(ctx->replay.p, p->replay_u64, (size_t)total * 8, cudaMemcpyHostToDevice, st));
      CU(cudaMemcpyAsync(ctx->replay_off.p, p->replay_offsets, (n_runs + 1) * 8, cudaMemcpyHostToDevice, st));
      tm.h2d_bytes += total * 8 + (n_runs + 1) * 8;
      u.stream = (const uint64_t*)ctx->replay.p;
      u.stream_off = (const uint64_t*)ctx->replay_off.p;
    }
    // Exp1 ziggurat tables, regenerated from the published recurrence (Marsaglia & Tsang 2000)
    std::vector<double> zig(514);
    {
      const double R = 7.69711747013104972, v = 3.949659822581572e-3;
      double* x = zig.data();
      double* f = zig.data() + 257;
      x[0] = v / std::exp(-R);
      x[1] = R;
      for (int i = 2; i < 256; ++i) x[i] = -std::log(v / x[i - 1] + std::exp(-x[i - 1]));
      x[256] = 0.0;
      for (int i = 0; i < 257; ++i) f[i] = std::exp(-x[i]);
    }
    CU(ctx->zig.ensure(zig.size() * 8));
    CU(cudaMemcpyAsync(ctx->zig.p, zig.data(), zig.size() * 8, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));  // `zig` is a stack vector
    u.zig_x = (const double*)ctx->zig.p;
    u.zig_f = (const double*)ctx->zig.p + 257;
    CU(cudaEventRecord(ctx->ev_k0, st));
    uniform_replay_kernel<<<(unsigned)((n_runs + 63) / 64), 64, 0, st>>>(u);
    CU(cudaGetLastError());
    CU(cudaEventRecord(ctx->ev_k1, st));
    tm.kernel_launches = 1; tm.tile_width = 1; tm.grid_blocks = (uint32_t)((n_runs + 63) / 64); tm.block_threads = 64;
    rc = ECDNA_B200_OK;
  }
  else rc = launch_all(ctx, a, st, p, L, replay);
  if (rc) return rc;

  if (want_sub) {  // main.rs:110-123, one warp per (replicate, size)
    CU(ctx->sub_sizes.ensure((size_t)p->n_subsamples * 8));
    CU(cudaMemcpyAsync(ctx->sub_sizes.p, p->subsample_cells, (size_t)p->n_subsamples * 8, cudaMemcpyHostToDevice, st));
    tm.h2d_bytes += (size_t)p->n_subsamples * 8;
    SubArgs sa{};
    sa.seed_lo = a.seed_lo; sa.seed_hi = a.seed_hi; sa.idx_begin = idx_begin;
    sa.n_runs = a.n_runs; sa.n_sub = p->n_subsamples; sa.stride = stride;
    sa.sizes = (const unsigned long long*)ctx->sub_sizes.p;
    sa.hist = dev.hist; sa.out = dev.sub_hist;
    const unsigned long long tasks = (unsigned long long)n_runs * p->n_subsamples;
    subsample_kernel<<<(unsigned)((tasks + 3) / 4), 128, 0, st>>>(sa);
    CU(cudaGetLastError());
    tm.kernel_launches += 1;
  }

  if (sparse) {  // measure every distribution and lay the windows out (sparse.cuh)
    SparseArgs sa{};
    sa.n_runs = a.n_runs; sa.n_snap = a.n_snap; sa.n_sub = dev.sub_hist ? p->n_subsamples : 0u; sa.stride = stride;
    sa.rows = (unsigned long long)n_runs * (1ull + sa.n_snap + sa.n_sub);
    sa.hist = dev.hist; sa.snap_hist = dev.snap_hist; sa.sub_hist = dev.sub_hist;
    sa.snap_count = dev.snap_count; sa.time = dev.time; sa.snap_time = dev.snap_time; sa.stop = dev.stop_reason;
    const uint64_t chunks = (sa.rows + kSparseChunk - 1) / kSparseChunk;
    CU(ctx->sp_desc.ensure((size_t)sa.rows * sizeof(ecdna_b200_dist_t)));
    CU(ctx->sp_len.ensure((size_t)sa.rows * 4));
    CU(ctx->sp_bsum.ensure((size_t)(chunks + 1) * 8));
    sa.desc = (ecdna_b200_dist_t*)ctx->sp_desc.p; sa.len = (uint32_t*)ctx->sp_len.p; sa.bsum = (unsigned long long*)ctx->sp_bsum.p;
    sparse_measure<<<(unsigned)((sa.rows + 7) / 8), 256, 0, st>>>(sa);
    sparse_chunk_sums<<<(unsigned)chunks, 256, 0, st>>>(sa);
    sparse_scan_chunks<<<1, 256, 0, st>>>(sa.bsum, (uint32_t)chunks);
    sparse_offsets<<<(unsigned)chunks, 256, 0, st>>>(sa);
    CU(cudaGetLastError());
    tm.kernel_launches += 4;
    ctx->sp.n_runs = n_runs; ctx->sp.n_snap = sa.n_snap; ctx->sp.n_sub = sa.n_sub; ctx->sp.rows = sa.rows; ctx->sp.stride = stride;
    ctx->sp.packed = false;
  }

  if (!device_io) {
    for (int c = 0; c < C_COUNT; ++c) {
      void** hs = col_slot(&host, c);
      void** ds = col_slot(&dev, c);
      if (!*hs || !*ds) continue;
      const size_t bytes = col_bytes(c, p, stride) * n_runs;
      CU(cudaMemcpyAsync(*hs, *ds, bytes, cudaMemcpyDeviceToHost, st));
      tm.d2h_bytes += bytes;
    }
    unsigned long long sparse_words = 0;
    if (sparse) {
      const uint64_t chunks = (ctx->sp.rows + kSparseChunk - 1) / kSparseChunk;
      CU(cudaMemcpyAsync(&sparse_words, (unsigned long long*)ctx->sp_bsum.p + chunks, 8, cudaMemcpyDeviceToHost, st));
      tm.d2h_bytes += 8;
    }
    CU(cudaEventRecord(ctx->ev_end, st));
    CU(cudaStreamSynchronize(st));
    if (sparse) {
      ctx->sp.words = sparse_words;
      ctx->sp.valid = true;
    }
    // every replicate of the batch must have gone through the epilogue (a lost one would leave zeros behind)
    unsigned long long fin = 0;
    CU(cudaMemcpy(&fin, (char*)ctx->counters.p + kTotalsOffset + 7 * 8, 8, cudaMemcpyDeviceToHost));
    if (fin != n_runs)
      return fail(ctx, ECDNA_B200_ERR_INTERNAL, "internal error: " + std::to_string(fin) + " of " + std::to_string(n_runs) + " replicates finished");
  }
  return ECDNA_B200_OK;
}

// ---------------------------------------------------------------------------------------------
// small utility kernels: ABC prior draws, compaction of accepted draws
// ---------------------------------------------------------------------------------------------
__global__ void prior_kernel(uint32_t seed_lo, uint32_t seed_hi, uint64_t idx_begin, uint32_t n, float b0, float lo1,
                             float hi1, float lo2, float hi2, float lo3, float hi3, float* out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t idx = idx_begin + i;
  const uint4 x = philox4x32_10(0xABC0ABC0u, 0xFFFFFFFFu, (uint32_t)idx, (uint32_t)(idx >> 32), seed_lo, seed_hi);
  const float s = 5.9604644775390625e-08f;  // 2^-24
  const float u1 = __uint2float_rn(x.x >> 8) * s, u2 = __uint2float_rn(x.y >> 8) * s, u3 = __uint2float_rn(x.z >> 8) * s;
  out[4 * (size_t)i + 0] = b0;
  out[4 * (size_t)i + 1] = __fmaf_rn(u1, hi1 - lo1, lo1);
  out[4 * (size_t)i + 2] = __fmaf_rn(u2, hi2 - lo2, lo2);
  out[4 * (size_t)i + 3] = __fmaf_rn(u3, hi3 - lo3, lo3);
}

}  // namespace

namespace ecdna {

int sparse_prepare(ecdna_b200_ctx* ctx, const ecdna_b200_params_t* p, uint64_t idx_begin, uint64_t n_runs,
                   const ecdna_b200_results_t* results, uint64_t* words) {
  static const ecdna_b200_results_t none{};
  const int rc = run_common(ctx, p, idx_begin, n_runs, results ? results : &none, ctx->stream, false, true);
  if (rc) return rc;
  *words = ctx->sp.words;
  return ECDNA_B200_OK;
}

int sparse_fetch(ecdna_b200_ctx* ctx, ecdna_b200_dist_t* final_dist, ecdna_b200_dist_t* snap_dist,
                 ecdna_b200_dist_t* sub_dist, uint32_t* arena, uint64_t base) {
  if (!ctx->sp.valid) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "no sparse batch on the device: call ecdna_b200_run_sparse first");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const auto& sp = ctx->sp;
  if (arena && sp.words && !sp.packed) {
    SparseArgs sa{};
    sa.n_runs = (uint32_t)sp.n_runs; sa.n_snap = (uint32_t)sp.n_snap; sa.n_sub = (uint32_t)sp.n_sub; sa.stride = sp.stride;
    sa.rows = sp.rows;
    sa.hist = (const uint32_t*)ctx->cols[C_HIST].p; sa.snap_hist = (const uint32_t*)ctx->cols[C_SNAPHIST].p;
    sa.sub_hist = (const uint32_t*)ctx->cols[C_SUBHIST].p;
    sa.snap_count = (const uint32_t*)ctx->cols[C_SNAPCOUNT].p; sa.time = (const float*)ctx->cols[C_TIME].p;
    sa.snap_time = (const float*)ctx->cols[C_SNAPTIME].p; sa.stop = (const uint32_t*)ctx->cols[C_STOP].p;
    sa.desc = (ecdna_b200_dist_t*)ctx->sp_desc.p; sa.len = (uint32_t*)ctx->sp_len.p; sa.bsum = (unsigned long long*)ctx->sp_bsum.p;
    CU(ctx->sp_arena.ensure((size_t)sp.words * 4));
    sa.arena = (uint32_t*)ctx->sp_arena.p;
    sparse_pack<<<(unsigned)((sa.rows + 7) / 8), 256, 0, st>>>(sa);
    CU(cudaGetLastError());
    ctx->timing.kernel_launches += 1;
    ctx->sp.packed = true;
  }
  const ecdna_b200_dist_t* d = (const ecdna_b200_dist_t*)ctx->sp_desc.p;
  const size_t ds = sizeof(ecdna_b200_dist_t);
  if (final_dist) { CU(cudaMemcpyAsync(final_dist, d, sp.n_runs * ds, cudaMemcpyDeviceToHost, st)); ctx->timing.d2h_bytes += sp.n_runs * ds; }
  if (snap_dist && sp.n_snap) {
    CU(cudaMemcpyAsync(snap_dist, d + sp.n_runs, sp.n_runs * sp.n_snap * ds, cudaMemcpyDeviceToHost, st));
    ctx->timing.d2h_bytes += sp.n_runs * sp.n_snap * ds;
  }
  if (sub_dist && sp.n_sub) {
    CU(cudaMemcpyAsync(sub_dist, d + sp.n_runs * (1 + sp.n_snap), sp.n_runs * sp.n_sub * ds, cudaMemcpyDeviceToHost, st));
    ctx->timing.d2h_bytes += sp.n_runs * sp.n_sub * ds;
  }
  if (arena && sp.words) {
    CU(cudaMemcpyAsync(arena + base, ctx->sp_arena.p, (size_t)sp.words * 4, cudaMemcpyDeviceToHost, st));
    ctx->timing.d2h_bytes += sp.words * 4;
  }
  CU(cudaEventRecord(ctx->ev_end, st));
  CU(cudaStreamSynchronize(st));
  if (base) {
    if (final_dist) for (uint64_t i = 0; i < sp.n_runs; ++i) final_dist[i].offset += base;
    if (snap_dist) for (uint64_t i = 0; i < sp.n_runs * sp.n_snap; ++i) snap_dist[i].offset += base;
    if (sub_dist) for (uint64_t i = 0; i < sp.n_runs * sp.n_sub; ++i) sub_dist[i].offset += base;
  }
  return ECDNA_B200_OK;
}

}  // namespace ecdna

extern "C" {

int ecdna_b200_run_sparse(ecdna_b200_ctx* ctx, const ecdna_b200_params_t* params, uint64_t idx_begin, uint64_t n_runs,
                          const ecdna_b200_results_t* results, ecdna_b200_sparse_t* sparse) {
  if (!ctx) return ECDNA_B200_ERR_BAD_PARAMS;
  if (!sparse) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "sparse is NULL");
  uint64_t words = 0;
  const int rc = sparse_prepare(ctx, params, idx_begin, n_runs, results, &words);
  if (rc) return rc;
  return ecdna_b200_sparse_fetch(ctx, sparse);
}

int ecdna_b200_sparse_fetch(ecdna_b200_ctx* ctx, ecdna_b200_sparse_t* sparse) {
  if (!ctx) return ECDNA_B200_ERR_BAD_PARAMS;
  if (!sparse) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "sparse is NULL");
  if (!ctx->sp.valid) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "no sparse batch on the device: call ecdna_b200_run_sparse first");
  sparse->arena_used = ctx->sp.words;
  const bool fits = ctx->sp.words == 0 || (sparse->arena && sparse->arena_words >= ctx->sp.words);
  const int rc = sparse_fetch(ctx, sparse->final_dist, sparse->snap_dist, sparse->sub_dist, fits ? sparse->arena : nullptr, 0);
  if (rc) return rc;
  if (!fits)
    return fail(ctx, ECDNA_B200_ERR_ARENA, "the batch needs an arena of " + std::to_string(ctx->sp.words) + " words, the caller gave " +
                                               std::to_string(sparse->arena ? sparse->arena_words : 0));
  return ECDNA_B200_OK;
}

int ecdna_b200_abi_version(void) { return ECDNA_B200_ABI_VERSION; }

int ecdna_b200_query_sizes(const ecdna_b200_params_t* params, uint64_t n_runs, ecdna_b200_result_sizes_t* sizes) {
  if (!params || !sizes || params->abi_version != ECDNA_B200_ABI_VERSION || n_runs == 0 || n_runs >= 0xFFFFFFF0ull)
    return ECDNA_B200_ERR_BAD_PARAMS;
  static_assert(sizeof(ecdna_b200_result_sizes_t) == C_COUNT * sizeof(uint64_t), "one size per result column");
  const uint32_t stride = params->hist_stride ? params->hist_stride : 512u;
  uint64_t* out = reinterpret_cast<uint64_t*>(sizes);
  for (int c = 0; c < C_COUNT; ++c) out[c] = (uint64_t)col_bytes(c, params, stride) * n_runs;
  if (!params->abc_enabled) sizes->abc_distance = sizes->abc_accept = 0;
  return ECDNA_B200_OK;
}

int ecdna_b200_plan(uint64_t n_runs, uint32_t tile_width, uint32_t slice_events, uint32_t sm_count, uint32_t max_blocks_per_sm,
                    uint32_t* lanes, uint32_t* blocks_per_sm, uint32_t* tiles, uint32_t* sliced) {
  if (n_runs == 0 || sm_count == 0 || max_blocks_per_sm == 0 || !lanes || !blocks_per_sm || !tiles || !sliced)
    return ECDNA_B200_ERR_BAD_PARAMS;
  const uint32_t L = tile_width ? tile_width : default_tile_width(n_runs, (int)sm_count, true, true);
  if (L != 1 && L != 2 && L != 4 && L != 8 && L != 16 && L != 32) return ECDNA_B200_ERR_BAD_PARAMS;
  int w = 0;
  bool sl = false;
  const int tiles_per_block = (L == 1 ? block_threads<1>() : kBlockThreads) / (int)L;
  plan_launch(n_runs, (int)sm_count, (int)max_blocks_per_sm, tiles_per_block, slice_events, (int)L, &w, &sl);
  uint64_t grid = (uint64_t)sm_count * (uint64_t)w;
  const uint64_t need = (n_runs + tiles_per_block - 1) / tiles_per_block;
  if (need < grid) grid = need;
  *lanes = L;
  *blocks_per_sm = (uint32_t)w;
  *tiles = (uint32_t)(grid * tiles_per_block);
  *sliced = sl ? 1u : 0u;
  return ECDNA_B200_OK;
}

int ecdna_b200_create(int device, ecdna_b200_ctx** out) {
  if (!out) return ECDNA_B200_ERR_BAD_PARAMS;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return ECDNA_B200_ERR_NO_DEVICE;
  if (device < 0 || device >= count) return ECDNA_B200_ERR_BAD_PARAMS;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return ECDNA_B200_ERR_CUDA;
  if (prop.major != 10) return ECDNA_B200_ERR_NO_DEVICE;  // the fatbin holds sm_100a code only
  ecdna_b200_ctx* ctx = new ecdna_b200_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&ctx->ev_begin) != cudaSuccess || cudaEventCreate(&ctx->ev_k0) != cudaSuccess ||
      cudaEventCreate(&ctx->ev_k1) != cudaSuccess || cudaEventCreate(&ctx->ev_end) != cudaSuccess) {
    delete ctx;
    return ECDNA_B200_ERR_CUDA;
  }
  *out = ctx;
  return ECDNA_B200_OK;
}

void ecdna_b200_destroy(ecdna_b200_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  ecdna_b200_comm_release(ctx);
  DevBuf* bufs[] = {&ctx->init_k, &ctx->init_c, &ctx->snap, &ctx->rates, &ctx->replay, &ctx->replay_off,
                    &ctx->abc_cdf, &ctx->arena, &ctx->counters, &ctx->scratch, &ctx->park_list, &ctx->park_rec, &ctx->park_list2, &ctx->park_rec2, &ctx->order, &ctx->order_hist, &ctx->ts_ring, &ctx->ts_rec, &ctx->sub_sizes, &ctx->hist_tmp,
                    &ctx->cells, &ctx->zig, &ctx->pack_idx, &ctx->pack_out, &ctx->pack_cnt, &ctx->sp_desc, &ctx->sp_len,
                    &ctx->sp_bsum, &ctx->sp_arena, &ctx->smc_prev, &ctx->smc_cum, &ctx->smc_new, &ctx->smc_parent,
                    &ctx->smc_tiles, &ctx->smc_sum, &ctx->smc_cov};
  for (DevBuf* b : bufs) b->release();
  for (auto& b : ctx->cols) b.release();
  cudaEventDestroy(ctx->ev_begin); cudaEventDestroy(ctx->ev_k0); cudaEventDestroy(ctx->ev_k1); cudaEventDestroy(ctx->ev_end);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* ecdna_b200_last_error(const ecdna_b200_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context"; }

int ecdna_b200_run(ecdna_b200_ctx* ctx, const ecdna_b200_params_t* params, uint64_t idx_begin, uint64_t n_runs,
                   const ecdna_b200_results_t* results) {
  if (!ctx) return ECDNA_B200_ERR_BAD_PARAMS;
  return run_common(ctx, params, idx_begin, n_runs, results, ctx->stream, false);
}

int ecdna_b200_run_device(ecdna_b200_ctx* ctx, const ecdna_b200_params_t* params, uint64_t idx_begin, uint64_t n_runs,
                          const ecdna_b200_results_t* results, void* cuda_stream) {
  if (!ctx) return ECDNA_B200_ERR_BAD_PARAMS;
  return run_common(ctx, params, idx_begin, n_runs, results, cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream, true);
}

int ecdna_b200_get_timing(ecdna_b200_ctx* ctx, ecdna_b200_timing_t* t) {
  if (!ctx || !t) return ECDNA_B200_ERR_BAD_PARAMS;
  CU(cudaSetDevice(ctx->device));
  CU(cudaEventSynchronize(ctx->ev_k1));
  CU(cudaEventElapsedTime(&ctx->timing.kernel_ms, ctx->ev_k0, ctx->ev_k1));
  if (ctx->have_total) {
    CU(cudaEventSynchronize(ctx->ev_end));
    CU(cudaEventElapsedTime(&ctx->timing.total_ms, ctx->ev_begin, ctx->ev_end));
  }
  unsigned long long tot[kTotalsCount];
  CU(cudaMemcpy(tot, (char*)ctx->counters.p + kTotalsOffset, sizeof tot, cudaMemcpyDeviceToHost));
  ctx->timing.n_finished = tot[7];
  ctx->timing.n_slices = tot[5];
  ctx->timing.n_idle_spells = tot[6];
  ctx->timing.total_events = tot[0];
  // SURVEY 8(d): division = 4K + 24 + 16, death = 4K + 8 + 16, ecDNA- event = 16 bytes
  ctx->timing.alg_bytes = 4ull * tot[1] + 24ull * tot[2] + 8ull * tot[3] + 16ull * tot[0];
  ctx->timing.n_spilled = (uint32_t)tot[4];
  *t = ctx->timing;
  if (ctx->expect_finished && tot[7] != ctx->expect_finished)
    return fail(ctx, ECDNA_B200_ERR_INTERNAL, "internal error: " + std::to_string(tot[7]) + " of " + std::to_string(ctx->expect_finished) + " replicates finished");
  return ECDNA_B200_OK;
}

int ecdna_b200_abc_draw_priors(ecdna_b200_ctx* ctx, uint64_t seed, uint64_t idx_begin, uint64_t n_runs, float b0,
                               const float b1_range[2], const float d0_range[2], const float d1_range[2],
                               float* rates_out) {
  if (!ctx || !rates_out || n_runs == 0 || n_runs >= (1ull << 32)) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "bad prior request");
  CU(cudaSetDevice(ctx->device));
  CU(ctx->rates.ensure(n_runs * 16));
  const uint32_t n = (uint32_t)n_runs;
  // (the grid in 64 bits: (n + 255) / 256 in 32 bits wraps to a few blocks for n > 2^32 - 256)
  prior_kernel<<<(uint32_t)((n_runs + 255) / 256), 256, 0, ctx->stream>>>(
      (uint32_t)seed, (uint32_t)(seed >> 32), idx_begin, n, b0, b1_range[0], b1_range[1], d0_range[0], d0_range[1],
      d1_range[0], d1_range[1], (float*)ctx->rates.p);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(rates_out, ctx->rates.p, n_runs * 16, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return ECDNA_B200_OK;
}

int ecdna_b200_abc_draw_priors_device(ecdna_b200_ctx* ctx, uint64_t seed, uint64_t idx_begin, uint64_t n_runs, float b0,
                                      const float b1_range[2], const float d0_range[2], const float d1_range[2],
                                      float* rates_dev, void* cuda_stream) {
  if (!ctx || !rates_dev || n_runs == 0 || n_runs >= (1ull << 32)) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "bad prior request");
  CU(cudaSetDevice(ctx->device));
  const uint32_t n = (uint32_t)n_runs;
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
  prior_kernel<<<(uint32_t)((n_runs + 255) / 256), 256, 0, st>>>((uint32_t)seed, (uint32_t)(seed >> 32), idx_begin, n, b0,
                                                                 b1_range[0], b1_range[1], d0_range[0], d0_range[1],
                                                                 d1_range[0], d1_range[1], rates_dev);
  CU(cudaGetLastError());
  return ECDNA_B200_OK;
}

}  // extern "C"

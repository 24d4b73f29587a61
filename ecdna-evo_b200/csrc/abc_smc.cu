// abc_smc.cu -- ABC-SMC (ABC population Monte Carlo) over the prior box of ecdna_b200_abc_draw_priors: the proposal
// kernel, the truncation normalisers, the all-pairs importance-weight kernel, and the driver loop over an
// ecdna_b200_multi handle (include/ecdna_b200.h, DESIGN.md section 9).
//
// Determinism: draw i's proposal reads Philox keyed (seed, i) and the previous population only; draw i is simulated
// as replicate i; the weight sums run over the previous population in index order with a fixed tree per tile and no
// atomics.  So a run gives the same bits whatever the chunk size and the number of GPUs.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "engine.cuh"

using namespace ecdna;

namespace {

constexpr uint32_t kProposalDomain = 0x5A1C5A1Cu;  // Philox counter word 0 of the proposals (the prior draws: 0xABC0ABC0)
constexpr int kPairBlock = 128;                     // new particles per block = previous particles per shared tile

struct Box {
  float lo[3], hi[3];
  double sigma[3];
  uint32_t free_mask;  // bit k: parameter k + 1 is perturbed (lo < hi and sigma > 0)
};

// u in [0, 1) from 53 bits of two Philox words (numpy's random_sample construction)
__device__ __forceinline__ double u53(uint32_t a, uint32_t b) {
  return __dadd_rn(__dmul_rn((double)(a >> 5), 67108864.0), (double)(b >> 6)) * 1.1102230246251565e-16;
}

__global__ void smc_propose_kernel(uint32_t seed_lo, uint32_t seed_hi, uint64_t idx_begin, uint32_t n,
                                   const float4* __restrict__ prev, const double* __restrict__ cum, uint32_t M, Box box,
                                   float4* __restrict__ out, uint32_t* __restrict__ parent_out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t idx = idx_begin + i;
  const uint4 x = philox4x32_10(kProposalDomain, 0u, (uint32_t)idx, (uint32_t)(idx >> 32), seed_lo, seed_hi);
  const uint4 y = philox4x32_10(kProposalDomain, 1u, (uint32_t)idx, (uint32_t)(idx >> 32), seed_lo, seed_hi);
  // parent: the first j with cum[j] > u * cum[M-1] (np.searchsorted(cum, target, side="right"))
  const double target = __dmul_rn(u53(x.x, x.y), cum[M - 1]);
  uint32_t l = 0, h = M - 1;
  while (l < h) {
    const uint32_t mid = (l + h) >> 1;
    if (cum[mid] > target) h = mid;
    else l = mid + 1;
  }
  const float4 p = prev[l];
  float v[3] = {p.y, p.z, p.w};
  const double u[3] = {u53(x.z, x.w), u53(y.x, y.y), u53(y.z, y.w)};
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    if (!(box.free_mask & (1u << k))) continue;
    // Gaussian around the parent truncated to [lo, hi] by inverse-CDF sampling: no rejection loop
    const double s = box.sigma[k], c = (double)v[k];
    const double a = __ddiv_rn(__dsub_rn((double)box.lo[k], c), s), b = __ddiv_rn(__dsub_rn((double)box.hi[k], c), s);
    const double fa = normcdf(a), fb = normcdf(b);
    const double z = normcdfinv(__dadd_rn(fa, __dmul_rn(u[k], __dsub_rn(fb, fa))));
    const float t = (float)__dadd_rn(c, __dmul_rn(s, z));
    v[k] = fminf(fmaxf(t, box.lo[k]), box.hi[k]);  // (rounding; and z = -inf when the sum rounds to 0)
  }
  out[i] = make_float4(p.x, v[0], v[1], v[2]);
  parent_out[i] = l;
}

// previous particle j as one float4 of the pair kernel's tiles: its parameters and W_j / Z_j, where
// Z_j = prod_k (Phi(b_jk) - Phi(a_jk)) is the mass of j's perturbation kernel inside the box
__global__ void smc_tiles_kernel(const float4* __restrict__ prev, const double* __restrict__ w, uint32_t M, Box box,
                                 float4* __restrict__ tiles) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= M) return;
  const float4 p = prev[j];
  const float v[3] = {p.y, p.z, p.w};
  double z = 1.0;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    if (!(box.free_mask & (1u << k))) continue;
    const double s = box.sigma[k], c = (double)v[k];
    const double a = __ddiv_rn(__dsub_rn((double)box.lo[k], c), s), b = __ddiv_rn(__dsub_rn((double)box.hi[k], c), s);
    z = __dmul_rn(z, __dsub_rn(normcdf(b), normcdf(a)));
  }
  tiles[j] = make_float4(v[0], v[1], v[2], (float)__ddiv_rn(w[j], z));
}

__device__ __forceinline__ float ex2_neg(float q) {  // 2^-q, q >= 0
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-q));
  return r;
}

// S_i = sum_j (W_j / Z_j) prod_k phi((theta_ik - theta_jk) / sigma_k) up to a constant factor common to every i:
// one thread per new particle, the previous population streamed through shared memory in tiles of kPairBlock.
// sc[k] = sqrt(log2(e) / 2) / sigma_k (0 for a fixed parameter), so that the product is 2^-(sum_k (d_k sc_k)^2).
// Every tile is summed in f32 over four interleaved partial sums in a fixed order, the tiles in f64.
__global__ void __launch_bounds__(kPairBlock) smc_pair_kernel(const float4* __restrict__ cand, uint32_t N,
                                                              const float4* __restrict__ tiles, uint32_t M, float sc1,
                                                              float sc2, float sc3, double* __restrict__ sum_out) {
  __shared__ float4 sh[kPairBlock];
  const uint32_t i = blockIdx.x * kPairBlock + threadIdx.x;
  const float4 x = i < N ? cand[i] : make_float4(0.f, 0.f, 0.f, 0.f);
  double total = 0.0;
  for (uint32_t base = 0; base < M; base += kPairBlock) {
    __syncthreads();
    const uint32_t j = base + threadIdx.x;
    sh[threadIdx.x] = j < M ? tiles[j] : make_float4(0.f, 0.f, 0.f, 0.f);  // (weight 0: adds nothing)
    __syncthreads();
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 8
    for (int jj = 0; jj < kPairBlock; ++jj) {
      const float4 t = sh[jj];
      const float d1 = __fmul_rn(__fsub_rn(x.y, t.x), sc1);
      const float d2 = __fmul_rn(__fsub_rn(x.z, t.y), sc2);
      const float d3 = __fmul_rn(__fsub_rn(x.w, t.z), sc3);
      const float q = __fmaf_rn(d3, d3, __fmaf_rn(d2, d2, __fmul_rn(d1, d1)));
      acc[jj & 3] = __fmaf_rn(t.w, ex2_neg(q), acc[jj & 3]);
    }
    total = __dadd_rn(total, (double)__fadd_rn(__fadd_rn(acc[0], acc[1]), __fadd_rn(acc[2], acc[3])));
  }
  if (i < N) sum_out[i] = total;
}

bool range_ok(const float* r) { return r && std::isfinite(r[0]) && std::isfinite(r[1]) && r[0] >= 0.f && r[0] <= r[1]; }

int make_box(ecdna_b200_ctx* ctx, const double sigma[3], const float* r1, const float* r2, const float* r3, Box* box) {
  if (!sigma) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "sigma is NULL");
  if (!range_ok(r1) || !range_ok(r2) || !range_ok(r3))
    return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "every prior range needs 0 <= lo <= hi (finite)");
  const float* r[3] = {r1, r2, r3};
  box->free_mask = 0;
  for (int k = 0; k < 3; ++k) {
    if (!(sigma[k] >= 0.0) || !std::isfinite(sigma[k])) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "sigma must be finite and >= 0");
    box->lo[k] = r[k][0];
    box->hi[k] = r[k][1];
    box->sigma[k] = sigma[k];
    // (sigma = 0: every particle of the population has the same value; the kernel is a point mass there)
    if (r[k][0] < r[k][1] && sigma[k] > 0.0) box->free_mask |= 1u << k;
  }
  return ECDNA_B200_OK;
}

float rho_of(const float* d, const float* thr, uint32_t stop) {
  const uint32_t code = stop & 0xFFu;
  if (code == ECDNA_B200_STOP_COPY_OVERFLOW || code == ECDNA_B200_STOP_HIST_OVERFLOW || (stop & ECDNA_B200_FLAG_HIST_TRUNCATED))
    return INFINITY;
  float rho = 0.f;
  for (int j = 0; j < 4; ++j) {
    if (!(thr[j] >= 0.f)) continue;  // disabled distance
    if (std::isnan(d[j])) return INFINITY;
    if (thr[j] == 0.f) {
      if (d[j] != 0.f) return INFINITY;
    } else {
      rho = std::max(rho, d[j] / thr[j]);
    }
  }
  return rho;
}

double ms_since(std::chrono::steady_clock::time_point t0) {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
}

}  // namespace

extern "C" {

int ecdna_b200_abc_smc_propose(ecdna_b200_ctx* ctx, uint64_t seed, uint64_t idx_begin, uint64_t n, const float* prev_rates,
                               const double* cum_weights, uint32_t M, const double sigma[3], const float b1_range[2],
                               const float d0_range[2], const float d1_range[2], float* rates_out, uint32_t* parent_out) {
  if (!ctx) return ECDNA_B200_ERR_BAD_PARAMS;
  if (!prev_rates || !cum_weights || !rates_out || !parent_out || M == 0 || n == 0 || n >= (1ull << 32))
    return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "bad proposal request (buffers, M >= 1, n in [1, 2^32))");
  if (!(cum_weights[M - 1] > 0.0) || !std::isfinite(cum_weights[M - 1]))
    return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "the cumulative weights must end with a finite value > 0");
  Box box;
  int rc = make_box(ctx, sigma, b1_range, d0_range, d1_range, &box);
  if (rc) return rc;
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  CU(ctx->smc_prev.ensure((size_t)M * 16));
  CU(ctx->smc_cum.ensure((size_t)M * 8));
  CU(ctx->smc_new.ensure((size_t)n * 16));
  CU(ctx->smc_parent.ensure((size_t)n * 4));
  CU(cudaMemcpyAsync(ctx->smc_prev.p, prev_rates, (size_t)M * 16, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(ctx->smc_cum.p, cum_weights, (size_t)M * 8, cudaMemcpyHostToDevice, st));
  const uint32_t n32 = (uint32_t)n;
  // (grids in 64 bits: (n + 255) / 256 in 32 bits wraps to a few blocks for n > 2^32 - 256)
  smc_propose_kernel<<<(uint32_t)((n + 255) / 256), 256, 0, st>>>((uint32_t)seed, (uint32_t)(seed >> 32), idx_begin,
                                                                  n32, (const float4*)ctx->smc_prev.p,
                                                                  (const double*)ctx->smc_cum.p, M, box,
                                                                  (float4*)ctx->smc_new.p, (uint32_t*)ctx->smc_parent.p);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(rates_out, ctx->smc_new.p, (size_t)n * 16, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(parent_out, ctx->smc_parent.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return ECDNA_B200_OK;
}

int ecdna_b200_abc_smc_weights(ecdna_b200_ctx* ctx, const float* new_rates, uint32_t N, const float* prev_rates,
                               const double* prev_weights, uint32_t M, const double sigma[3], const float b1_range[2],
                               const float d0_range[2], const float d1_range[2], double* weights_out) {
  if (!ctx) return ECDNA_B200_ERR_BAD_PARAMS;
  if (!new_rates || !prev_rates || !prev_weights || !weights_out || N == 0 || M == 0)
    return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "bad weight request (buffers, N >= 1, M >= 1)");
  Box box;
  int rc = make_box(ctx, sigma, b1_range, d0_range, d1_range, &box);
  if (rc) return rc;
  float sc[3] = {0.f, 0.f, 0.f};
  for (int k = 0; k < 3; ++k)
    if (box.free_mask & (1u << k)) sc[k] = (float)(std::sqrt(0.5 / std::log(2.0)) / box.sigma[k]);  // log2(e)/2 = 1/(2 ln 2)
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  CU(ctx->smc_prev.ensure((size_t)M * 16));
  CU(ctx->smc_cum.ensure((size_t)M * 8));
  CU(ctx->smc_tiles.ensure((size_t)M * 16));
  CU(ctx->smc_new.ensure((size_t)N * 16));
  CU(ctx->smc_sum.ensure((size_t)N * 8));
  CU(cudaMemcpyAsync(ctx->smc_prev.p, prev_rates, (size_t)M * 16, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(ctx->smc_cum.p, prev_weights, (size_t)M * 8, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(ctx->smc_new.p, new_rates, (size_t)N * 16, cudaMemcpyHostToDevice, st));
  smc_tiles_kernel<<<(uint32_t)(((uint64_t)M + 255) / 256), 256, 0, st>>>((const float4*)ctx->smc_prev.p,
                                                                           (const double*)ctx->smc_cum.p, M, box,
                                                                           (float4*)ctx->smc_tiles.p);
  smc_pair_kernel<<<(uint32_t)(((uint64_t)N + kPairBlock - 1) / kPairBlock), kPairBlock, 0, st>>>(
      (const float4*)ctx->smc_new.p, N, (const float4*)ctx->smc_tiles.p, M, sc[0], sc[1], sc[2], (double*)ctx->smc_sum.p);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(weights_out, ctx->smc_sum.p, (size_t)N * 8, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  double total = 0.0;
  for (uint32_t i = 0; i < N; ++i) {
    if (!(weights_out[i] > 0.0) || !std::isfinite(weights_out[i]))
      return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "particle " + std::to_string(i) + " has proposal density 0 under the previous population");
    weights_out[i] = 1.0 / weights_out[i];
    total += weights_out[i];
  }
  for (uint32_t i = 0; i < N; ++i) weights_out[i] /= total;
  return ECDNA_B200_OK;
}

int ecdna_b200_abc_smc(ecdna_b200_multi* m, const ecdna_b200_params_t* params, const ecdna_b200_smc_options_t* o,
                       ecdna_b200_smc_result_t* r) {
  if (!m) return ECDNA_B200_ERR_BAD_PARAMS;
  auto bad = [&](const std::string& msg) { m->err = msg; return ECDNA_B200_ERR_BAD_PARAMS; };
  if (!params || !o || !r) return bad("params, options and result must not be NULL");
  if (params->abi_version != ECDNA_B200_ABI_VERSION) return bad("abi_version mismatch");
  if (o->population == 0) return bad("population must be >= 1");
  if (!(o->quantile > 0.0 && o->quantile < 1.0)) return bad("quantile must be in (0, 1)");
  if (o->max_generations == 0) return bad("max_generations must be >= 1");
  if (!params->abc_enabled || !params->abc_target_hist || params->abc_target_len == 0)
    return bad("ABC-SMC needs abc_enabled and a target distribution");
  const float* thr = params->abc_thresholds;
  if (!(thr[0] >= 0.f) && !(thr[1] >= 0.f) && !(thr[2] >= 0.f) && !(thr[3] >= 0.f)) return bad("every ABC threshold is disabled");
  if (!range_ok(o->b1_range) || !range_ok(o->d0_range) || !range_ok(o->d1_range))
    return bad("every prior range needs 0 <= lo <= hi (finite)");
  if (params->rates_per_run) return bad("rates_per_run must be NULL: the driver sets the rates of every draw");

  ecdna_b200_ctx* ctx0 = m->ctx[0];
  const uint32_t M = o->population;
  const uint64_t limit = o->max_simulations ? o->max_simulations : UINT64_MAX;
  const uint64_t n_gpus = m->ctx.size();
  // one population: the accepted draws in index order
  struct Pop {
    std::vector<float> rates, dist, rho;
    std::vector<uint64_t> idx, parent, cells;
    std::vector<double> w;
    void resize(uint32_t n) {
      rates.assign((size_t)n * 4, 0.f); dist.assign((size_t)n * 4, 0.f); rho.assign(n, 0.f);
      idx.assign(n, 0); parent.assign(n, UINT64_MAX); cells.assign(n, 0); w.assign(n, 0.0);
    }
  } cur, prev;
  cur.resize(M);
  prev.resize(M);
  std::vector<double> cum(M);
  double sigma[3] = {0.0, 0.0, 0.0};
  std::vector<float> rates;
  std::vector<uint32_t> parent, stop;
  std::vector<float> dist;
  std::vector<uint8_t> accept;
  std::vector<uint64_t> nminus, nplus;

  float eps = INFINITY;
  uint64_t next = o->idx_begin, used = 0;
  double prev_rate = 0.0;
  r->generations = 0;
  r->status = ECDNA_B200_SMC_MAX_GENERATIONS;
  for (uint32_t g = 0; g < o->max_generations; ++g) {
    ecdna_b200_params_t p = *params;
    for (int j = 0; j < 4; ++j) p.abc_thresholds[j] = thr[j] > 0.f ? thr[j] * eps : thr[j];
    const uint64_t start = next;
    uint64_t pos = start, simulated = 0, end = 0, last_n = 0;
    uint32_t acc = 0;
    double t_sim = 0.0, t_prop = 0.0, t_w = 0.0;
    while (acc < M) {
      const uint64_t left = limit - used - (pos - start);
      if (left == 0) break;
      uint64_t n = o->chunk;
      if (n == 0) {  // enough draws for the acceptances still missing at the rate seen so far, 20 % to spare
        // (draws past the M-th acceptance are simulated for nothing; below a few thousand per GPU a launch is
        //  bound by its longest replicate rather than by its size)
        const uint64_t lo_n = 4096ull * n_gpus, hi_n = 4ull << 20;
        const double rate = simulated ? (double)acc / (double)simulated : prev_rate * o->quantile;
        if (rate > 0.0) n = (uint64_t)std::min(1.2 * (double)(M - acc) / rate + 1.0, (double)hi_n);
        else n = last_n ? 4 * last_n : lo_n;
        n = std::min(std::max(n, lo_n), hi_n);
      }
      n = std::min<uint64_t>(std::min<uint64_t>(n, left), 0xFFFFFFF0ull - 1);
      last_n = n;
      rates.resize(n * 4); parent.resize(n); stop.resize(n); dist.resize(n * 4); accept.resize(n);
      nminus.resize(n); nplus.resize(n);
      auto t0 = std::chrono::steady_clock::now();
      int rc = g == 0 ? ecdna_b200_abc_draw_priors(ctx0, params->seed, pos, n, params->b0, o->b1_range, o->d0_range, o->d1_range, rates.data())
                      : ecdna_b200_abc_smc_propose(ctx0, params->seed, pos, n, prev.rates.data(), cum.data(), M, sigma, o->b1_range,
                                                   o->d0_range, o->d1_range, rates.data(), parent.data());
      if (rc != ECDNA_B200_OK) { m->err = std::string("proposals: ") + ecdna_b200_last_error(ctx0); return rc; }
      t_prop += ms_since(t0);
      p.rates_per_run = rates.data();
      ecdna_b200_results_t res;
      std::memset(&res, 0, sizeof res);
      res.stop_reason = stop.data(); res.nminus = nminus.data(); res.nplus = nplus.data();
      res.abc_distance = dist.data(); res.abc_accept = accept.data();
      t0 = std::chrono::steady_clock::now();
      rc = ecdna_b200_multi_run(m, &p, pos, n, &res);
      if (rc != ECDNA_B200_OK) return rc;
      t_sim += ms_since(t0);
      simulated += n;
      for (uint64_t i = 0; i < n && acc < M; ++i) {
        if (!accept[i]) continue;
        const float rho = rho_of(&dist[4 * i], thr, stop[i]);
        if (!(rho < INFINITY)) continue;
        std::memcpy(&cur.rates[4 * (size_t)acc], &rates[4 * i], 16);
        std::memcpy(&cur.dist[4 * (size_t)acc], &dist[4 * i], 16);
        cur.rho[acc] = rho;
        cur.idx[acc] = pos + i;
        cur.parent[acc] = g == 0 ? UINT64_MAX : prev.idx[parent[i]];
        cur.cells[acc] = nminus[i] + nplus[i];
        if (++acc == M) end = pos + i + 1;
      }
      pos += n;
    }
    if (acc < M) {  // the budget ends the run inside this generation: the ones before it are the result
      r->status = ECDNA_B200_SMC_BUDGET;
      break;
    }
    const uint64_t consumed = end - start;
    used += consumed;
    next = end;
    prev_rate = (double)M / (double)consumed;
    auto t0 = std::chrono::steady_clock::now();
    if (g == 0) std::fill(cur.w.begin(), cur.w.end(), 1.0 / M);
    else {
      const int rc = ecdna_b200_abc_smc_weights(ctx0, cur.rates.data(), M, prev.rates.data(), prev.w.data(), M, sigma,
                                                o->b1_range, o->d0_range, o->d1_range, cur.w.data());
      if (rc != ECDNA_B200_OK) { m->err = std::string("weights: ") + ecdna_b200_last_error(ctx0); return rc; }
    }
    t_w = ms_since(t0);
    double w2 = 0.0;
    for (uint32_t i = 0; i < M; ++i) w2 += cur.w[i] * cur.w[i];
    const size_t off = (size_t)g * M;
    if (r->idx) std::copy(cur.idx.begin(), cur.idx.end(), r->idx + off);
    if (r->parent_idx) std::copy(cur.parent.begin(), cur.parent.end(), r->parent_idx + off);
    if (r->rates) std::copy(cur.rates.begin(), cur.rates.end(), r->rates + 4 * off);
    if (r->distance) std::copy(cur.dist.begin(), cur.dist.end(), r->distance + 4 * off);
    if (r->weight) std::copy(cur.w.begin(), cur.w.end(), r->weight + off);
    if (r->cells) std::copy(cur.cells.begin(), cur.cells.end(), r->cells + off);
    if (r->epsilon) r->epsilon[g] = eps;
    if (r->consumed) r->consumed[g] = consumed;
    if (r->simulated) r->simulated[g] = simulated;
    if (r->ess) r->ess[g] = 1.0 / w2;
    if (r->time_ms) { r->time_ms[3 * g] = (float)t_sim; r->time_ms[3 * g + 1] = (float)t_prop; r->time_ms[3 * g + 2] = (float)t_w; }
    r->generations = g + 1;
    if (eps == 1.f) {
      r->status = ECDNA_B200_SMC_REACHED;
      break;
    }
    // the next generation: kernel widths (sigma_k^2 = 2 x weighted variance), cumulative weights and tolerance,
    // all sums sequential in index order
    for (int k = 0; k < 3; ++k) {
      double mean = 0.0, var = 0.0;
      for (uint32_t i = 0; i < M; ++i) mean += cur.w[i] * (double)cur.rates[4 * (size_t)i + 1 + k];
      for (uint32_t i = 0; i < M; ++i) {
        const double d = (double)cur.rates[4 * (size_t)i + 1 + k] - mean;
        var += cur.w[i] * d * d;
      }
      sigma[k] = std::sqrt(2.0 * var);
    }
    double c = 0.0;
    for (uint32_t i = 0; i < M; ++i) cum[i] = c += cur.w[i];
    std::vector<float> rho = cur.rho;
    const uint32_t k = std::min<uint32_t>(M, std::max<uint32_t>(1u, (uint32_t)std::ceil(o->quantile * (double)M)));
    std::nth_element(rho.begin(), rho.begin() + (k - 1), rho.end());
    eps = std::min(eps, std::max(1.f, rho[k - 1]));
    std::swap(prev, cur);
  }
  return ECDNA_B200_OK;
}

}  // extern "C"

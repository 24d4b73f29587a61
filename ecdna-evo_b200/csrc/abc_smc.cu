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
#include <type_traits>
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

// ---- correlated kernels: N(c_j, Sigma_j) truncated to the box by sequential conditioning (DESIGN.md section 9) ----
// Over the D free parameters (in the order b1, d0, d1) with L = chol(Sigma): coordinate t is drawn from the normal
// of mean m_t = c_t + sum_{l<t} L_tl e_l and sd L_tt truncated to [lo_t, hi_t] by inverse CDF, e_t = (theta_t - m_t)
// / L_tt.  Its density is prod_t phi(e_t) / (L_tt (Phi(b_t) - Phi(a_t))), e = L^-1 (theta - c).  Packed lower
// triangles are (11, 21, 22, 31, 32, 33).
constexpr double kTail = 5.0;                     // sample intervals beyond +-5 sds in log space
constexpr double kRsqrt2 = 0.70710678118654752440;
constexpr double kLog2e = 1.4426950408889634074;

struct CovArgs {
  float lo[3], hi[3];  // of the free parameters, in free order
  int D, f[3];         // number of free parameters; f[t]: the parameter (0 = b1, 1 = d0, 2 = d1) of free coordinate t
  double L[6], Li[6];  // a shared Sigma: its Cholesky factor and the inverse of that, packed over the free coordinates
};

struct CovRec {  // previous particle j with a per-parent Sigma_j: c_j (free order), log2 weight, L_j^-1
  double c[3], logw, li[6];
};
struct CovRecShared {  // ... and with a shared Sigma, whose L^-1 the pair kernel holds in registers
  double c[3], logw;
};

__host__ __device__ __forceinline__ int tri(int r, int c) { return r * (r + 1) / 2 + c; }  // r >= c

// L over the free coordinates of the packed 3 x 3 Sigma S; false when Sigma is not positive definite there
__host__ __device__ inline bool chol_free(const double* S, const CovArgs& b, double L[6]) {
  for (int t = 0; t < 3 && t < b.D; ++t)
    for (int l = 0; l <= t; ++l) {
      double s = S[tri(b.f[t], b.f[l])];
      for (int m = 0; m < l; ++m) s -= L[tri(t, m)] * L[tri(l, m)];
      if (l < t) {
        L[tri(t, l)] = s / L[tri(l, l)];
      } else {
        if (!(s > 0.0 && s < INFINITY)) return false;
        L[tri(t, t)] = sqrt(s);
      }
    }
  return true;
}

__host__ __device__ inline void tri_inverse(const double L[6], int D, double Li[6]) {
  for (int i = 0; i < 6; ++i) Li[i] = 0.0;
  for (int t = 0; t < 3 && t < D; ++t) {
    Li[tri(t, t)] = 1.0 / L[tri(t, t)];
    for (int l = 0; l < t; ++l) {
      double s = 0.0;
      for (int m = l; m < t; ++m) s += L[tri(t, m)] * Li[tri(m, l)];
      Li[tri(t, l)] = -s / L[tri(t, t)];
    }
  }
}

// log Phi(x) for any x (Phi(x) = exp(-x^2/2) erfcx(-x/sqrt2)/2): finite far below the range of Phi itself
__device__ __forceinline__ double log_phi(double x) { return -0.5 * x * x + log(0.5 * erfcx(-x * kRsqrt2)); }

// log(Phi(b) - Phi(a)), a <= b; an interval on one side of 0 is taken on the positive side, where
// Phi-bar(a) - Phi-bar(b) = Phi-bar(a) (1 - Phi-bar(b) / Phi-bar(a)) has no cancellation
__device__ inline double log_mass(double a, double b) {
  if (b < 0.0) {
    const double t = a;
    a = -b;
    b = -t;
  }
  if (a > 0.0) {
    const double ea = erfcx(a * kRsqrt2);
    const double r = -0.5 * (b - a) * (b + a) + log(erfcx(b * kRsqrt2) / ea);  // log(Phi-bar(b) / Phi-bar(a))
    return -0.5 * a * a + log(0.5 * ea) + log(-expm1(r));
  }
  return log(normcdf(b) - normcdf(a));
}

// log(phi(e) sqrt(2 pi) / (Phi(b) - Phi(a))) for e in [a, b], given ea = e - a and be = b - e from the edge distances.
// In a tail it is -(e - a)(e + a)/2 - log(erfcx(a/sqrt2)/2) - log1p(-Phi-bar(b)/Phi-bar(a)): no cancellation of
// e^2/2 against a^2/2, which matters because the far-tail pair is usually the parent's own.
__device__ inline double log_trunc_density(double e, double a, double b, double ea, double be) {
  if (b < 0.0) {  // mirror onto the positive side
    const double t = a;
    a = -b;
    b = -t;
    e = -e;
    const double s = ea;
    ea = be;
    be = s;
  }
  if (a > 0.0) {
    const double xa = erfcx(a * kRsqrt2);
    const double r = -0.5 * (ea + be) * (b + a) + log(erfcx(b * kRsqrt2) / xa);
    return -0.5 * ea * (e + a) - log(0.5 * xa) - log(-expm1(r));
  }
  return -0.5 * e * e - log(normcdf(b) - normcdf(a));
}

// a standard normal truncated to [a, b] with b < -kTail, by inverse CDF in log space: log Phi(e) = log Phi(b) +
// log(u + (1 - u) Phi(a) / Phi(b)), inverted by Newton on the concave log Phi from the asymptotic start (every step
// after the first approaches from below; 3 steps reach the f64 limit, 4 are taken)
__device__ inline double trunc_normal_lower_tail(double a, double b, double u) {
  const double la = log_phi(a), lb = log_phi(b);
  const double T = lb + log(u + (1.0 - u) * exp(la - lb));
  if (!(T > -INFINITY)) return T == -INFINITY ? a : b;  // (u = 0 with Phi(a) / Phi(b) below 2^-1074; NaN: |a|, |b| ~ 1e154)
  double y = sqrt(-2.0 * T);
  y = sqrt(fmax(-2.0 * T - 2.0 * log(y) - 1.8378770664093454836, 1.0));  // log(2 pi)
  double x = -y;
#pragma unroll
  for (int it = 0; it < 4; ++it) x -= (log_phi(x) - T) * erfcx(-x * kRsqrt2) * 1.2533141373155002512;  // sqrt(pi/2)
  return fmax(a, fmin(b, x));  // (a NaN gives b)
}

// e ~ N(0, 1) truncated to [a, b], from u in [0, 1).  The central case is smc_propose_kernel's operations exactly
// (its result may round to -inf when u (Phi(b) - Phi(a)) + Phi(a) rounds to 0; the caller clamps theta)
__device__ inline double trunc_normal(double a, double b, double u) {
  if (b < -kTail) return trunc_normal_lower_tail(a, b, u);
  if (a > kTail) return -trunc_normal_lower_tail(-b, -a, 1.0 - u);  // (Phi-bar(x) = Phi(-x); 1 - u is exact)
  const double fa = normcdf(a), fb = normcdf(b);
  return normcdfinv(__dadd_rn(fa, __dmul_rn(u, __dsub_rn(fb, fa))));
}

__global__ void smc_propose_cov_kernel(uint32_t seed_lo, uint32_t seed_hi, uint64_t idx_begin, uint32_t n,
                                       const float4* __restrict__ prev, const double* __restrict__ cum, uint32_t M,
                                       const double* __restrict__ cov, uint32_t per_parent, CovArgs cb,
                                       float4* __restrict__ out, uint32_t* __restrict__ parent_out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t idx = idx_begin + i;
  const uint4 x = philox4x32_10(kProposalDomain, 0u, (uint32_t)idx, (uint32_t)(idx >> 32), seed_lo, seed_hi);
  const uint4 y = philox4x32_10(kProposalDomain, 1u, (uint32_t)idx, (uint32_t)(idx >> 32), seed_lo, seed_hi);
  const double target = __dmul_rn(u53(x.x, x.y), cum[M - 1]);  // the parent exactly as smc_propose_kernel picks it
  uint32_t l = 0, h = M - 1;
  while (l < h) {
    const uint32_t mid = (l + h) >> 1;
    if (cum[mid] > target) h = mid;
    else l = mid + 1;
  }
  const float4 p = prev[l];
  float v[3] = {p.y, p.z, p.w};
  const double u[3] = {u53(x.z, x.w), u53(y.x, y.y), u53(y.z, y.w)};
  double L[6];
  if (per_parent) {
    if (!chol_free(cov + 6 * (size_t)l, cb, L)) return;  // (the host checked every Sigma)
  } else {
#pragma unroll
    for (int q = 0; q < 6; ++q) L[q] = cb.L[q];
  }
  double e[3] = {0.0, 0.0, 0.0};
#pragma unroll
  for (int t = 0; t < 3; ++t) {
    if (t >= cb.D) break;
    const int k = cb.f[t];
    double m = (double)v[k];
    for (int q = 0; q < t; ++q) m = __dadd_rn(m, __dmul_rn(L[tri(t, q)], e[q]));
    const double s = L[tri(t, t)];
    const double a = __ddiv_rn(__dsub_rn((double)cb.lo[t], m), s), b = __ddiv_rn(__dsub_rn((double)cb.hi[t], m), s);
    const double z = trunc_normal(a, b, u[k]);
    const float th = fminf(fmaxf((float)__dadd_rn(m, __dmul_rn(s, z)), cb.lo[t]), cb.hi[t]);
    v[k] = th;
    e[t] = __ddiv_rn(__dsub_rn((double)th, m), s);  // of the rounded theta: the density is evaluated there
  }
  out[i] = make_float4(p.x, v[0], v[1], v[2]);
  parent_out[i] = l;
}

__device__ __forceinline__ unsigned long long ordered_bits(double x) {  // monotone in x (for atomicMax)
  const unsigned long long b = (unsigned long long)__double_as_longlong(x);
  return (b >> 63) ? ~b : b | 0x8000000000000000ull;
}
__device__ __forceinline__ double from_ordered_bits(unsigned long long b) {
  return __longlong_as_double((long long)((b >> 63) ? b & 0x7FFFFFFFFFFFFFFFull : ~b));
}

// previous particle j: log2 W_j - sum_t log2 L_tt - log2(its first coordinate's mass), c_j and (per parent) L_j^-1;
// the largest log2 weight goes to *shift_bits (the pair kernel's terms are taken relative to it: max is exact, so the
// result does not depend on the order)
template <bool kShared>
__global__ void smc_tiles_cov_kernel(const float4* __restrict__ prev, const double* __restrict__ w, uint32_t M,
                                     const double* __restrict__ cov, CovArgs cb,
                                     typename std::conditional<kShared, CovRecShared, CovRec>::type* __restrict__ tiles,
                                     unsigned long long* __restrict__ shift_bits) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= M) return;
  const float4 p = prev[j];
  const float v[3] = {p.y, p.z, p.w};
  double L[6], Li[6];
  bool ok = true;
  if (kShared) {
#pragma unroll
    for (int q = 0; q < 6; ++q) { L[q] = cb.L[q]; Li[q] = cb.Li[q]; }
  } else {
    ok = chol_free(cov + 6 * (size_t)j, cb, L);
    tri_inverse(L, cb.D, Li);
  }
  typename std::conditional<kShared, CovRecShared, CovRec>::type r;
  double logw = log2(w[j]);
#pragma unroll
  for (int t = 0; t < 3; ++t) {
    r.c[t] = t < cb.D ? (double)v[cb.f[t]] : 0.0;
    if (t < cb.D) logw -= log2(L[tri(t, t)]);
  }
  if (cb.D > 0) {
    const double s = L[0], c = r.c[0];
    logw -= kLog2e * log_mass(((double)cb.lo[0] - c) / s, ((double)cb.hi[0] - c) / s);
  }
  r.logw = ok ? logw : NAN;
  if constexpr (!kShared) {
#pragma unroll
    for (int q = 0; q < 6; ++q) r.li[q] = Li[q];
  }
  tiles[j] = r;
  atomicMax(shift_bits, ordered_bits(r.logw));
}

// S_i = sum_j 2^(logw_j - shift) prod_t (the truncated factors of pair (i, j)), up to a factor common to every i: the
// whitening and the log density in f64, one ex2.approx.f32 per pair, every tile summed in f32 over four interleaved
// partial sums in a fixed order, the tiles in f64 (as smc_pair_kernel)
template <bool kShared>
__global__ void __launch_bounds__(kPairBlock) smc_pair_cov_kernel(
    const float4* __restrict__ cand, uint32_t N,
    const typename std::conditional<kShared, CovRecShared, CovRec>::type* __restrict__ tiles, uint32_t M, CovArgs cb,
    const unsigned long long* __restrict__ shift_bits, double* __restrict__ sum_out) {
  using Rec = typename std::conditional<kShared, CovRecShared, CovRec>::type;
  __shared__ Rec sh[kPairBlock];
  const uint32_t i = blockIdx.x * kPairBlock + threadIdx.x;
  const float4 xi = i < N ? cand[i] : make_float4(0.f, 0.f, 0.f, 0.f);
  const float vi[3] = {xi.y, xi.z, xi.w};
  const double shift = from_ordered_bits(*shift_bits);
  double x[3], ea[3], be[3];  // the candidate in free order and its edge distances in units of L_tt (shared Sigma)
#pragma unroll
  for (int t = 0; t < 3; ++t) {
    const int k = t < cb.D ? cb.f[t] : 0;
    x[t] = (double)vi[k];
    ea[t] = x[t] - (double)cb.lo[t];
    be[t] = (double)cb.hi[t] - x[t];
  }
  double total = 0.0;
  for (uint32_t base = 0; base < M; base += kPairBlock) {
    __syncthreads();
    const uint32_t j = base + threadIdx.x;
    if (j < M) {
      sh[threadIdx.x] = tiles[j];
    } else {
      Rec z{};
      z.logw = -INFINITY;  // (a term 2^-inf = 0: adds nothing)
      sh[threadIdx.x] = z;
    }
    __syncthreads();
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
    for (int jj = 0; jj < kPairBlock; ++jj) {
      const Rec& r = sh[jj];
      const double* li = kShared ? cb.Li : reinterpret_cast<const CovRec&>(r).li;
      double d[3], lg = 0.0;
#pragma unroll
      for (int t = 0; t < 3; ++t) {
        if (t >= cb.D) break;
        d[t] = x[t] - r.c[t];
        double e = 0.0;
#pragma unroll
        for (int q = 0; q <= t; ++q) e += li[tri(t, q)] * d[q];
        if (t == 0) {
          lg -= 0.5 * e * e;  // (the first coordinate's mass is in logw)
        } else {
          const double l = li[tri(t, t)], p = ea[t] * l, q = be[t] * l;
          lg += log_trunc_density(e, e - p, e + q, p, q);
        }
      }
      const float arg = (float)(r.logw - shift + kLog2e * lg);
      float pw;
      asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(pw) : "f"(arg));
      // (W_j = 0 or a padding slot adds nothing, whatever its factors: a padding slot's L^-1 is 0, its factor +inf)
      acc[jj & 3] = __fadd_rn(acc[jj & 3], r.logw == -INFINITY ? 0.f : pw);
    }
    total = __dadd_rn(total, (double)__fadd_rn(__fadd_rn(acc[0], acc[1]), __fadd_rn(acc[2], acc[3])));
  }
  if (i < N) sum_out[i] = total;
}

bool range_ok(const float* r) { return r && std::isfinite(r[0]) && std::isfinite(r[1]) && r[0] >= 0.f && r[0] <= r[1]; }

// The free parameters of cov [n_cov][6] (lo < hi and Sigma_kk > 0 in every Sigma; lo < hi with Sigma_kk = 0 in every
// Sigma fixes k), every Sigma positive definite over them, and a shared Sigma's L and L^-1.  min_pivot (optional)
// receives the smallest L_tt / (hi_t - lo_t) over every Sigma.
int make_cov_args(const double* cov, uint32_t n_cov, uint32_t M, const float* r1, const float* r2, const float* r3,
                  CovArgs* cb, double* min_pivot, std::string* err) {
  if (!cov || (n_cov != 1 && n_cov != M)) { *err = "cov must hold 1 or M packed Sigma"; return ECDNA_B200_ERR_BAD_PARAMS; }
  if (!range_ok(r1) || !range_ok(r2) || !range_ok(r3)) { *err = "every prior range needs 0 <= lo <= hi (finite)"; return ECDNA_B200_ERR_BAD_PARAMS; }
  const float* r[3] = {r1, r2, r3};
  std::memset(cb, 0, sizeof *cb);
  for (int k = 0; k < 3; ++k) {
    if (!(r[k][0] < r[k][1])) continue;
    uint64_t pos = 0;
    for (uint32_t s = 0; s < n_cov; ++s) {
      const double* S = cov + 6 * (size_t)s;
      for (int l = 0; l < 3; ++l)
        if (r[l][0] < r[l][1] && !std::isfinite(S[k >= l ? tri(k, l) : tri(l, k)])) {
          *err = "Sigma " + std::to_string(s) + " has a non-finite entry";
          return ECDNA_B200_ERR_BAD_PARAMS;
        }
      const double skk = S[tri(k, k)];
      if (skk < 0.0) { *err = "Sigma " + std::to_string(s) + " has a negative variance"; return ECDNA_B200_ERR_BAD_PARAMS; }
      pos += skk > 0.0;
    }
    if (pos != 0 && pos != n_cov) {
      *err = "parameter " + std::to_string(k + 1) + " has variance 0 in some Sigma and not in others";
      return ECDNA_B200_ERR_BAD_PARAMS;
    }
    if (pos == 0) continue;
    cb->lo[cb->D] = r[k][0];
    cb->hi[cb->D] = r[k][1];
    cb->f[cb->D++] = k;
  }
  double worst = INFINITY;
  for (uint32_t s = 0; s < n_cov; ++s) {
    double L[6];
    if (!chol_free(cov + 6 * (size_t)s, *cb, L)) {
      *err = "Sigma " + std::to_string(s) + " is not positive definite over the free parameters";
      return ECDNA_B200_ERR_BAD_PARAMS;
    }
    for (int t = 0; t < cb->D; ++t) worst = std::min(worst, L[tri(t, t)] / ((double)cb->hi[t] - (double)cb->lo[t]));
    if (n_cov == 1) {
      std::memcpy(cb->L, L, sizeof L);
      tri_inverse(L, cb->D, cb->Li);
    }
  }
  if (min_pivot) *min_pivot = worst;
  return ECDNA_B200_OK;
}

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

// the sums S_i of a pair kernel -> weights 1 / S_i normalised to sum 1 (f64, in index order)
int normalise_weights(ecdna_b200_ctx* ctx, double* w, uint32_t N) {
  double total = 0.0;
  for (uint32_t i = 0; i < N; ++i) {
    if (!(w[i] > 0.0) || !std::isfinite(w[i]))
      return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "particle " + std::to_string(i) + " has proposal density 0 under the previous population");
    w[i] = 1.0 / w[i];
    total += w[i];
  }
  for (uint32_t i = 0; i < N; ++i) w[i] /= total;
  return ECDNA_B200_OK;
}

double ms_since(std::chrono::steady_clock::time_point t0) {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
}

// Sigma = 2 x the weighted covariance of the population (the diagonal with smc_sigma's sums: sqrt(Sigma_kk) is the
// component kernel's sigma_k bit for bit); sums sequential in index order in f64
std::vector<double> mvn_sigma(const float* rates, const double* w, uint32_t M) {
  double mean[3];
  for (int k = 0; k < 3; ++k) {
    mean[k] = 0.0;
    for (uint32_t i = 0; i < M; ++i) mean[k] += w[i] * (double)rates[4 * (size_t)i + 1 + k];
  }
  std::vector<double> S(6);
  for (int k = 0; k < 3; ++k)
    for (int l = 0; l <= k; ++l) {
      double v = 0.0;
      for (uint32_t i = 0; i < M; ++i) {
        const double dk = (double)rates[4 * (size_t)i + 1 + k] - mean[k], dl = (double)rates[4 * (size_t)i + 1 + l] - mean[l];
        v += k == l ? w[i] * dk * dk : w[i] * dk * dl;
      }
      S[tri(k, l)] = 2.0 * v;
    }
  return S;
}

// OLCM (Filippi, Barnes, Cornebise, Stumpf 2013): Sigma_j = C + (m - theta_j)(m - theta_j)^T with m and C the
// weighted mean and covariance of the particles with rho <= eps, their weights renormalised; sums sequential in f64
std::vector<double> olcm_sigma(const float* rates, const double* w, const float* rho, uint32_t M, float eps) {
  double sw = 0.0;
  for (uint32_t i = 0; i < M; ++i)
    if (rho[i] <= eps) sw += w[i];
  double m[3], C[6];
  for (int k = 0; k < 3; ++k) {
    m[k] = 0.0;
    for (uint32_t i = 0; i < M; ++i)
      if (rho[i] <= eps) m[k] += w[i] / sw * (double)rates[4 * (size_t)i + 1 + k];
  }
  for (int k = 0; k < 3; ++k)
    for (int l = 0; l <= k; ++l) {
      double v = 0.0;
      for (uint32_t i = 0; i < M; ++i) {
        if (!(rho[i] <= eps)) continue;
        const double dk = (double)rates[4 * (size_t)i + 1 + k] - m[k], dl = (double)rates[4 * (size_t)i + 1 + l] - m[l];
        v += w[i] / sw * dk * dl;
      }
      C[tri(k, l)] = v;
    }
  std::vector<double> S((size_t)M * 6);
  for (uint32_t j = 0; j < M; ++j)
    for (int k = 0; k < 3; ++k)
      for (int l = 0; l <= k; ++l)
        S[6 * (size_t)j + tri(k, l)] = C[tri(k, l)] + (m[k] - (double)rates[4 * (size_t)j + 1 + k]) *
                                                          (m[l] - (double)rates[4 * (size_t)j + 1 + l]);
  return S;
}

// a Sigma the proposal can use: valid for ecdna_b200_abc_smc_*_cov and every Cholesky pivot L_tt >= 2^-12 (hi - lo)
// (rates are f32: a narrower conditional kernel is below their resolution over the box)
bool cov_usable(const std::vector<double>& cov, uint32_t M, const ecdna_b200_smc_options_t* o) {
  CovArgs cb;
  std::string err;
  double pivot = 0.0;
  return make_cov_args(cov.data(), (uint32_t)(cov.size() / 6), M, o->b1_range, o->d0_range, o->d1_range, &cb, &pivot,
                       &err) == ECDNA_B200_OK &&
         pivot >= 0x1p-12;
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
  return normalise_weights(ctx, weights_out, N);
}

int ecdna_b200_abc_smc_propose_cov(ecdna_b200_ctx* ctx, uint64_t seed, uint64_t idx_begin, uint64_t n,
                                   const float* prev_rates, const double* cum_weights, uint32_t M, const double* cov,
                                   uint32_t n_cov, const float b1_range[2], const float d0_range[2],
                                   const float d1_range[2], float* rates_out, uint32_t* parent_out) {
  if (!ctx) return ECDNA_B200_ERR_BAD_PARAMS;
  if (!prev_rates || !cum_weights || !rates_out || !parent_out || M == 0 || n == 0 || n >= (1ull << 32))
    return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "bad proposal request (buffers, M >= 1, n in [1, 2^32))");
  if (!(cum_weights[M - 1] > 0.0) || !std::isfinite(cum_weights[M - 1]))
    return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "the cumulative weights must end with a finite value > 0");
  CovArgs cb;
  std::string err;
  if (make_cov_args(cov, n_cov, M, b1_range, d0_range, d1_range, &cb, nullptr, &err)) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, err);
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  CU(ctx->smc_prev.ensure((size_t)M * 16));
  CU(ctx->smc_cum.ensure((size_t)M * 8));
  CU(ctx->smc_cov.ensure((size_t)n_cov * 48));
  CU(ctx->smc_new.ensure((size_t)n * 16));
  CU(ctx->smc_parent.ensure((size_t)n * 4));
  CU(cudaMemcpyAsync(ctx->smc_prev.p, prev_rates, (size_t)M * 16, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(ctx->smc_cum.p, cum_weights, (size_t)M * 8, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(ctx->smc_cov.p, cov, (size_t)n_cov * 48, cudaMemcpyHostToDevice, st));
  smc_propose_cov_kernel<<<(uint32_t)((n + 255) / 256), 256, 0, st>>>(
      (uint32_t)seed, (uint32_t)(seed >> 32), idx_begin, (uint32_t)n, (const float4*)ctx->smc_prev.p,
      (const double*)ctx->smc_cum.p, M, (const double*)ctx->smc_cov.p, n_cov > 1 ? 1u : 0u, cb, (float4*)ctx->smc_new.p,
      (uint32_t*)ctx->smc_parent.p);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(rates_out, ctx->smc_new.p, (size_t)n * 16, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(parent_out, ctx->smc_parent.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return ECDNA_B200_OK;
}

int ecdna_b200_abc_smc_weights_cov(ecdna_b200_ctx* ctx, const float* new_rates, uint32_t N, const float* prev_rates,
                                   const double* prev_weights, uint32_t M, const double* cov, uint32_t n_cov,
                                   const float b1_range[2], const float d0_range[2], const float d1_range[2],
                                   double* weights_out) {
  if (!ctx) return ECDNA_B200_ERR_BAD_PARAMS;
  if (!new_rates || !prev_rates || !prev_weights || !weights_out || N == 0 || M == 0)
    return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, "bad weight request (buffers, N >= 1, M >= 1)");
  CovArgs cb;
  std::string err;
  if (make_cov_args(cov, n_cov, M, b1_range, d0_range, d1_range, &cb, nullptr, &err)) return fail(ctx, ECDNA_B200_ERR_BAD_PARAMS, err);
  const bool shared = n_cov == 1 && M > 1;  // (M = 1: one Sigma either way)
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  CU(ctx->smc_prev.ensure((size_t)M * 16));
  CU(ctx->smc_cum.ensure((size_t)M * 8));
  CU(ctx->smc_cov.ensure((size_t)n_cov * 48 + 8));
  CU(ctx->smc_tiles.ensure((size_t)M * (shared ? sizeof(CovRecShared) : sizeof(CovRec))));
  CU(ctx->smc_new.ensure((size_t)N * 16));
  CU(ctx->smc_sum.ensure((size_t)N * 8));
  CU(cudaMemcpyAsync(ctx->smc_prev.p, prev_rates, (size_t)M * 16, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(ctx->smc_cum.p, prev_weights, (size_t)M * 8, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(ctx->smc_cov.p, cov, (size_t)n_cov * 48, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(ctx->smc_new.p, new_rates, (size_t)N * 16, cudaMemcpyHostToDevice, st));
  unsigned long long* shift = (unsigned long long*)((char*)ctx->smc_cov.p + (size_t)n_cov * 48);
  CU(cudaMemsetAsync(shift, 0, 8, st));
  const uint32_t tgrid = (uint32_t)(((uint64_t)M + 255) / 256), pgrid = (uint32_t)(((uint64_t)N + kPairBlock - 1) / kPairBlock);
  const double* dcov = (const double*)ctx->smc_cov.p;
  if (shared) {
    smc_tiles_cov_kernel<true><<<tgrid, 256, 0, st>>>((const float4*)ctx->smc_prev.p, (const double*)ctx->smc_cum.p, M,
                                                      dcov, cb, (CovRecShared*)ctx->smc_tiles.p, shift);
    smc_pair_cov_kernel<true><<<pgrid, kPairBlock, 0, st>>>((const float4*)ctx->smc_new.p, N,
                                                             (const CovRecShared*)ctx->smc_tiles.p, M, cb, shift,
                                                             (double*)ctx->smc_sum.p);
  } else {
    smc_tiles_cov_kernel<false><<<tgrid, 256, 0, st>>>((const float4*)ctx->smc_prev.p, (const double*)ctx->smc_cum.p, M,
                                                       dcov, cb, (CovRec*)ctx->smc_tiles.p, shift);
    smc_pair_cov_kernel<false><<<pgrid, kPairBlock, 0, st>>>((const float4*)ctx->smc_new.p, N,
                                                              (const CovRec*)ctx->smc_tiles.p, M, cb, shift,
                                                              (double*)ctx->smc_sum.p);
  }
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(weights_out, ctx->smc_sum.p, (size_t)N * 8, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return normalise_weights(ctx, weights_out, N);
}

int ecdna_b200_abc_smc(ecdna_b200_multi* m, const ecdna_b200_params_t* params, const ecdna_b200_smc_options_t* o,
                       ecdna_b200_smc_result_t* r) {
  return ecdna_b200_abc_smc_ex(m, params, o, nullptr, r, nullptr);
}

int ecdna_b200_abc_smc_ex(ecdna_b200_multi* m, const ecdna_b200_params_t* params, const ecdna_b200_smc_options_t* o,
                          const ecdna_b200_smc_kernel_t* kernel, ecdna_b200_smc_result_t* r, uint32_t* kernel_used) {
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
  const uint32_t want = kernel ? kernel->kernel : (uint32_t)ECDNA_B200_SMC_KERNEL_COMPONENT;
  if (want > ECDNA_B200_SMC_KERNEL_OLCM) return bad("kernel must be one of ECDNA_B200_SMC_KERNEL_*");
  if (kernel && (kernel->reserved[0] || kernel->reserved[1] || kernel->reserved[2])) return bad("kernel.reserved must be 0");

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
  std::vector<double> cov;  // the Sigma of the correlated kernels: 6 (mvn) or 6 M (olcm) packed lower triangles
  uint32_t used_kernel = ECDNA_B200_SMC_KERNEL_COMPONENT;
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
      int rc = g == 0
             ? ecdna_b200_abc_draw_priors(ctx0, params->seed, pos, n, params->b0, o->b1_range, o->d0_range, o->d1_range, rates.data())
             : used_kernel == ECDNA_B200_SMC_KERNEL_COMPONENT
                 ? ecdna_b200_abc_smc_propose(ctx0, params->seed, pos, n, prev.rates.data(), cum.data(), M, sigma,
                                              o->b1_range, o->d0_range, o->d1_range, rates.data(), parent.data())
                 : ecdna_b200_abc_smc_propose_cov(ctx0, params->seed, pos, n, prev.rates.data(), cum.data(), M,
                                                  cov.data(), (uint32_t)(cov.size() / 6), o->b1_range, o->d0_range,
                                                  o->d1_range, rates.data(), parent.data());
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
      const int rc = used_kernel == ECDNA_B200_SMC_KERNEL_COMPONENT
                         ? ecdna_b200_abc_smc_weights(ctx0, cur.rates.data(), M, prev.rates.data(), prev.w.data(), M,
                                                      sigma, o->b1_range, o->d0_range, o->d1_range, cur.w.data())
                         : ecdna_b200_abc_smc_weights_cov(ctx0, cur.rates.data(), M, prev.rates.data(), prev.w.data(),
                                                          M, cov.data(), (uint32_t)(cov.size() / 6), o->b1_range,
                                                          o->d0_range, o->d1_range, cur.w.data());
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
    if (kernel_used) kernel_used[g] = g == 0 ? UINT32_MAX : used_kernel;
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
    // the correlated kernels' Sigma, falling back olcm -> mvn -> component until one is usable
    used_kernel = ECDNA_B200_SMC_KERNEL_COMPONENT;
    if (want == ECDNA_B200_SMC_KERNEL_OLCM) {
      cov = olcm_sigma(cur.rates.data(), cur.w.data(), cur.rho.data(), M, eps);
      if (cov_usable(cov, M, o)) used_kernel = ECDNA_B200_SMC_KERNEL_OLCM;
    }
    if (want != ECDNA_B200_SMC_KERNEL_COMPONENT && used_kernel == ECDNA_B200_SMC_KERNEL_COMPONENT) {
      cov = mvn_sigma(cur.rates.data(), cur.w.data(), M);
      if (cov_usable(cov, M, o)) used_kernel = ECDNA_B200_SMC_KERNEL_MVN;
    }
    std::swap(prev, cur);
  }
  return ECDNA_B200_OK;
}

}  // extern "C"

// ecdna_oracle.cpp -- CPU ORACLE for the ecDNA SSA hot path.  TEST INFRASTRUCTURE ONLY; see
// ecdna_oracle.h for the contract, the "parity unpinned" statement and the citation rules.
//
// Build: g++ -O3 -std=c++17 -ffp-contract=off -march=x86-64-v3 -shared -fPIC (oracle/Makefile).
// -ffp-contract=off matters: the philox-mode float arithmetic is specified operation by
// operation (explicit fmaf only) so that the CUDA kernel reproduces it bit for bit.
#include "ecdna_oracle.h"

#include <atomic>
#include <cmath>
#include <cstring>
#include <limits>
#include <thread>
#include <type_traits>
#include <vector>

namespace {

// ------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11).  Counter-based: the GPU's native stream.
// ------------------------------------------------------------------------------------------
inline void philox_round(uint32_t c[4], uint32_t k0, uint32_t k1) {
  const uint64_t p0 = (uint64_t)0xD2511F53u * c[0];
  const uint64_t p1 = (uint64_t)0xCD9E8D57u * c[2];
  const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0;
  const uint32_t n1 = (uint32_t)p1;
  const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
  const uint32_t n3 = (uint32_t)p0;
  c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
}
inline void philox(uint32_t c[4], uint32_t k0, uint32_t k1) {
  for (int r = 0; r < 10; ++r) {
    philox_round(c, k0, k1);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
}
struct PhiloxKey { uint32_t k0, k1, r0, r1; };
inline void philox_slot(const PhiloxKey& key, uint32_t event, uint32_t slot, uint32_t out[4]) {
  out[0] = event; out[1] = slot; out[2] = key.r0; out[3] = key.r1;
  philox(out, key.k0, key.k1);
}

// -ln((m+1) * 2^-24) for a 24-bit m, in f32 with a fixed operation order (cephes-style logf
// polynomial).  Every operation is a single IEEE f32 op or an explicit fmaf.
inline float neg_log_u24(uint32_t m) {
  const float v = (float)(m + 1u);  // 1 .. 2^24, exact
  uint32_t bits; std::memcpy(&bits, &v, 4);
  int e = (int)(bits >> 23) - 127;
  uint32_t fb = (bits & 0x007FFFFFu) | 0x3F800000u;
  float f; std::memcpy(&f, &fb, 4);  // [1,2)
  if (f > 1.41421356f) { f = f * 0.5f; e += 1; }
  const float x = f - 1.0f;
  const float z = x * x;
  float y = 7.0376836292E-2f;
  y = fmaf(y, x, -1.1514610310E-1f);
  y = fmaf(y, x, 1.1676998740E-1f);
  y = fmaf(y, x, -1.2420140846E-1f);
  y = fmaf(y, x, 1.4249322787E-1f);
  y = fmaf(y, x, -1.6668057665E-1f);
  y = fmaf(y, x, 2.0000714765E-1f);
  y = fmaf(y, x, -2.4999993993E-1f);
  y = fmaf(y, x, 3.3333331174E-1f);
  y = y * x;
  y = y * z;
  y = fmaf(-0.5f, z, y);
  const float lf = x + y;  // ln(f)
  const float ne = (float)(24 - e);
  return fmaf(ne, 0.693359375f, fmaf(ne, -2.12194440e-4f, -lf));
}

inline uint64_t hist_weight(uint32_t k) {
  uint64_t z = (uint64_t)(k + 1u) * 0x9E3779B97F4A7C15ull;
  z ^= z >> 32;
  z *= 0xD6E8FEB86659FD93ull;
  z ^= z >> 29;
  return z;
}
inline uint64_t chain_step(uint64_t chain, uint64_t hash, uint64_t nminus, float time) {
  uint32_t tb; std::memcpy(&tb, &time, 4);
  uint64_t c = chain ^ (hash + nminus * 0x9E3779B97F4A7C15ull + (uint64_t)tb);
  c *= 0xD6E8FEB86659FD93ull;
  c ^= c >> 29;
  return c;
}

// ------------------------------------------------------------------------------------------
// rand_chacha 0.3.1 ChaCha8Rng + rand_core 0.6.4 seed_from_u64 + BlockRng [RECALL R7]
// ------------------------------------------------------------------------------------------
inline uint32_t rotl(uint32_t x, int n) { return (x << n) | (x >> (32 - n)); }
inline void qround(uint32_t* s, int a, int b, int c, int d) {
  s[a] += s[b]; s[d] = rotl(s[d] ^ s[a], 16);
  s[c] += s[d]; s[b] = rotl(s[b] ^ s[c], 12);
  s[a] += s[b]; s[d] = rotl(s[d] ^ s[a], 8);
  s[c] += s[d]; s[b] = rotl(s[b] ^ s[c], 7);
}
void chacha_block(const uint32_t key[8], uint64_t counter, uint64_t stream, int rounds, uint32_t out[16]) {
  uint32_t in[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u,
                     key[0], key[1], key[2], key[3], key[4], key[5], key[6], key[7],
                     (uint32_t)counter, (uint32_t)(counter >> 32), (uint32_t)stream, (uint32_t)(stream >> 32)};
  uint32_t s[16];
  std::memcpy(s, in, sizeof s);
  for (int r = 0; r < rounds; r += 2) {
    qround(s, 0, 4, 8, 12); qround(s, 1, 5, 9, 13); qround(s, 2, 6, 10, 14); qround(s, 3, 7, 11, 15);
    qround(s, 0, 5, 10, 15); qround(s, 1, 6, 11, 12); qround(s, 2, 7, 8, 13); qround(s, 3, 4, 9, 14);
  }
  for (int i = 0; i < 16; ++i) out[i] = s[i] + in[i];
}
void seed_from_u64(uint64_t state, uint32_t key[8]) {
  // rand_core::SeedableRng::seed_from_u64: PCG32 (XSH-RR) fills the 32-byte seed
  for (int i = 0; i < 8; ++i) {
    state = state * 6364136223846793005ull + 11634580027462260723ull;
    const uint32_t xs = (uint32_t)(((state >> 18) ^ state) >> 27);
    const uint32_t rot = (uint32_t)(state >> 59);
    key[i] = (xs >> rot) | (xs << ((32 - rot) & 31));
  }
}
struct ChaCha8 {
  uint32_t key[8];
  uint64_t counter = 0, stream = 0;
  uint32_t buf[64];
  int index = 64;  // 4 blocks buffered, refilled when exhausted
  uint64_t* rec = nullptr;  // optional export of every u64 handed out (what a recording RngCore sees)
  uint64_t rec_cap = 0, rec_len = 0;
  // optional EXTERNAL stream: the u64 log of a real reference run (INTEGRATION.md section 5) replaces the
  // generator, so that every conversion downstream of it is checked against the reference's own output
  const uint64_t* ext = nullptr;
  uint64_t ext_len = 0, ext_pos = 0;
  bool dry = false;
  ChaCha8(uint64_t seed, uint64_t stream_id) : stream(stream_id) { seed_from_u64(seed, key); }
  void refill() {
    for (int b = 0; b < 4; ++b) chacha_block(key, counter + b, stream, 8, buf + 16 * b);
    counter += 4;
  }
  uint64_t next_u64() {
    if (ext) {
      if (ext_pos >= ext_len) { dry = true; return 0; }  // (0 ends every rejection loop downstream)
      return ext[ext_pos++];
    }
    const uint64_t v = raw_u64();
    if (rec) {
      if (rec_len < rec_cap) rec[rec_len] = v;
      rec_len++;
    }
    return v;
  }
  uint64_t raw_u64() {
    if (index < 63) {
      const uint64_t v = ((uint64_t)buf[index + 1] << 32) | buf[index];
      index += 2;
      return v;
    }
    if (index >= 64) {
      refill();
      index = 2;
      return ((uint64_t)buf[1] << 32) | buf[0];
    }
    const uint32_t lo = buf[63];
    refill();
    index = 1;
    return ((uint64_t)buf[0] << 32) | lo;
  }
  // rand 0.8.5 Standard f64: 53 random bits scaled by 2^-53
  double gen_f64() { return (double)(next_u64() >> 11) * (1.0 / 9007199254740992.0); }
  // rand 0.8.5 UniformInt<usize>::sample_single: widening multiply, conservative zone [RECALL R5]
  uint64_t gen_range(uint64_t n) {
    const uint64_t zone = (n << __builtin_clzll(n)) - 1;
    for (;;) {
      const uint64_t v = next_u64();
      const unsigned __int128 m = (unsigned __int128)v * n;
      if ((uint64_t)m <= zone) return (uint64_t)(m >> 64);
    }
  }
  // rand 0.8.5 UniformFloat<f64>::sample: 52 mantissa bits -> [1,2) - 1, then * scale + low
  double uniform(double low, double scale) {
    const uint64_t b = (next_u64() >> 12) | 0x3FF0000000000000ull;
    double v12; std::memcpy(&v12, &b, 8);
    return (v12 - 1.0) * scale + low;
  }
};

// rand_distr 0.4.3 Exp1: 256-layer ziggurat (Marsaglia & Tsang 2000), tables REGENERATED from the
// published recurrence (the crate ships them as constants that are not available here) [RECALL R2]
struct ZigExp {
  double x[257], f[257];
  static constexpr double R = 7.69711747013104972;
  ZigExp() {
    const double v = 3.949659822581572e-3;
    x[0] = v / std::exp(-R);
    x[1] = R;
    for (int i = 2; i < 256; ++i) x[i] = -std::log(v / x[i - 1] + std::exp(-x[i - 1]));
    x[256] = 0.0;
    for (int i = 0; i < 257; ++i) f[i] = std::exp(-x[i]);
  }
};
const ZigExp& zig() { static const ZigExp z; return z; }
inline double exp1_f64(ChaCha8& g) {
  const ZigExp& z = zig();
  for (;;) {
    const uint64_t bits = g.next_u64();
    const int i = (int)(bits & 0xff);
    const uint64_t mb = (bits >> 12) | 0x3FF0000000000000ull;
    double u12; std::memcpy(&u12, &mb, 8);
    const double u = u12 - (1.0 - std::numeric_limits<double>::epsilon() / 2.0);
    const double xx = u * z.x[i];
    if (xx < z.x[i + 1]) return xx;
    if (i == 0) return ZigExp::R - std::log(g.gen_f64());
    if (z.f[i + 1] + (z.f[i] - z.f[i + 1]) * g.gen_f64() < std::exp(-xx)) return xx;
  }
}

// rand_distr 0.4.3 Binomial::sample: BINV below n*min(p,1-p) < 10, BTPE (Kachitvichyanukul &
// Schmeiser 1988, with the GSL sign convention for the Stirling terms) otherwise [RECALL R6]
inline double stirling_corr(double a) {
  const double a2 = a * a;
  return (13860. - (462. - (132. - (99. - 140. / a2) / a2) / a2) / a2) / a / 166320.;
}
uint64_t rand_binomial(ChaCha8& g, uint64_t n_int, double p_in) {
  if (p_in == 0.0) return 0;
  if (p_in == 1.0) return n_int;
  const double p = p_in <= 0.5 ? p_in : 1.0 - p_in;
  const double q = 1.0 - p;
  const double n = (double)n_int;
  int64_t res;
  if (n * p < 10.0 && n_int <= 0x7fffffffull) {
    const double s = p / q;
    const double a = (double)(n_int + 1) * s;
    double r = std::pow(q, (double)(int)n_int);  // powi
    double u = g.gen_f64();
    int64_t xv = 0;
    while (u > r) {
      u -= r;
      xv += 1;
      r *= a / (double)xv - s;
    }
    res = xv;
  } else {
    const double np = n * p, npq = np * q, fm = np + p;
    const int64_t m = (int64_t)fm;
    const double p1 = std::floor(2.195 * std::sqrt(npq) - 4.6 * q) + 0.5;
    const double xm = (double)m + 0.5, xl = xm - p1, xr = xm + p1;
    const double c = 0.134 + 20.5 / (15.3 + (double)m);
    const double p2 = p1 * (1.0 + 2.0 * c);
    auto lam = [](double a) { return a * (1.0 + 0.5 * a); };
    const double ll = lam((fm - xl) / (fm - xl * p));
    const double lr = lam((xr - fm) / (xr * q));
    const double p3 = p2 + c / ll;
    const double p4 = p3 + c / lr;
    int64_t y;
    for (;;) {
      const double u = g.uniform(0.0, p4);
      double v = g.uniform(0.0, 1.0);
      if (!(u > p1)) { y = (int64_t)(xm - p1 * v + u); break; }
      if (!(u > p2)) {
        const double xx = xl + (u - p1) / c;
        v = v * c + 1.0 - std::fabs(xx - xm) / p1;
        if (v > 1.0) continue;
        y = (int64_t)xx;
      } else if (!(u > p3)) {
        y = (int64_t)(xl + std::log(v) / ll);
        if (y < 0) continue;
        v *= (u - p2) * ll;
      } else {
        y = (int64_t)(xr - std::log(v) / lr);
        if (y > 0 && (uint64_t)y > n_int) continue;
        v *= (u - p3) * lr;
      }
      const int64_t kk = y > m ? y - m : m - y;
      if (!(kk > 20 && (double)kk < 0.5 * npq - 1.0)) {
        const double s = p / q, a = s * (n + 1.0);
        double ff = 1.0;
        if (m < y) { for (int64_t i = m + 1; i <= y; ++i) ff *= a / (double)i - s; }
        else if (m > y) { for (int64_t i = y + 1; i <= m; ++i) ff /= a / (double)i - s; }
        if (v > ff) continue;
        break;
      }
      const double kd = (double)kk;
      const double rho = (kd / npq) * ((kd * (kd / 3.0 + 0.625) + 1.0 / 6.0) / npq + 0.5);
      const double t = -0.5 * kd * kd / npq;
      const double alpha = std::log(v);
      if (alpha < t - rho) break;
      if (alpha > t + rho) continue;
      const double x1 = (double)(y + 1), f1 = (double)(m + 1);
      const double zz = (double)((int64_t)n + 1 - m), w = (double)((int64_t)n - y + 1);
      const double bound = xm * std::log(f1 / x1) + (n - (double)m + 0.5) * std::log(zz / w) +
                           (double)(y - m) * std::log(w * p / (x1 * q)) + stirling_corr(f1) +
                           stirling_corr(zz) - stirling_corr(x1) - stirling_corr(w);
      if (alpha > bound) continue;
      break;
    }
    res = y;
  }
  return p != p_in ? n_int - (uint64_t)res : (uint64_t)res;
}

// ------------------------------------------------------------------------------------------
// random sources behind one interface
// ------------------------------------------------------------------------------------------
constexpr float F_INF = std::numeric_limits<float>::infinity();

// sosa's exprand [RECALL R2]: a normal rate draws Exp(rate); an infinite rate gives 0; anything else
// (zero, subnormal, NaN) gives +inf WITHOUT consuming randomness.
struct RandSource {  // rng 0
  static constexpr bool kDirect = false;
  ChaCha8 g;
  RandSource(uint64_t seed, uint64_t run) : g(seed, run) {}
  bool dry() const { return g.dry; }
  void begin_event(uint32_t) {}
  float wait(int, float lambda) {
    if (std::isnormal(lambda)) return (float)exp1_f64(g) * (1.0f / lambda);
    return std::isinf(lambda) ? 0.0f : F_INF;
  }
  uint64_t pick(uint64_t n) { return g.gen_range(n); }
  uint64_t binomial_half(uint64_t n, uint32_t) { return rand_binomial(g, n, 0.5); }
};

struct PhiloxSource {  // rng 1: every draw is a pure function of (seed, run, event, slot)
  // NATIVE STREAM v2 (the specification of the CUDA kernel's native mode):
  //   slot 0            word 0 -> the exponential waiting time of the NEXT event (Gillespie's direct
  //                     method: dt ~ Exp(sum of propensities)); word 1 -> which reaction fires;
  //                     words 2,3 -> high / low half of the 64-bit uniform of the cell pick
  //   slot a*1024+1+i   all four words: bits 128i..128i+127 of segregation attempt a
  //   slot 2^31 + j     words 0,1: the j-th redraw of the cell pick (Lemire rejection)
  // Statistically the same process as sosa's first-reaction scheme (SURVEY 8a a2): total rate L = sum
  // of the lambda_i, dt ~ Exp(L), reaction i with probability lambda_i / L.
  static constexpr bool kDirect = true;
  bool dry() const { return false; }
  PhiloxKey key;
  uint32_t ev = 0;
  PhiloxSource(uint64_t seed, uint64_t run)
      : key{(uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)run, (uint32_t)(run >> 32)} {}
  void begin_event(uint32_t e) { ev = e; }
  float wait(int, float) { return F_INF; }  // (first-reaction interface: unused by this source)
  // One event of the direct method.  Propensities that are not normal numbers do not fire (sosa's
  // exprand gives them an infinite waiting time), +inf fires at once.  Every operation is a single
  // IEEE f32 operation in a fixed order: the kernel performs the same sequence.
  bool next_reaction(const float lam[4], uint32_t* event, float* dt) {
    float c[4], run = 0.f;
    for (int i = 0; i < 4; ++i) {
      const float lz = (std::isnormal(lam[i]) && lam[i] > 0.f) ? lam[i] : ((std::isinf(lam[i]) && lam[i] > 0.f) ? F_INF : 0.f);
      run = i == 0 ? lz : run + lz;
      c[i] = run;
    }
    if (!(c[3] > 0.f)) return false;  // absorbing: nothing can happen
    uint32_t x[4];
    philox_slot(key, ev, 0u, x);
    const float e = neg_log_u24(x[0] >> 8);
    const float ur = (float)(x[1] >> 8) * 5.9604644775390625e-08f;  // 24 bits * 2^-24, exact
    const bool inf = std::isinf(c[3]);
    *dt = inf ? 0.f : e / c[3];
    const float v = inf ? std::numeric_limits<float>::max() : ur * c[3];
    // the number of cumulative sums <= v: v < c[3] always (ur <= 1 - 2^-24), and a reaction whose
    // propensity is zero has the same cumulative sum as its predecessor, so it is never chosen
    *event = (uint32_t)(v >= c[0]) + (uint32_t)(v >= c[1]) + (uint32_t)(v >= c[2]);
    return true;
  }
  // Lemire's unbiased bounded integer from a 64-bit uniform
  uint64_t pick(uint64_t n) {
    for (uint32_t j = 0;; ++j) {
      uint32_t a[4];
      philox_slot(key, ev, j == 0 ? 0u : (0x80000000u + j), a);
      const uint64_t x = j == 0 ? (((uint64_t)a[2] << 32) | a[3]) : (((uint64_t)a[0] << 32) | a[1]);
      const unsigned __int128 m = (unsigned __int128)x * n;
      const uint64_t lo = (uint64_t)m;
      if (lo >= n || j >= 13) return (uint64_t)(m >> 64);
      const uint64_t t = (0 - n) % n;
      if (lo >= t) return (uint64_t)(m >> 64);
    }
  }
  // Binomial(n, 1/2) = popcount of n independent fair bits: bit b lives in slot
  // attempt*1024 + 1 + b/128, word (b%128)/32, bit b%32.  Exact, integer only.
  uint64_t binomial_half(uint64_t n, uint32_t attempt) {
    uint64_t count = 0;
    uint32_t slot = attempt * 1024u + 1u;
    for (uint64_t left = n; left > 0; ++slot) {
      uint32_t x[4];
      philox_slot(key, ev, slot, x);
      for (int w = 0; w <= 3 && left > 0; ++w) {
        const uint32_t take = left >= 32 ? 32u : (uint32_t)left;
        const uint32_t mask = take == 32 ? 0xFFFFFFFFu : ((1u << take) - 1u);
        count += (uint64_t)__builtin_popcount(x[w] & mask);
        left -= take;
      }
    }
    return count;
  }
};

// ------------------------------------------------------------------------------------------
// state layouts
// ------------------------------------------------------------------------------------------
struct VectorState {  // ecdna-lib 3.0.2 EcDNADistribution [RECALL R4], memory.md:5-8
  uint64_t nminus = 0;
  std::vector<uint16_t> cells;
  uint64_t nplus() const { return cells.size(); }
  // pick_remove_random_nplus: uniform index + swap_remove (proliferation.rs:57)
  uint32_t remove_at(uint64_t idx) {
    const uint16_t k = cells[idx];
    cells[idx] = cells.back();
    cells.pop_back();
    return k;
  }
  void push(uint32_t k) { cells.push_back((uint16_t)k); }
};

struct HistState {  // the GPU layout: h[k] = number of cells carrying k copies, k >= 1
  uint64_t nminus = 0, np = 0;
  uint32_t kmax = 0;
  std::vector<uint32_t> h;
  explicit HistState(uint32_t cap) : h(cap, 0) {}
  uint64_t nplus() const { return np; }
  // canonical enumeration of the cells: residue (k mod 32) major, then k ascending
  uint32_t class_at(uint64_t r) const {
    for (uint32_t res = 0; res < 32; ++res)
      for (uint32_t k = res; k <= kmax; k += 32) {
        if (r < h[k]) return k;
        r -= h[k];
      }
    return 0;  // unreachable when r < nplus
  }
};

struct Recorder {
  const orc_opts* o;
  orc_out* out;
  uint32_t snap_front = 0;
  uint32_t dyn_next = 0;
};

template <class HistFn>
void dense_hist(uint64_t* dst, uint32_t cap, uint64_t nminus, HistFn&& each) {
  std::memset(dst, 0, sizeof(uint64_t) * cap);
  if (cap) dst[0] = nminus;
  each([&](uint32_t k, uint64_t c) { if (k < cap) dst[k] += c; });
}

// One term of the entropy, -p log2(p) for p = c / n, 0 < c <= n < 2^32, as a 2^-40 fixed-point integer: single
// IEEE f32 operations in a fixed order (the polynomial of neg_log_u24 on the mantissa of p = f32(c) / f32(n)), so
// that the sum - an integer - does not depend on the order of the terms.  A class that holds at least 3/4 of the
// cells gives the polynomial x = p - 1 = -f32(n - c) / f32(n) directly, which keeps 1 - p when it is small.  The
// kernel's epilogue computes the same bits.
inline uint64_t entropy_term_q40(uint64_t c, uint64_t n) {
  const float nf = (float)n;
  const bool near1 = 4 * c >= 3 * n;
  const float q = (float)(near1 ? n - c : c) / nf;  // 1 - p or p
  const float p = near1 ? 1.0f - q : q;
  uint32_t bits; std::memcpy(&bits, &p, 4);
  int e = (int)(bits >> 23) - 127;
  uint32_t fb = (bits & 0x007FFFFFu) | 0x3F800000u;
  float f; std::memcpy(&f, &fb, 4);
  if (f > 1.41421356f) { f = f * 0.5f; e += 1; }
  const float x = near1 ? -q : f - 1.0f;  // (p in [3/4, 1]: its mantissa reduces to p itself, e = 0)
  const float z = x * x;
  float y = 7.0376836292E-2f;
  y = fmaf(y, x, -1.1514610310E-1f);
  y = fmaf(y, x, 1.1676998740E-1f);
  y = fmaf(y, x, -1.2420140846E-1f);
  y = fmaf(y, x, 1.4249322787E-1f);
  y = fmaf(y, x, -1.6668057665E-1f);
  y = fmaf(y, x, 2.0000714765E-1f);
  y = fmaf(y, x, -2.4999993993E-1f);
  y = fmaf(y, x, 3.3333331174E-1f);
  y = y * x;
  y = y * z;
  y = fmaf(-0.5f, z, y);
  const float lf = x + y;
  const float ef = (float)e;
  const float ln_p = fmaf(ef, 0.693359375f, fmaf(ef, -2.12194440e-4f, lf));
  const float t = (p * ln_p) * -1.44269504088896f;
  return (uint64_t)(std::fmax(t, 0.0f) * 1099511627776.0f);
}

// (n s2 - s1^2) / n^2 from the exact moments (n < 2^32): the numerator exact in 128 bits, rounded once to f64
// (an FMA of its 48-bit halves), two f64 divisions by n, one rounding to f32.  The kernel's epilogue computes the
// same bits.
inline float variance_from_moments(uint64_t n, uint64_t s1, uint64_t s2) {
  const unsigned __int128 d = (unsigned __int128)n * s2 - (unsigned __int128)s1 * s1;
  const double hi = (double)(uint64_t)(d >> 48), lo = (double)(uint64_t)(d & 0xFFFFFFFFFFFFull);
  const double nd = (double)n;
  return (float)(std::fma(hi, 281474976710656.0, lo) / nd / nd);
}

void stats_from_dense(const uint64_t* hist, uint32_t cap, float* mean, float* freq, float* entropy, float* variance) {
  // ecdna-lib 3.0.2 summary statistics [RECALL R8]: all cells counted, zeros included; entropy in bits
  uint64_t n = 0, s1 = 0, s2 = 0;
  for (uint32_t k = 0; k < cap; ++k) { n += hist[k]; s1 += (uint64_t)k * hist[k]; s2 += (uint64_t)k * k * hist[k]; }
  if (n == 0) { *mean = *freq = *entropy = *variance = 0.f; return; }
  const float nf = (float)n;
  const float mu = (float)s1 / nf;
  uint64_t eq = 0;
  for (uint32_t k = 0; k < cap; ++k)
    if (hist[k]) eq += entropy_term_q40(hist[k], n);
  *mean = mu;
  *freq = (float)(n - hist[0]) / nf;
  *entropy = (float)eq * 9.094947017729282e-13f;  // 2^-40
  *variance = variance_from_moments(n, s1, s2);
}

template <class State> struct StateOps;
template <> struct StateOps<VectorState> {
  static void for_each(const VectorState& s, uint32_t cap, uint64_t* dst) {
    std::memset(dst, 0, sizeof(uint64_t) * cap);
    if (cap) dst[0] = s.nminus;
    for (uint16_t k : s.cells) if (k < cap) dst[k] += 1;
  }
};
template <> struct StateOps<HistState> {
  static void for_each(const HistState& s, uint32_t cap, uint64_t* dst) {
    std::memset(dst, 0, sizeof(uint64_t) * cap);
    if (cap) dst[0] = s.nminus;
    for (uint32_t k = 1; k <= s.kmax && k < cap; ++k) dst[k] = s.h[k];
  }
};

// the snapshot rule of process.rs:122-145 / 267-290, evaluated against the PRE-event population:
// while any remaining snapshot size equals the current cell count, pop the FRONT one and save.
template <class State>
void snapshot_check(Recorder& rec, const State& st, float time) {
  const orc_opts* o = rec.o;
  orc_out* out = rec.out;
  const uint64_t cells = st.nminus + st.nplus();
  for (;;) {
    bool any = false;
    for (uint32_t i = rec.snap_front; i < o->n_snap; ++i) any |= (o->snap_cells[i] == cells);
    if (!any) break;
    const uint32_t slot = rec.snap_front++;
    if (out->snap_cells_out) out->snap_cells_out[slot] = cells;
    if (out->snap_time) out->snap_time[slot] = time;
    if (out->snap_hist) StateOps<State>::for_each(st, out->hist_cap, out->snap_hist + (size_t)slot * out->hist_cap);
    out->n_snap_taken = rec.snap_front;
  }
}

// dynamics (CHANGELOG.md:34-40): fixed-width bins of Gillespie time; slot j holds the state seen
// by the first loop iteration whose clock is >= j*dyn_dt.
template <class State>
void dynamics_check(Recorder& rec, const State& st, float time, std::vector<uint64_t>& scratch) {
  const orc_opts* o = rec.o;
  orc_out* out = rec.out;
  while (rec.dyn_next < o->dyn_points && time >= (float)rec.dyn_next * o->dyn_dt) {
    if (out->dyn_out) {
      const uint32_t cap = (uint32_t)scratch.size();
      StateOps<State>::for_each(st, cap, scratch.data());
      float mean, freq, ent, var;
      stats_from_dense(scratch.data(), cap, &mean, &freq, &ent, &var);
      float* d = out->dyn_out + (size_t)rec.dyn_next * 5;
      d[0] = (float)st.nminus; d[1] = (float)st.nplus(); d[2] = mean; d[3] = var; d[4] = ent;
    }
    rec.dyn_next++;
    out->dyn_count = rec.dyn_next;
  }
}

// ------------------------------------------------------------------------------------------
// one replicate: sosa::simulate (called at main.rs:92-99, 166-173) with the reference's
// AdvanceStep callbacks (process.rs:117-185, 262-337) inlined.  Order of operations per
// iteration (SURVEY 8a): stop checks; one waiting time per reaction in the order
// [n- birth, n+ birth, n- death, n+ death] (main.rs:140-145); first minimum wins; snapshot check
// on the pre-event population; event body; time += dt in f32; population copied; iter += 1.
// ------------------------------------------------------------------------------------------
template <class State, class Source, bool REPLAY>
int simulate(const orc_opts& o, orc_out& out, State& st, Source& src, uint64_t hash0) {
  Recorder rec{&o, &out};
  const float rates[4] = {o.b0, o.b1, o.d0, o.d1};
  const int n_react = 4;  // a pure-birth run is the d0=d1=0 case: those reactions never fire
  float time = 0.f;
  uint64_t iter = 0;
  uint64_t hash = hash0, chain = 0;
  uint64_t sum_k = 0, n_div = 0, n_death = 0, trace_len = 0;
  uint32_t kmax = out.kmax;
  std::vector<uint64_t> scratch(o.dyn_points ? std::max<uint32_t>(out.hist_cap, 1u << 16) : 0);
  uint32_t stop;
  for (;;) {
    const uint64_t nplus = st.nplus(), nminus = st.nminus;
    const uint64_t cells = nminus + nplus;
    const uint64_t counted = (o.bd_count_mode == 1 && o.birth_death) ? 2 * cells : cells;
    if (counted == 0) { stop = ORC_STOP_NO_INDIVIDUALS; break; }
    if (iter >= o.max_iter - 1) { stop = ORC_STOP_MAX_ITERS; break; }
    if (time >= o.max_time) { stop = ORC_STOP_MAX_TIME; break; }
    if (counted >= o.max_cells) { stop = ORC_STOP_MAX_CELLS; break; }

    uint32_t event; float dt; uint32_t rk = 0, rk1 = 0;
    if (REPLAY) {
      if (iter >= o.replay_len) { stop = ORC_STOP_REPLAY_END; break; }
      const orc_replay_event& r = o.replay_in[iter];
      event = r.event; dt = r.dt; rk = r.k; rk1 = r.k1;
    } else {
      src.begin_event((uint32_t)iter);
      if constexpr (Source::kDirect) {  // the GPU's native stream: Gillespie's direct method
        float lam[4];
        for (int i = 0; i < n_react; ++i) lam[i] = rates[i] * (float)((i & 1) ? nplus : nminus);
        if (!src.next_reaction(lam, &event, &dt)) { stop = ORC_STOP_ABSORBING; break; }
      } else {  // sosa [RECALL R2, R3]: one waiting time per reaction, first minimum wins
        float best = F_INF; event = 0xffffffffu;
        for (int i = 0; i < n_react; ++i) {
          const float lambda = rates[i] * (float)((i & 1) ? nplus : nminus);
          const float t = src.wait(i, lambda);
          if (t < best) { best = t; event = (uint32_t)i; }
        }
        if (src.dry()) { stop = ORC_STOP_REPLAY_END; break; }
        if (event == 0xffffffffu) { stop = ORC_STOP_ABSORBING; break; }
        dt = best;
      }
    }

    if (o.n_snap) snapshot_check(rec, st, time);
    if (o.dyn_points) dynamics_check(rec, st, time, scratch);

    uint32_t k = 0, k1 = 0;
    if (event == ORC_EV_BIRTH_NMINUS) {
      st.nminus += 1;  // proliferation.rs:113-117
    } else if (event == ORC_EV_DEATH_NMINUS) {
      if (REPLAY && st.nminus == 0) { stop = ORC_STOP_REPLAY_BAD; break; }
      st.nminus -= 1;  // proliferation.rs:135-139
    } else {
      if (REPLAY && nplus == 0) { stop = ORC_STOP_REPLAY_BAD; break; }
      // pick a uniformly random ecDNA+ cell and take it out (proliferation.rs:57 / 126-133)
      uint64_t pidx = 0;
      if (!REPLAY) {
        pidx = src.pick(nplus);
        if (src.dry()) { stop = ORC_STOP_REPLAY_END; break; }
      }
      sum_k += (uint64_t)kmax + 1;
      if constexpr (std::is_same<State, VectorState>::value) {
        k = st.remove_at(pidx);
      } else {
        if (REPLAY) {
          k = rk;
          if (k == 0 || k > st.kmax || st.h[k] == 0) { stop = ORC_STOP_REPLAY_BAD; break; }
        } else {
          k = st.class_at(pidx);
        }
        st.h[k] -= 1; st.np -= 1;
      }
      hash -= hist_weight(k);
      if (event == ORC_EV_DEATH_NPLUS) {
        n_death += 1;
      } else {
        n_div += 1;
        if (k >= 32768) { stop = ORC_STOP_COPY_OVERFLOW; break; }  // checked_mul(2), proliferation.rs:63-67
        const uint32_t n = 2 * k;
        uint32_t k2;
        bool uneven;
        if (REPLAY) {
          k1 = rk1;
          if (k1 > n) { stop = ORC_STOP_REPLAY_BAD; break; }
          k2 = n - k1;
          uneven = (k1 == 0 || k2 == 0);
        } else if (o.segregation == ORC_SEG_DETERMINISTIC) {
          k1 = k2 = k; uneven = false;  // segregation.rs:142-155
        } else {
          uint32_t attempt = 0;
          for (;;) {  // segregation.rs:110-140; redraw loop of segregation.rs:157-174
            k1 = (uint32_t)src.binomial_half(n, attempt);
            k2 = n - k1;
            uneven = (k1 == 0 || k2 == 0);
            if (src.dry() || !(uneven && o.segregation == ORC_SEG_BINOMIAL_NO_UNEVEN)) break;
            ++attempt;
          }
          if (src.dry()) { stop = ORC_STOP_REPLAY_END; break; }
        }
        auto add = [&](uint32_t kk) {
          if constexpr (std::is_same<State, VectorState>::value) st.push(kk);
          else { st.h[kk] += 1; st.np += 1; if (kk > st.kmax) st.kmax = kk; }
          hash += hist_weight(kk);
          if (kk > kmax) kmax = kk;
        };
        if (!uneven) {  // proliferation.rs:82-90
          add(k1); add(k2);
        } else {        // proliferation.rs:91-99: one daughter keeps all 2k copies
          if (REPLAY ? (o.segregation != ORC_SEG_BINOMIAL_NO_NMINUS) : (o.segregation == ORC_SEG_BINOMIAL)) st.nminus += 1;
          add(n);
        }
      }
    }
    time += dt;  // process.rs:184 / 336
    if (out.trace_out && trace_len < out.trace_cap) {
      orc_replay_event& r = out.trace_out[trace_len];
      std::memset(&r, 0, sizeof r);
      r.dt = dt; r.k = (uint16_t)k; r.k1 = (uint16_t)k1; r.event = (uint8_t)event;
    }
    trace_len++;
    chain = chain_step(chain, hash, st.nminus, time);
    if (out.traj_out && iter < out.traj_cap) {
      uint32_t tb; std::memcpy(&tb, &time, 4);
      uint64_t* t = out.traj_out + 4 * iter;
      t[0] = st.nminus; t[1] = st.nplus(); t[2] = tb; t[3] = hash;
    }
    iter++;
  }
  out.stop_reason = stop;
  out.kmax = kmax;
  out.nminus = st.nminus; out.nplus = st.nplus(); out.n_events = iter; out.time = time;
  out.hash = hash; out.chain = chain; out.sum_k = sum_k; out.n_div = n_div; out.n_death = n_death;
  out.trace_len = trace_len;
  if (out.hist && out.hist_cap) StateOps<State>::for_each(st, out.hist_cap, out.hist);
  return 0;
}

template <class State>
uint64_t init_state(const orc_opts& o, State& st, uint32_t& kmax, uint32_t cap);
template <>
uint64_t init_state<VectorState>(const orc_opts& o, VectorState& st, uint32_t& kmax, uint32_t) {
  // EcDNADistribution::new expands the histogram into the per-cell vector [RECALL R4]; entries are
  // expanded in the order given (the reference's HashMap order is unspecified for multi-bin input)
  uint64_t hash = 0;
  for (uint32_t i = 0; i < o.n_init; ++i) {
    if (o.init_k[i] == 0) { st.nminus += o.init_c[i]; continue; }
    for (uint64_t c = 0; c < o.init_c[i]; ++c) st.cells.push_back(o.init_k[i]);
    hash += hist_weight(o.init_k[i]) * o.init_c[i];
    if (o.init_k[i] > kmax) kmax = o.init_k[i];
  }
  return hash;
}
template <>
uint64_t init_state<HistState>(const orc_opts& o, HistState& st, uint32_t& kmax, uint32_t cap) {
  uint64_t hash = 0;
  for (uint32_t i = 0; i < o.n_init; ++i) {
    if (o.init_k[i] == 0) { st.nminus += o.init_c[i]; continue; }
    if (o.init_k[i] >= cap) continue;
    st.h[o.init_k[i]] += (uint32_t)o.init_c[i];
    st.np += o.init_c[i];
    hash += hist_weight(o.init_k[i]) * o.init_c[i];
    if (o.init_k[i] > st.kmax) st.kmax = o.init_k[i];
  }
  kmax = st.kmax;
  return hash;
}

}  // namespace

extern "C" {

int orc_run(const orc_opts* o, orc_out* out) {
  out->kmax = 0; out->n_snap_taken = 0; out->dyn_count = 0;
  if (o->state == 0) {
    if (o->rng == 2) return -1;  // a decision stream cannot address a per-cell vector (SURVEY H2)
    VectorState st;
    st.cells.reserve((size_t)std::min<uint64_t>(o->max_cells + 2, 1ull << 28));
    uint32_t kmax = 0;
    const uint64_t h0 = init_state(*o, st, kmax, 0);
    out->kmax = kmax;
    if (o->rng == 0) {
      RandSource s(o->seed, o->run_idx);
      s.g.rec = out->u64_out; s.g.rec_cap = out->u64_cap;
      if (o->u64_in) { s.g.ext = o->u64_in; s.g.ext_len = o->u64_in_len; }
      const int rc = simulate<VectorState, RandSource, false>(*o, *out, st, s, h0);
      out->u64_len = o->u64_in ? s.g.ext_pos : s.g.rec_len;
      return rc;
    }
    PhiloxSource s(o->seed, o->run_idx);
    return simulate<VectorState, PhiloxSource, false>(*o, *out, st, s, h0);
  }
  HistState st(1u << 16);
  uint32_t kmax = 0;
  const uint64_t h0 = init_state(*o, st, kmax, 1u << 16);
  out->kmax = kmax;
  if (o->rng == 0) { RandSource s(o->seed, o->run_idx); return simulate<HistState, RandSource, false>(*o, *out, st, s, h0); }
  PhiloxSource s(o->seed, o->run_idx);
  if (o->rng == 1) return simulate<HistState, PhiloxSource, false>(*o, *out, st, s, h0);
  return simulate<HistState, PhiloxSource, true>(*o, *out, st, s, h0);
}

uint64_t orc_run_batch(const orc_opts* o, uint64_t idx_begin, uint64_t n_runs, int n_threads, uint64_t* nminus,
                       uint64_t* nplus, float* time, uint64_t* n_events, uint32_t* stop, uint64_t* hist,
                       uint32_t hist_cap, const float* rates_per_run) {
  if (n_threads <= 0) n_threads = (int)std::thread::hardware_concurrency();
  if (n_threads <= 0) n_threads = 1;
  std::atomic<uint64_t> next{0}, total{0};
  auto worker = [&]() {
    uint64_t local = 0;
    for (;;) {
      const uint64_t i = next.fetch_add(1);
      if (i >= n_runs) break;
      orc_opts oo = *o;
      oo.run_idx = idx_begin + i;
      if (rates_per_run) { oo.b0 = rates_per_run[4 * i]; oo.b1 = rates_per_run[4 * i + 1]; oo.d0 = rates_per_run[4 * i + 2]; oo.d1 = rates_per_run[4 * i + 3]; }
      orc_out out;
      std::memset(&out, 0, sizeof out);
      out.hist_cap = hist_cap;
      out.hist = hist ? hist + (size_t)i * hist_cap : nullptr;
      orc_run(&oo, &out);
      if (nminus) nminus[i] = out.nminus;
      if (nplus) nplus[i] = out.nplus;
      if (time) time[i] = out.time;
      if (n_events) n_events[i] = out.n_events;
      if (stop) stop[i] = out.stop_reason;
      local += out.n_events;
    }
    total += local;
  };
  std::vector<std::thread> th;
  for (int t = 1; t < n_threads; ++t) th.emplace_back(worker);
  worker();
  for (auto& t : th) t.join();
  return total.load();
}

// ABC over a batch of prior draws (abc.md:38-55): every draw is one replicate with its own rates plus the
// four distances of its final distribution to the target (KS on the ecDNA distribution, relative mean,
// relative entropy, relative frequency) and the accept flag; what the kernel's fused epilogue computes.
uint64_t orc_abc_batch(const orc_opts* o, uint64_t idx_begin, uint64_t n_runs, int n_threads, const float* rates_per_run,
                       const uint64_t* target, uint32_t target_len, const float thresholds[4], uint32_t hist_cap,
                       float* distances /* [n][4] */, uint8_t* accept /* [n] */, uint64_t* n_events /* [n] or NULL */,
                       uint32_t* stop /* [n] or NULL */) {
  if (n_threads <= 0) n_threads = (int)std::thread::hardware_concurrency();
  if (n_threads <= 0) n_threads = 1;
  float tm, tf, te, tv;
  stats_from_dense(target, target_len, &tm, &tf, &te, &tv);
  std::atomic<uint64_t> next{0}, total{0};
  auto worker = [&]() {
    uint64_t local = 0;
    std::vector<uint64_t> hist(hist_cap);
    for (;;) {
      const uint64_t i = next.fetch_add(1);
      if (i >= n_runs) break;
      orc_opts oo = *o;
      oo.run_idx = idx_begin + i;
      if (rates_per_run) { oo.b0 = rates_per_run[4 * i]; oo.b1 = rates_per_run[4 * i + 1]; oo.d0 = rates_per_run[4 * i + 2]; oo.d1 = rates_per_run[4 * i + 3]; }
      orc_out out;
      std::memset(&out, 0, sizeof out);
      out.hist_cap = hist_cap;
      out.hist = hist.data();
      orc_run(&oo, &out);
      float m, f, e, v;
      stats_from_dense(hist.data(), hist_cap, &m, &f, &e, &v);
      float d[4];
      d[0] = orc_ks_distance(hist.data(), hist_cap, target, target_len);
      d[1] = std::fabs(m - tm) / tm;
      d[2] = std::fabs(e - te) / te;
      d[3] = std::fabs(f - tf) / tf;
      bool ok = true;
      for (int j = 0; j < 4; ++j) {
        if (distances) distances[4 * i + j] = d[j];
        if (thresholds[j] >= 0.f && !(d[j] <= thresholds[j])) ok = false;
      }
      if (accept) accept[i] = ok ? 1 : 0;
      if (n_events) n_events[i] = out.n_events;
      if (stop) stop[i] = out.stop_reason;
      local += out.n_events;
    }
    total += local;
  };
  std::vector<std::thread> th;
  for (int t = 1; t < n_threads; ++t) th.emplace_back(worker);
  worker();
  for (auto& t : th) t.join();
  return total.load();
}

void orc_stats(const uint64_t* hist, uint32_t cap, float* mean, float* frequency, float* entropy, float* variance) {
  stats_from_dense(hist, cap, mean, frequency, entropy, variance);
}

float orc_ks_distance(const uint64_t* h1, uint32_t cap1, const uint64_t* h2, uint32_t cap2) {
  // sup_k |F1(k) - F2(k)| over the two empirical CDFs, zero-copy class included [RECALL R8]
  uint64_t n1 = 0, n2 = 0;
  for (uint32_t k = 0; k < cap1; ++k) n1 += h1[k];
  for (uint32_t k = 0; k < cap2; ++k) n2 += h2[k];
  if (n1 == 0 || n2 == 0) return 1.0f;
  const uint32_t cap = cap1 > cap2 ? cap1 : cap2;
  uint64_t c1 = 0, c2 = 0;
  float best = 0.f;
  for (uint32_t k = 0; k < cap; ++k) {
    if (k < cap1) c1 += h1[k];
    if (k < cap2) c2 += h2[k];
    const float d = std::fabs((float)c1 / (float)n1 - (float)c2 / (float)n2);
    if (d > best) best = d;
  }
  return best;
}

void orc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  std::memcpy(out, ctr, 16);
  philox(out, key[0], key[1]);
}
void orc_chacha_block(const uint32_t key[8], uint64_t counter, uint64_t stream, int rounds, uint32_t out[16]) {
  chacha_block(key, counter, stream, rounds, out);
}
void orc_seed_from_u64(uint64_t seed, uint32_t key[8]) { seed_from_u64(seed, key); }
void orc_chacha8_u64(uint64_t seed, uint64_t stream, uint64_t n, uint64_t* out) {
  ChaCha8 g(seed, stream);
  for (uint64_t i = 0; i < n; ++i) out[i] = g.next_u64();
}
float orc_neg_log_u24(uint32_t m) { return neg_log_u24(m); }
uint32_t orc_binomial_half_philox(uint64_t seed, uint64_t run, uint32_t event, uint32_t attempt, uint32_t n) {
  PhiloxSource s(seed, run);
  s.begin_event(event);
  return (uint32_t)s.binomial_half(n, attempt);
}
uint64_t orc_pick_philox(uint64_t seed, uint64_t run, uint32_t event, uint64_t n) {
  PhiloxSource s(seed, run);
  s.begin_event(event);
  return s.pick(n);
}
void orc_rand_binomial(uint64_t seed, uint64_t stream, uint64_t n, double p, uint64_t count, uint64_t* out) {
  ChaCha8 g(seed, stream);
  for (uint64_t i = 0; i < count; ++i) out[i] = rand_binomial(g, n, p);
}
void orc_rand_exp1_f32(uint64_t seed, uint64_t stream, uint64_t count, float* out) {
  ChaCha8 g(seed, stream);
  for (uint64_t i = 0; i < count; ++i) out[i] = (float)exp1_f64(g);
}
void orc_rand_gen_range(uint64_t seed, uint64_t stream, uint64_t n, uint64_t count, uint64_t* out) {
  ChaCha8 g(seed, stream);
  for (uint64_t i = 0; i < count; ++i) out[i] = g.gen_range(n);
}
void orc_subsample(const uint64_t* hist, uint32_t len, uint64_t want, uint64_t seed, uint64_t run_idx, uint32_t j,
                   uint64_t* out) {
  uint64_t total = 0;
  for (uint32_t k = 0; k < len; ++k) { out[k] = hist[k]; total += hist[k]; }
  if (want >= total) return;
  const bool remove = want > total - want;  // draw the smaller side
  const uint64_t draws = remove ? total - want : want;
  const PhiloxKey key{(uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)run_idx, (uint32_t)(run_idx >> 32)};
  std::vector<uint64_t> w(hist, hist + len);
  for (uint64_t d = 0; d < draws; ++d) {
    const uint64_t n = total - d;
    uint64_t u = 0;
    for (uint32_t attempt = 0;; ++attempt) {  // Lemire's unbiased bounded integer
      uint32_t x[4];
      philox_slot(key, (uint32_t)d, 0x40000000u + j + 65536u * (attempt >> 1), x);
      const uint64_t v = (attempt & 1u) ? (((uint64_t)x[2] << 32) | x[3]) : (((uint64_t)x[0] << 32) | x[1]);
      const unsigned __int128 m = (unsigned __int128)v * n;
      u = (uint64_t)(m >> 64);
      const uint64_t lo = (uint64_t)m;
      if (lo >= n || attempt >= 25u) break;
      if (lo >= (0 - n) % n) break;
    }
    for (uint32_t k = 0; k < len; ++k) {  // the first class whose cumulative count exceeds u
      if (u < w[k]) { w[k] -= 1; break; }
      u -= w[k];
    }
  }
  for (uint32_t k = 0; k < len; ++k) out[k] = remove ? w[k] : hist[k] - w[k];
}

uint64_t orc_hist_weight(uint32_t k) { return hist_weight(k); }

int orc_segregate(uint32_t rule, uint32_t copies, uint64_t seed, uint64_t* k1, uint64_t* k2, uint32_t* uneven) {
  // segregation.rs:28-40: the doubled copy number must be even and > 1
  if (copies <= 1 || (copies & 1)) return -1;
  ChaCha8 g(seed, 0);
  if (rule == ORC_SEG_DETERMINISTIC) { *k1 = *k2 = copies / 2; *uneven = 0; return 0; }
  for (;;) {
    *k1 = rand_binomial(g, copies, 0.5);
    *k2 = copies - *k1;
    const bool u = (*k1 == 0 || *k2 == 0);
    if (u && rule == ORC_SEG_BINOMIAL_NO_UNEVEN) continue;
    *uneven = u ? (rule == ORC_SEG_BINOMIAL_NO_NMINUS ? 2u : 1u) : 0u;  // IsUneven::{False,True,TrueWithoutNMinusIncrease}
    return 0;
  }
}

int orc_apply_event(uint64_t* hist, uint32_t cap, uint32_t event, uint32_t segregation, uint64_t seed,
                    uint32_t* k_out, uint32_t* k1_out, uint32_t* k2_out, uint32_t* uneven_out) {
  // one step of Exponential::increase_nplus / increase_nminus / CellDeath::* on a vector state built
  // from `hist`, exactly as the event loop does it; returns -1 when no ecDNA+ cell exists (the Err
  // of proliferation.rs:57).
  VectorState st;
  st.nminus = hist[0];
  for (uint32_t k = 1; k < cap; ++k) for (uint64_t c = 0; c < hist[k]; ++c) st.cells.push_back((uint16_t)k);
  ChaCha8 g(seed, 0);
  uint32_t k = 0, k1 = 0, k2 = 0, un = 0;
  if (event == ORC_EV_BIRTH_NMINUS) st.nminus += 1;
  else if (event == ORC_EV_DEATH_NMINUS) st.nminus -= 1;
  else {
    if (st.cells.empty()) return -1;
    k = st.remove_at(g.gen_range(st.cells.size()));
    if (event == ORC_EV_BIRTH_NPLUS) {
      if (k >= 32768) return -2;
      const uint32_t n = 2 * k;
      if (segregation == ORC_SEG_DETERMINISTIC) { k1 = k2 = k; }
      else for (;;) {
        k1 = (uint32_t)rand_binomial(g, n, 0.5); k2 = n - k1;
        if ((k1 == 0 || k2 == 0) && segregation == ORC_SEG_BINOMIAL_NO_UNEVEN) continue;
        break;
      }
      if (k1 == 0 || k2 == 0) {
        un = segregation == ORC_SEG_BINOMIAL_NO_NMINUS ? 2 : 1;
        if (un == 1) st.nminus += 1;
        st.push(n);
      } else { st.push(k1); st.push(k2); }
    }
  }
  std::memset(hist, 0, sizeof(uint64_t) * cap);
  hist[0] = st.nminus;
  for (uint16_t c : st.cells) if (c < cap) hist[c] += 1;
  if (k_out) *k_out = k;
  if (k1_out) *k1_out = k1;
  if (k2_out) *k2_out = k2;
  if (uneven_out) *uneven_out = un;
  return 0;
}

}  // extern "C"

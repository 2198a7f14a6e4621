// Device-side building blocks of the B200 stochastic-mapping sampler: arithmetic policy, keyed uniform
// streams (Philox4x32-10 / replay table), R-compatible exponential deviate, categorical draws and the
// small-matrix helpers.  Everything here is header-only and templated on
//   Real   : float | double            (precision of partials, path lengths, weights)
//   NS     : 2 | 4 | 0                 (compile-time state count; 0 = run-time n <= PM_NMAX)
//   EXACT  : deterministic mode        (reference order of operations, no FMA, R's exp_rand, sorted draw)
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#define PM_NMAX 32           // largest state count (generic path)
#define PM_DIC_NMAX 8        // largest state count of the DIC log-likelihood kernels (2-state and k <= 3 hidden-rate models)
#define PM_LOCAL_PATH_MAX 64 // largest merged-path capacity per (branch, site)
#define PM_SMEM_POW 8        // powers of B kept in shared memory (fast mode, NS <= 4)

// device-side error bits (sticky, OR-ed into ChainParams::err_flag)
#define PM_DE_SAMPLE_NA 1u
#define PM_DE_SAMPLE_NEG 2u
#define PM_DE_SAMPLE_ZERO 4u
#define PM_DE_PATH_CAP 8u
#define PM_DE_M_OVERFLOW 16u
#define PM_DE_REPLAY 32u
#define PM_DE_INCONSISTENT 64u
#define PM_DE_BAD_STATE 128u
#define PM_DE_JUMP_LIMIT 256u  // deterministic mode: more real jumps on one branch than a path can hold (63)
#define PM_DE_ZERO_LIK 512u    // pm_expected_sumstats: a site whose data have zero (or, in FP32, underflowed) likelihood

namespace pm {

// ------------------------------------------------------------------------------------------------
// Arithmetic policy.  EXACT pins every product and sum to a separately rounded IEEE operation so the result
// is the one an x86-64 build of the reference (no FMA contraction) computes.
// ------------------------------------------------------------------------------------------------
template <typename Real, bool EXACT> struct Ar;
template <> struct Ar<double, true> {
  static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
  static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
  static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
  static __device__ __forceinline__ double div(double a, double b) { return __ddiv_rn(a, b); }
};
template <> struct Ar<float, true> {
  static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
  static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
  static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
  static __device__ __forceinline__ float div(float a, float b) { return __fdiv_rn(a, b); }
};
template <typename Real> struct Ar<Real, false> {
  static __device__ __forceinline__ Real mul(Real a, Real b) { return a * b; }
  static __device__ __forceinline__ Real add(Real a, Real b) { return a + b; }
  static __device__ __forceinline__ Real sub(Real a, Real b) { return a - b; }
  static __device__ __forceinline__ Real div(Real a, Real b) { return a / b; }
};

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon, Moraes, Dror, Shaw; SC'11).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t o[4]) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  o[0] = c0; o[1] = c1; o[2] = c2; o[3] = c3;
}

// The same with the ten round keys precomputed on the host (RngDesc::rk, kernel-parameter constants): the key schedule
// costs no instructions.
__device__ __forceinline__ void philox4x32_10_rk(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const uint32_t (&rk)[20],
                                                 uint32_t o[4]) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    uint32_t n0 = hi1 ^ c1 ^ rk[2 * r], n2 = hi0 ^ c3 ^ rk[2 * r + 1];
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
  }
  o[0] = c0; o[1] = c1; o[2] = c2; o[3] = c3;
}

enum SlotKind : uint32_t { K_NODE = 0, K_BRSTATE = 1, K_BREXP = 2, K_NODEGRP = 3, K_BRPAIR = 4, K_BRCNT = 5, K_BRPOS = 6, K_BRGAP = 7 };
__device__ __forceinline__ uint32_t make_slot(uint32_t kind, uint32_t idx) { return (kind << 28) | idx; }

// Description of where uniforms come from (per launch).
struct RngDesc {
  uint32_t k0, k1;        // Philox key (per tree)
  uint32_t rk[20];        // its ten round keys: k0 + r * 0x9E3779B9, k1 + r * 0xBB67AE85
  uint32_t site0;         // global index of local site 0
  const int64_t* tab_off; // replay table (device), or nullptr
  const double* tab_u;
  int64_t tab_site_stride;  // N * slots_per_iter
  int64_t tab_base;         // tree * S_global * N * slots_per_iter
  int32_t slots_per_iter;   // 2T-1 + 2E
  int32_t n_nodes;          // 2T-1
};

// 53-bit uniforms strictly inside (0,1), two per Philox block; optionally replayed from a table.
struct StreamD {
  uint32_t k0, k1, site, iter, slot, k;
  uint32_t o0, o1, o2, o3;
  const double* tab; int64_t tab_n; unsigned* err;
  __device__ __forceinline__ void open(const RngDesc& d, uint32_t local_site, uint32_t it, uint32_t kind, uint32_t idx,
                                      unsigned* err_flag) {
    k0 = d.k0; k1 = d.k1; site = d.site0 + local_site; iter = it; slot = make_slot(kind, idx); k = 0; err = err_flag;
    tab = nullptr; tab_n = 0;
    if (d.tab_u) {
      int64_t lin = d.tab_base + (int64_t)site * d.tab_site_stride + (int64_t)it * d.slots_per_iter +
                    (kind == K_NODE ? (int64_t)idx : (int64_t)d.n_nodes + 2 * (int64_t)idx + (kind - 1));
      int64_t a = d.tab_off[lin], b = d.tab_off[lin + 1];
      tab = d.tab_u + a; tab_n = b - a;
    }
  }
  __device__ __forceinline__ double next() {
    double u;
    if (tab) {
      if ((int64_t)k >= tab_n) { atomicOr(err, PM_DE_REPLAY); u = 0.5; } else u = tab[k];
    } else {
      if ((k & 1u) == 0u) {
        uint32_t o[4];
        philox4x32_10(k >> 1, slot, iter, site, k0, k1, o);
        o0 = o[0]; o1 = o[1]; o2 = o[2]; o3 = o[3];
      }
      uint32_t hi = (k & 1u) ? o2 : o0, lo = (k & 1u) ? o3 : o1;
      unsigned long long bits = ((unsigned long long)hi << 21) | (unsigned long long)(lo >> 11);
      u = ((double)bits + 0.5) * (1.0 / 9007199254740992.0);
    }
    k++;
    return u;
  }
};

// 24-bit uniforms strictly inside (0,1), four per Philox block (production, float).  The block is kept in four
// scalar registers (a dynamically indexed array would live in local memory).
struct StreamF {
  uint32_t k0, k1, site, iter, slot, k;
  uint32_t o0, o1, o2, o3;
  __device__ __forceinline__ void open(const RngDesc& d, uint32_t local_site, uint32_t it, uint32_t kind, uint32_t idx,
                                      unsigned*) {
    k0 = d.k0; k1 = d.k1; site = d.site0 + local_site; iter = it; slot = make_slot(kind, idx); k = 0;
  }
  __device__ __forceinline__ float next() {
    const uint32_t j = k & 3u;
    if (j == 0u) {
      uint32_t o[4];
      philox4x32_10(k >> 2, slot, iter, site, k0, k1, o);
      o0 = o[0]; o1 = o[1]; o2 = o[2]; o3 = o[3];
    }
    const uint32_t x = j == 0u ? o0 : j == 1u ? o1 : j == 2u ? o2 : o3;
    k++;
    return ((float)(x >> 8) + 0.5f) * (1.0f / 16777216.0f);
  }
};

template <typename Real, bool EXACT> struct StreamSel { typedef StreamD type; };
template <> struct StreamSel<float, false> { typedef StreamF type; };

// ------------------------------------------------------------------------------------------------
// Standard exponential deviate of the deterministic mode: R's exp_rand (sexp.c, Ahrens & Dieter 1972) on the keyed
// stream — variable uniform consumption.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double exp_rand_R(StreamD& g) {
  const double q[16] = {0.6931471805599453, 0.9333736875190459, 0.9888777961838675, 0.9984589039328340,
                        0.9998292811061389, 0.9999833164100727, 0.9999985691438767, 0.9999998906925558,
                        0.9999999924734159, 0.9999999995283275, 0.9999999999728814, 0.9999999999985598,
                        0.9999999999999289, 0.9999999999999968, 0.9999999999999999, 1.0000000000000000};
  double a = 0.;
  double u = g.next();
  while (u <= 0. || u >= 1.) u = g.next();
  for (;;) {
    u = __dadd_rn(u, u);
    if (u > 1.) break;
    a = __dadd_rn(a, q[0]);
  }
  u = __dsub_rn(u, 1.);
  if (u <= q[0]) return __dadd_rn(a, u);
  int i = 0;
  double ustar = g.next(), umin = ustar;
  do {
    ustar = g.next();
    if (umin > ustar) umin = ustar;
    i++;
  } while (u > q[i]);
  return __dadd_rn(a, __dmul_rn(umin, q[0]));
}

// ------------------------------------------------------------------------------------------------
// Production model of the virtual jumps (statistically the reference's Poisson process of rate Omega + Q_ss on every
// run of the path, src/phylomap.cpp:391-410, drawn differently).  For a run of length L in state s,
// lambda = (Omega + Q_ss) L:
//   lambda <= PM_LAMBDA_INV : the NUMBER of jumps is drawn by inversion of the Poisson cdf from ONE uniform; their
//                             positions are the order statistics of that many uniforms, generated in increasing order
//                             (x <- x + (1 - x)(1 - u^(1/remaining))) and only when a later sweep needs them;
//   lambda >  PM_LAMBDA_INV : exponential gaps until the run is exhausted, like the reference.
// Everything is a pure function of (seed, site, sweep, branch, run, index) through Philox4x32-10, so the sweep that
// consumes the jumps regenerates exactly what the sweep that counted them drew; nothing but the count is stored.
// Word map of one (site, sweep, branch e):
//   pair block  (K_BRPAIR, e >> 1): words 2(e&1), 2(e&1)+1 = A, B.  A: count uniform of run 0.  B: count uniform of
//               run 1 if the path has >= 2 runs, else the uniform of the FIRST position on run 0.
//   (K_BRCNT, e): count uniforms of runs 2, 3, ...      (K_BRPOS, e; run r): the other position uniforms of run r
//   (K_BRGAP, e; run r): exponential gaps of run r      (K_BRSTATE, e): the state draws
// All arithmetic that decides a count or a position is pinned to single IEEE operations so that every kernel that
// evaluates it gets the same bits.
// ------------------------------------------------------------------------------------------------
#define PM_LAMBDA_INV 16

template <typename Real> struct Pin;
template <> struct Pin<float> {
  static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
  static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
  static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
  static __device__ __forceinline__ float div(float a, float b) { return __fdiv_rn(a, b); }
  // (w >> 9 + 1/2) 2^-23: exact in FP32 (24 significant bits), strictly inside (0, 1), one fused multiply-add
  static __device__ __forceinline__ float u01(uint32_t w) { return __fmaf_rn((float)(w >> 9), 1.0f / 8388608.0f, 1.0f / 16777216.0f); }
  // exp(-x) for 0 <= x <= PM_LAMBDA_INV: ex2.approx of x * -log2(e), the two instructions __expf(-x) boils down to once
  // its fix-up for results below 2^-126 is dropped (never needed here: the argument is >= -24); same bits everywhere
  static __device__ __forceinline__ float expm(float x) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(__fmul_rn(x, -1.4426950216293334961f)));
    return r;
  }
  // u^(1/k), 0 < u < 1: lg2.approx / ex2.approx (relative error ~1e-6: it places a jump on its run, nothing compares it)
  static __device__ __forceinline__ float root(float u, int k) {
    float l, r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(u));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(__fdiv_rn(l, (float)k)));
    return r;
  }
  static __device__ __forceinline__ float neglog(float u) { return -logf(u); }
  static __device__ __forceinline__ int above3(float u, float a, float b, float c) {  // three set-on-compare, one 3-input add
    unsigned x, y, z;
    asm("set.gt.u32.f32 %0, %1, %2;" : "=r"(x) : "f"(u), "f"(a));
    asm("set.gt.u32.f32 %0, %1, %2;" : "=r"(y) : "f"(u), "f"(b));
    asm("set.gt.u32.f32 %0, %1, %2;" : "=r"(z) : "f"(u), "f"(c));
    return -(int)(x + y + z);
  }
};
template <> struct Pin<double> {
  static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
  static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
  static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
  static __device__ __forceinline__ double div(double a, double b) { return __ddiv_rn(a, b); }
  static __device__ __forceinline__ double u01(uint32_t w) { return ((double)w + 0.5) * (1.0 / 4294967296.0); }
  static __device__ __forceinline__ double expm(double x) { return exp(-x); }
  static __device__ __forceinline__ double root(double u, int k) { return exp2(__ddiv_rn(log2(u), (double)k)); }
  static __device__ __forceinline__ double neglog(double u) { return -log(u); }
  static __device__ __forceinline__ int above3(double u, double a, double b, double c) { return (u > a ? 1 : 0) + (u > b ? 1 : 0) + (u > c ? 1 : 0); }
};

// number of Poisson(lam) events by inversion of the cdf.  p_k = p_{k-1} * lam * (1/k) with the reciprocal from a
// table (one rounding per multiply, the same in every kernel), so the loop body is two multiplies and an add.
__constant__ float pm_recip[65] = {
    0.f, 1.f, 1.f / 2, 1.f / 3, 1.f / 4, 1.f / 5, 1.f / 6, 1.f / 7, 1.f / 8, 1.f / 9, 1.f / 10, 1.f / 11, 1.f / 12, 1.f / 13,
    1.f / 14, 1.f / 15, 1.f / 16, 1.f / 17, 1.f / 18, 1.f / 19, 1.f / 20, 1.f / 21, 1.f / 22, 1.f / 23, 1.f / 24, 1.f / 25,
    1.f / 26, 1.f / 27, 1.f / 28, 1.f / 29, 1.f / 30, 1.f / 31, 1.f / 32, 1.f / 33, 1.f / 34, 1.f / 35, 1.f / 36, 1.f / 37,
    1.f / 38, 1.f / 39, 1.f / 40, 1.f / 41, 1.f / 42, 1.f / 43, 1.f / 44, 1.f / 45, 1.f / 46, 1.f / 47, 1.f / 48, 1.f / 49,
    1.f / 50, 1.f / 51, 1.f / 52, 1.f / 53, 1.f / 54, 1.f / 55, 1.f / 56, 1.f / 57, 1.f / 58, 1.f / 59, 1.f / 60, 1.f / 61,
    1.f / 62, 1.f / 63, 1.f / 64};

template <typename Real>
__device__ __forceinline__ int poisson_inv(Real lam, uint32_t word) {
  typedef Pin<Real> PN;
  const Real u = PN::u01(word);
  // the first three terms without branches (k <= 2 covers all but ~1e-3 of the draws at lam ~ 0.2) ...
  const Real p0 = PN::expm(lam);
  const Real p1 = PN::mul(p0, lam);
  const Real p2 = PN::mul(PN::mul(p1, lam), (Real)0.5);
  const Real c1 = PN::add(p0, p1), c2 = PN::add(c1, p2);
  int k = Pin<Real>::above3(u, p0, c1, c2);  // (u > p0) + (u > c1) + (u > c2)
  if (k == 3) {  // ... then the general recurrence p_k = p_{k-1} * lam * (1/k)
    Real p = p2, c = c2;
    k = 2;
    while (u > c && k < 64) {
      k++;
      p = PN::mul(PN::mul(p, lam), (Real)pm_recip[k]);
      c = PN::add(c, p);
      if (p < (Real)1e-12 && (Real)k > lam) break;  // cdf saturated below u (resolution of u): stop in the tail
    }
  }
  return k;
}

// position of the next of `remaining` jumps that are uniform on (x, L)
template <typename Real>
__device__ __forceinline__ Real next_order_stat(Real x, Real L, int remaining, uint32_t word) {
  const Real u = Pin<Real>::u01(word);
  const Real frac = Pin<Real>::sub((Real)1, remaining == 1 ? u : Pin<Real>::root(u, remaining));
  return Pin<Real>::add(x, Pin<Real>::mul(Pin<Real>::sub(L, x), frac));
}

// A position on a branch of length t_e is stored as a 16-bit fraction of t_e (upper half of the `meta` word):
// q t_e / 65536, q rounded to nearest -- dyadic fractions (the midpoint of a caller's two-piece map) are exact, and
// encoding a decoded value gives q back, so a jump that survives a sweep does not drift.  Every kernel computes with the
// decoded value only -- lengths, rates, the count-mode decision -- so writer and reader of a path agree to the bit.
// A uniformly distributed position is pos_rand(word): 17 random bits rounded to 16, symmetric about the midpoint.
template <typename Real>
__device__ __forceinline__ Real pos_dec(uint32_t q, Real Le) { return Pin<Real>::mul((Real)q, Pin<Real>::mul(Le, (Real)(1.0 / 65536.0))); }
template <typename Real>
__device__ __forceinline__ uint32_t pos_enc(Real p, Real Le) {
  const Real f = Pin<Real>::add(Pin<Real>::mul(p, Pin<Real>::div((Real)65536, Le)), (Real)0.5);  // NaN (t_e = 0) converts to 0
  return (uint32_t)min(max((int)f, 0), 65535);
}
__device__ __forceinline__ uint32_t pos_rand(uint32_t word) { return min(((word >> 15) + 1u) >> 1, 65535u); }
// shape word of a stored path (16 bits): real jumps nj (0-5; 63 = "63 or more, see the record header") | state of the
// first run (6-10) | state of the second run (11-15)
#define PM_SHAPE(nj, s0, s1) ((uint16_t)((uint32_t)(nj) | ((uint32_t)(s0) << 6) | ((uint32_t)(s1) << 11)))

// lazily evaluated sequence of Philox words: (kind, idx) stream, sub-stream `hi` (run index), word j
struct WordStream {
  uint32_t k0, k1, site, iter, slot, hi, j;
  uint32_t o0, o1, o2, o3;
  __device__ __forceinline__ void open(const RngDesc& d, uint32_t local_site, uint32_t it, uint32_t kind, uint32_t idx, uint32_t run) {
    k0 = d.k0; k1 = d.k1; site = d.site0 + local_site; iter = it; slot = make_slot(kind, idx); hi = run << 20; j = 0;
  }
  __device__ __forceinline__ uint32_t next() {
    const uint32_t q = j & 3u;
    if (q == 0u) {
      uint32_t o[4];
      philox4x32_10(hi | (j >> 2), slot, iter, site, k0, k1, o);
      o0 = o[0]; o1 = o[1]; o2 = o[2]; o3 = o[3];
    }
    j++;
    return q == 0u ? o0 : q == 1u ? o1 : q == 2u ? o2 : o3;
  }
};

__device__ __forceinline__ void pair_block(const RngDesc& d, uint32_t local_site, uint32_t it, uint32_t e, uint32_t o[4]) {
  philox4x32_10_rk(e >> 1, make_slot(K_BRPAIR, 0u), it, d.site0 + local_site, d.rk, o);
}

// pair_block for a kernel that draws many pair blocks of ONE sweep: of the counter (e >> 1, K_BRPAIR slot, sweep, site)
// only the site differs between threads and only e >> 1 between pairs, so what the first three rounds compute from the
// other words is computed once (the same integer operations, regrouped: the same words)
struct PairBlocks {
  uint32_t a, k2, k3, k5;
  // hi and lo word of m * c as ONE wide multiply (written as two, the products are sometimes issued as two instructions)
  static __device__ __forceinline__ void mulw(uint32_t m, uint32_t c, uint32_t& hi, uint32_t& lo) {
    const uint64_t p = (uint64_t)m * c;
    hi = (uint32_t)(p >> 32); lo = (uint32_t)p;
  }
  __device__ __forceinline__ PairBlocks(const RngDesc& d, uint32_t it) {
    a = __umulhi(0xCD9E8D57u, it) ^ make_slot(K_BRPAIR, 0u) ^ d.rk[0];  // round 1: c0' (c2 = it)
    k2 = (0xCD9E8D57u * it) ^ d.rk[2];                                  // round 2: c1 ^ key (c1 = round 1's lo(M1 it))
    k3 = __umulhi(0xD2511F53u, a) ^ d.rk[3];                            // round 2: hi(M0 c0) ^ key
    k5 = (0xD2511F53u * a) ^ d.rk[5];                                   // round 3: c3 ^ key (c3 = round 2's lo(M0 c0))
  }
  // the block of pair j = e >> 1 at global site gsite (= d.site0 + local site)
  __device__ __forceinline__ void block(const RngDesc& d, uint32_t j, uint32_t gsite, uint32_t o[4]) const {
    uint32_t h0, l0, h1, l1;
    mulw(0xD2511F53u, j, h0, l0);                                       // round 1: c2' = h0 ^ site ^ key, c3' = l0
    mulw(0xCD9E8D57u, h0 ^ gsite ^ d.rk[1], h1, l1);                    // round 2
    uint32_t c0 = h1 ^ k2, c1 = l1, c2 = l0 ^ k3, c3;
    mulw(0xD2511F53u, c0, h0, l0);                                      // round 3
    mulw(0xCD9E8D57u, c2, h1, l1);
    c0 = h1 ^ c1 ^ d.rk[4]; c2 = h0 ^ k5; c1 = l1; c3 = l0;
#pragma unroll
    for (int r = 3; r < 10; r++) {
      mulw(0xD2511F53u, c0, h0, l0);
      mulw(0xCD9E8D57u, c2, h1, l1);
      c0 = h1 ^ c1 ^ d.rk[2 * r]; c2 = h0 ^ c3 ^ d.rk[2 * r + 1]; c1 = l1; c3 = l0;
    }
    o[0] = c0; o[1] = c1; o[2] = c2; o[3] = c3;
  }
};

// ------------------------------------------------------------------------------------------------
// Categorical draw.
//  EXACT: RcppArmadillo::sample(sts, 1, TRUE, w): FixProb (validate, divide by the sum of the positive entries),
//         descending insertion sort carrying indices (ties keep index order), cumsum, first j < n-1 with u <= c[j].
//  fast : inverse CDF on the unsorted weights.
// ------------------------------------------------------------------------------------------------
template <typename Real, int NC, bool EXACT, typename U>
__device__ __forceinline__ int categorical(const Real* w, int n, U u, unsigned* err) {
  if (EXACT) {
    Real sum = 0; int npos = 0; unsigned bad = 0;
#pragma unroll
    for (int i = 0; i < n; i++) {
      Real v = w[i];
      if (!isfinite(v)) bad |= PM_DE_SAMPLE_NA;
      else if (v < (Real)0) bad |= PM_DE_SAMPLE_NEG;
      if (v > (Real)0) { npos++; sum = Ar<Real, true>::add(sum, v); }
    }
    if (npos == 0) bad |= PM_DE_SAMPLE_ZERO;
    if (bad) { atomicOr(err, bad); return 0; }
    Real p[NC]; int perm[NC];
#pragma unroll
    for (int i = 0; i < n; i++) { p[i] = Ar<Real, true>::div(w[i], sum); perm[i] = i; }
    // insertion sort, descending, stable: fixed compare-exchange pattern (a non-swap leaves a sorted prefix alone)
#pragma unroll
    for (int i = 1; i < n; i++) {
#pragma unroll
      for (int j = i; j >= 1; j--) {
        if (p[j] > p[j - 1]) {
          Real tp = p[j]; p[j] = p[j - 1]; p[j - 1] = tp;
          int ti = perm[j]; perm[j] = perm[j - 1]; perm[j - 1] = ti;
        }
      }
    }
    Real c = 0;
    int pick = -1;
    const int last = perm[n - 1];
#pragma unroll
    for (int j = 0; j < n - 1; j++) {
      c = (j == 0) ? p[0] : Ar<Real, true>::add(c, p[j]);
      if (pick < 0 && (double)u <= (double)c) pick = perm[j];
    }
    return pick < 0 ? last : pick;
  } else {
    Real tot = 0;
#pragma unroll
    for (int i = 0; i < n; i++) tot += w[i];
    if (!(tot > (Real)0) || !isfinite(tot)) { atomicOr(err, tot > (Real)0 ? PM_DE_SAMPLE_NA : PM_DE_SAMPLE_ZERO); return 0; }
    Real t = (Real)u * tot, c = 0;
    int pick = -1, lastpos = 0;
#pragma unroll
    for (int i = 0; i < n; i++) {
      c += w[i];
      if (w[i] > (Real)0) lastpos = i;
      if (pick < 0 && t < c && w[i] > (Real)0) pick = i;
    }
    return pick < 0 ? lastpos : pick;
  }
}

// ------------------------------------------------------------------------------------------------
// y = M v  (M row-major n x n, left-to-right dot products) and y = M^T v.
// ------------------------------------------------------------------------------------------------
template <typename Real, int NC, bool EXACT>
__device__ __forceinline__ void matvec(const Real* __restrict__ M, int n, Real* v) {
  Real y[NC];
#pragma unroll
  for (int i = 0; i < n; i++) {
    Real acc = 0;
#pragma unroll
    for (int j = 0; j < n; j++) acc = Ar<Real, EXACT>::add(acc, Ar<Real, EXACT>::mul(M[i * n + j], v[j]));
    y[i] = acc;
  }
#pragma unroll
  for (int i = 0; i < n; i++) v[i] = y[i];
}
template <typename Real, int NC, bool EXACT>
__device__ __forceinline__ void matvec_t(const Real* __restrict__ M, int n, Real* v) {
  Real y[NC];
#pragma unroll
  for (int j = 0; j < n; j++) {
    Real acc = 0;
#pragma unroll
    for (int i = 0; i < n; i++) acc = Ar<Real, EXACT>::add(acc, Ar<Real, EXACT>::mul(M[i * n + j], v[i]));
    y[j] = acc;
  }
#pragma unroll
  for (int j = 0; j < n; j++) v[j] = y[j];
}

// Vector load/store of one partial-likelihood row (NS reals) — 16-byte accesses for NS in {2,4}.
template <typename Real, int NS> struct VecIO {
  static __device__ __forceinline__ void load(const Real* p, int n, Real* v) { for (int i = 0; i < n; i++) v[i] = p[i]; }
  static __device__ __forceinline__ void store(Real* p, int n, const Real* v) { for (int i = 0; i < n; i++) p[i] = v[i]; }
};
template <> struct VecIO<float, 4> {
  static __device__ __forceinline__ void load(const float* p, int, float* v) {
    float4 t = *reinterpret_cast<const float4*>(p); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
  static __device__ __forceinline__ void store(float* p, int, const float* v) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]); }
};
template <> struct VecIO<float, 2> {
  static __device__ __forceinline__ void load(const float* p, int, float* v) {
    float2 t = *reinterpret_cast<const float2*>(p); v[0] = t.x; v[1] = t.y; }
  static __device__ __forceinline__ void store(float* p, int, const float* v) {
    *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]); }
};
template <> struct VecIO<double, 4> {
  static __device__ __forceinline__ void load(const double* p, int, double* v) {
    double2 a = reinterpret_cast<const double2*>(p)[0], b = reinterpret_cast<const double2*>(p)[1];
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; }
  static __device__ __forceinline__ void store(double* p, int, const double* v) {
    reinterpret_cast<double2*>(p)[0] = make_double2(v[0], v[1]); reinterpret_cast<double2*>(p)[1] = make_double2(v[2], v[3]); }
};
template <> struct VecIO<double, 2> {
  static __device__ __forceinline__ void load(const double* p, int, double* v) {
    double2 a = *reinterpret_cast<const double2*>(p); v[0] = a.x; v[1] = a.y; }
  static __device__ __forceinline__ void store(double* p, int, const double* v) {
    *reinterpret_cast<double2*>(p) = make_double2(v[0], v[1]); }
};

}  // namespace pm

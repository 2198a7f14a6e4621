// log p(y | Q) by matrix exponentiation — the extra column of the DIC chains maketreelistMCMC2sDICt / ksDICt
// (reference src/phylomap.cpp:3135-3178 PPmakePLD, :3268-3297 PPmakePLksD, :3242-3250, :3383-3390).
//   k_transprob  one thread per branch: P(t_e) = exp(Q t_e) in FP64 (scaling and squaring of a degree-18 Taylor series,
//                expm_taylor; the reference calls arma::expmat, a Pade scheme — same matrix to ~1e-15)
//   k_loglik     Felsenstein pruning with those matrices, same tiling as k_prune (block = 32 sites x 8 warps, level by
//                level), every node rescaled to sum 1 and the logs of the scale factors accumulated in FP64 per site;
//                block partial = sum over its sites of log(sum_j pid_j PL[root][j]) + S; optionally also each site's
//                term on its own (pm_expected_sumstats)
//   k_reduce_ll  fixed-order sum of the block partials into the statistics row
#pragma once
#include "pm_kernels.cuh"

namespace pm {

// exp(t Q) by scaling and squaring of a degree-18 Taylor series in FP64 (Qrow: n x n row-major) into Ex.  VANLOAN: also
// F = int_0^t e^{Qs} C e^{Q(t-s)} ds, the upper-right block of exp(t [[Q, C], [0, Q]]) (Van Loan 1978).  That block matrix
// is upper triangular with Q on both diagonal blocks, so n x n arrays carry it: Taylor term k is (A^k / k!, X_k) with
// X_k = (X_{k-1} A + A^{k-1} / (k-1)! D) / k (A = s Q, D = s C, s = t / 2^squarings), and a squaring maps (E, F) to
// (E^2, E F + F E).  Works for any Q (no eigendecomposition: defective or complex-spectrum generators included).
template <bool VANLOAN>
__device__ __forceinline__ void expm_taylor(const double* __restrict__ Qrow, const double* C, double t, int n, double* Ex, double* F) {
  constexpr int NN = PM_DIC_NMAX * PM_DIC_NMAX, NV = VANLOAN ? NN : 1;
  double X[NN], T[NN], N2[NN], D[NV], Xk[NV], N3[NV];
  double nrm = 0;
  for (int i = 0; i < n; i++) {
    double r = 0;
    for (int j = 0; j < n; j++) r += fabs(Qrow[i * n + j] * t);
    if constexpr (VANLOAN) for (int j = 0; j < n; j++) r += fabs(C[i * n + j] * t);
    nrm = fmax(nrm, r);
  }
  int sq = 0;
  while (nrm > 0.5) { nrm *= 0.5; sq++; }
  const double sc = ldexp(1.0, -sq) * t;
  for (int i = 0; i < n * n; i++) { X[i] = Qrow[i] * sc; Ex[i] = 0; T[i] = 0; }
  for (int i = 0; i < n; i++) { Ex[i * n + i] = 1.0; T[i * n + i] = 1.0; }
  if constexpr (VANLOAN) for (int i = 0; i < n * n; i++) { D[i] = C[i] * sc; Xk[i] = 0; F[i] = 0; }
  for (int k = 1; k <= 18; k++) {
    for (int i = 0; i < n; i++) for (int j = 0; j < n; j++) {
      double acc = 0;
      for (int l = 0; l < n; l++) acc += T[i * n + l] * X[l * n + j];
      N2[i * n + j] = acc / k;
      if constexpr (VANLOAN) {
        double ax = 0;
        for (int l = 0; l < n; l++) ax += Xk[i * n + l] * X[l * n + j] + T[i * n + l] * D[l * n + j];
        N3[i * n + j] = ax / k;
      }
    }
    for (int i = 0; i < n * n; i++) { T[i] = N2[i]; Ex[i] += N2[i]; }
    if constexpr (VANLOAN) for (int i = 0; i < n * n; i++) { Xk[i] = N3[i]; F[i] += N3[i]; }
  }
  for (int r = 0; r < sq; r++) {
    for (int i = 0; i < n; i++) for (int j = 0; j < n; j++) {
      double acc = 0;
      for (int l = 0; l < n; l++) acc += Ex[i * n + l] * Ex[l * n + j];
      N2[i * n + j] = acc;
      if constexpr (VANLOAN) {
        double af = 0;
        for (int l = 0; l < n; l++) af += Ex[i * n + l] * F[l * n + j] + F[i * n + l] * Ex[l * n + j];
        N3[i * n + j] = af;
      }
    }
    for (int i = 0; i < n * n; i++) Ex[i] = N2[i];
    if constexpr (VANLOAN) for (int i = 0; i < n * n; i++) F[i] = N3[i];
  }
}

template <typename Real>
__global__ void k_transprob(const double* __restrict__ Qrow /* n*n row-major */, const double* __restrict__ elen, int E, int n,
                            Real* __restrict__ TP /* [E][n*n] row-major */) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  double Ex[PM_DIC_NMAX * PM_DIC_NMAX];
  expm_taylor<false>(Qrow, nullptr, elen[e], n, Ex, nullptr);
  for (int i = 0; i < n * n; i++) TP[(size_t)e * n * n + i] = (Real)Ex[i];
}

template <typename Real, int NS>
__global__ void __launch_bounds__(256) k_loglik(ChainParams<Real> P, const Real* __restrict__ TP, double* __restrict__ ll_partial,
                                                 double* __restrict__ site_ll /* [S] or nullptr */) {
  constexpr int NC = NS > 0 ? NS : PM_NMAX;  // the direct sampler prunes with this kernel for any n <= PM_NMAX (the DIC chains stop at PM_DIC_NMAX)
  const int n = NS > 0 ? NS : P.n;
  __shared__ double s_S[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const long long S = P.S;
  const long long site_raw = (long long)blockIdx.x * 32 + lane;
  const bool active = site_raw < S;
  const long long site = active ? site_raw : S - 1;
  const bool parity = P.parity_tips != 0;
  const int T = P.T;
  double Sacc = 0.0;
  for (int l = 0; l < P.n_up_levels; l++) {
    const int beg = __ldg(P.up_off + l), end = __ldg(P.up_off + l + 1);
    for (int idx = beg + warp; idx < end; idx += nw) {
      const int* en = P.up_entries + 5 * idx;
      const int pn = __ldg(en), a = __ldg(en + 1), ea = __ldg(en + 2), b = __ldg(en + 3), eb = __ldg(en + 4);
      Real ca[NC], cb[NC];
      if (a < T) tip_partial<Real, NC>(P.tipcode[(long long)a * P.TS + site], n, parity, ca);
      else VecIO<Real, NS>::load(P.PL + ((long long)(a - T) * S + site) * n, n, ca);
      if (b < T) tip_partial<Real, NC>(P.tipcode[(long long)b * P.TS + site], n, parity, cb);
      else VecIO<Real, NS>::load(P.PL + ((long long)(b - T) * S + site) * n, n, cb);
      const Real* __restrict__ Pa = TP + (size_t)ea * n * n;
      const Real* __restrict__ Pb = TP + (size_t)eb * n * n;
      Real out[NC];
      Real sum = 0;
#pragma unroll
      for (int r = 0; r < n; r++) {
        Real xa = 0, xb = 0;
#pragma unroll
        for (int c = 0; c < n; c++) { xa += __ldg(Pa + r * n + c) * ca[c]; xb += __ldg(Pb + r * n + c) * cb[c]; }
        out[r] = xa * xb;
        sum += out[r];
      }
      Sacc += log((double)sum);
      const Real inv = (Real)1 / sum;
#pragma unroll
      for (int r = 0; r < n; r++) out[r] *= inv;
      if (active) VecIO<Real, NS>::store(P.PL + ((long long)(pn - T) * S + site) * n, n, out);
    }
    __syncthreads();
  }
  s_S[warp][lane] = Sacc;
  __syncthreads();
  if (warp == 0) {
    double tot = 0;
    for (int w = 0; w < nw; w++) tot += s_S[w][lane];
    Real pl[NC];
    VecIO<Real, NS>::load(P.PL + ((long long)(P.root - T) * S + site) * n, n, pl);
    double X = 0;
    for (int j = 0; j < n; j++) X += (double)pl[j] * (double)P.model[2 * n * n + j];  // pid
    double v = active ? log(X) + tot : 0.0;
    if (site_ll && active) site_ll[site] = v;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if (lane == 0) ll_partial[blockIdx.x] = v;
  }
}

__global__ void __launch_bounds__(256) k_reduce_ll(const double* __restrict__ ll_partial, long long nblocks, double* out) {
  __shared__ double sh[256];
  double acc = 0;
  for (long long b = threadIdx.x; b < nblocks; b += 256) acc += ll_partial[b];
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) { if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o]; __syncthreads(); }
  if (threadIdx.x == 0) *out = sh[0];
}

}  // namespace pm

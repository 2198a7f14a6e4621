// Exact posterior expectations under a fixed Q, without sampling (pm_expected_sumstats): the simulation-free stochastic
// mapping of Minin & Suchard (2008).  For every site, E[R_i | y] (time in state i) and E[N_ij | y] (i -> j changes) in the
// fixed-Q sampler row layout, and for selected sites the same per branch plus P(X_v = s | y) of every node.
//   k_branch_integrals  one thread per (branch, statistic) k: M_e[k] = int_0^t P(s) C_k P(t - s) ds in FP64
//                       (expm_taylor<true>, pm_loglik.cuh), C_k = E_ii for the dwell in i, Q_ij E_ij for the i -> j changes
//   k_loglik            (pm_loglik.cuh) the inside pass: alpha of every internal node, normalised, in PL
//   k_expect            the outside pass: level by level from the root down, same tiling as k_loglik (block = 32 sites x
//                       8 warps); per entry (parent p, children a, b) y_c = P_c alpha_c, Z = sum beta_p y_a y_b and for each
//                       child c with sibling d, u_c = beta_p (.) y_d:
//                         stats[k] += u_c^T M_{e_c}[k] alpha_c / Z      (every k)
//                         beta_c = P_{e_c}^T u_c, normalised, written over alpha_c (read for the last time here)
//                       so one partials array serves both passes.  Every quantity is a ratio in which the scales of alpha
//                       and beta cancel: a site's result does not depend on the other sites of its block.
// Column k of a statistic: k < n dwell in state k, then the changes (i, j), i != j, row-major with the diagonal skipped.
#pragma once
#include "pm_loglik.cuh"

namespace pm {

template <typename Real>
__global__ void k_branch_integrals(const double* __restrict__ Qrow /* n*n row-major */, const double* __restrict__ elen, int E,
                                   int n, Real* __restrict__ M /* [E][n*n][n*n], each M_e[k] row-major */) {
  const int NK = n * n;
  const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= (long long)E * NK) return;
  const int e = (int)(id / NK), k = (int)(id % NK);
  double C[PM_DIC_NMAX * PM_DIC_NMAX], Ex[PM_DIC_NMAX * PM_DIC_NMAX], F[PM_DIC_NMAX * PM_DIC_NMAX];
  for (int i = 0; i < NK; i++) C[i] = 0;
  if (k < n) C[k * n + k] = 1.0;
  else {
    const int r = k - n, i = r / (n - 1), jj = r % (n - 1), j = jj + (jj >= i ? 1 : 0);
    C[i * n + j] = Qrow[i * n + j];
  }
  expm_taylor<true>(Qrow, C, elen[e], n, Ex, F);
  for (int i = 0; i < NK; i++) M[(size_t)id * NK + i] = (Real)F[i];
}

// WRITE: also the per-branch statistics [S][E][n*n] and the node marginals [S][2T-1][n] of every site of the launch.
// Dynamic shared memory: 8 warps x n*n x 32 doubles (the per-warp accumulators, summed over the warps in a fixed order).
template <typename Real, int NS, bool WRITE>
__global__ void __launch_bounds__(256) k_expect(ChainParams<Real> P, const Real* __restrict__ TP, const Real* __restrict__ M,
                                                double* __restrict__ stats /* [n*n][S] */, double* __restrict__ branch_out,
                                                double* __restrict__ node_out) {
  constexpr int NC = NS > 0 ? NS : PM_DIC_NMAX;
  const int n = NS > 0 ? NS : P.n, NK = n * n;
  extern __shared__ double s_acc[];  // [nw][NK][32]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const long long S = P.S;
  const long long site_raw = (long long)blockIdx.x * 32 + lane;
  const bool active = site_raw < S;
  const long long site = active ? site_raw : S - 1;
  const bool parity = P.parity_tips != 0;
  const int T = P.T, E = P.E;
  // NS = 2 / 4: the accumulators live in registers (4 / 16 doubles); run-time n: in this warp's slice of s_acc
  double acc[NS > 0 ? NS * NS : 1];
  if constexpr (NS > 0) {
#pragma unroll
    for (int k = 0; k < NS * NS; k++) acc[k] = 0;
  } else {
    for (int k = 0; k < NK; k++) s_acc[(warp * NK + k) * 32 + lane] = 0;
  }
  const Real* pid = P.model + 2 * n * n;
  for (int l = P.n_up_levels - 1; l >= 0; l--) {
    const int beg = __ldg(P.up_off + l), end = __ldg(P.up_off + l + 1);
    for (int idx = beg + warp; idx < end; idx += nw) {
      const int* en = P.up_entries + 5 * idx;
      const int pn = __ldg(en);
      const int ch[2] = {__ldg(en + 1), __ldg(en + 3)}, ed[2] = {__ldg(en + 2), __ldg(en + 4)};
      Real bp[NC], al[2][NC], y[2][NC];
      int code[2];
      if (pn == P.root) {
#pragma unroll
        for (int j = 0; j < n; j++) bp[j] = pid[j];
      } else VecIO<Real, NS>::load(P.PL + ((long long)(pn - T) * S + site) * n, n, bp);  // beta_p, written by p's parent's entry
#pragma unroll
      for (int s = 0; s < 2; s++) {
        if (ch[s] < T) { code[s] = P.tipcode[(long long)ch[s] * P.TS + site]; tip_partial<Real, NC>(code[s], n, parity, al[s]); }
        else { code[s] = -1; VecIO<Real, NS>::load(P.PL + ((long long)(ch[s] - T) * S + site) * n, n, al[s]); }
        const Real* __restrict__ Pe = TP + (size_t)ed[s] * n * n;
#pragma unroll
        for (int r = 0; r < n; r++) {
          Real x = 0;
#pragma unroll
          for (int c = 0; c < n; c++) x += __ldg(Pe + r * n + c) * al[s][c];
          y[s][r] = x;
        }
      }
      double Z = 0;
#pragma unroll
      for (int j = 0; j < n; j++) Z += (double)bp[j] * (double)y[0][j] * (double)y[1][j];
      const bool ok = Z > 0 && Z < HUGE_VAL;
      if (!ok && active) atomicOr(P.err_flag, PM_DE_ZERO_LIK);
      const Real iz = ok ? (Real)(1.0 / Z) : (Real)0;
      if (WRITE && pn == P.root && active) {  // the root: pid (.) alpha_root, normalised
        Real ar[NC];
        VecIO<Real, NS>::load(P.PL + ((long long)(pn - T) * S + site) * n, n, ar);
        double m[NC], tot = 0;
        for (int j = 0; j < n; j++) { m[j] = (double)pid[j] * (double)ar[j]; tot += m[j]; }
        for (int j = 0; j < n; j++) node_out[((long long)site * (2 * T - 1) + pn) * n + j] = m[j] / tot;
      }
#pragma unroll
      for (int s = 0; s < 2; s++) {
        Real u[NC], uz[NC];
#pragma unroll
        for (int j = 0; j < n; j++) { u[j] = bp[j] * y[1 - s][j]; uz[j] = u[j] * iz; }
        const Real* __restrict__ Me = M + (size_t)ed[s] * NK * NK;
        double* bo = WRITE ? branch_out + ((long long)site * E + ed[s]) * NK : nullptr;
        // a one-hot tip: u^T M alpha is column `code` of M times u (n terms instead of n^2)
        const bool onehot = !parity && code[s] >= 0;
#pragma unroll
        for (int k = 0; k < NK; k++) {
          const Real* Mk = Me + k * NK;
          Real dot = 0;
          if (onehot) {
#pragma unroll
            for (int a = 0; a < n; a++) dot += __ldg(Mk + a * n + code[s]) * uz[a];
          } else {
#pragma unroll
            for (int a = 0; a < n; a++) {
              Real row[NC];
              VecIO<Real, NS>::load(Mk + a * n, n, row);
              Real x = 0;
#pragma unroll
              for (int b = 0; b < n; b++) x += row[b] * al[s][b];
              dot += uz[a] * x;
            }
          }
          if constexpr (NS > 0) acc[k] += (double)dot;
          else s_acc[(warp * NK + k) * 32 + lane] += (double)dot;
          if (WRITE && active) bo[k] = (double)dot;
        }
        if (code[s] >= 0 && !WRITE) continue;  // a tip's beta is needed for its marginal only
        const Real* __restrict__ Pe = TP + (size_t)ed[s] * n * n;
        Real bc[NC];
        Real sb = 0;
#pragma unroll
        for (int x = 0; x < n; x++) {
          Real v = 0;
#pragma unroll
          for (int r = 0; r < n; r++) v += __ldg(Pe + r * n + x) * u[r];
          bc[x] = v;
          sb += v;
        }
        const Real ib = (Real)1 / sb;
#pragma unroll
        for (int x = 0; x < n; x++) bc[x] *= ib;
        if (code[s] < 0 && active) VecIO<Real, NS>::store(P.PL + ((long long)(ch[s] - T) * S + site) * n, n, bc);
        if (WRITE && active) {
          double m[NC], tot = 0;
          for (int j = 0; j < n; j++) { m[j] = (double)al[s][j] * (double)bc[j]; tot += m[j]; }
          for (int j = 0; j < n; j++) node_out[((long long)site * (2 * T - 1) + ch[s]) * n + j] = m[j] / tot;
        }
      }
    }
    __syncthreads();
  }
  if constexpr (NS > 0) {
#pragma unroll
    for (int k = 0; k < NS * NS; k++) s_acc[(warp * NK + k) * 32 + lane] = acc[k];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < NK * 32; i += blockDim.x) {
    const int k = i >> 5, ln = i & 31;
    const long long s = (long long)blockIdx.x * 32 + ln;
    double tot = 0;
    for (int w = 0; w < nw; w++) tot += s_acc[(w * NK + k) * 32 + ln];
    if (s < S) stats[(long long)k * S + s] = tot;
  }
}

}  // namespace pm

// One character on a small tree: the whole chain of a site in ONE block, its state in shared memory.
//
// The production kernels of pm_kernels.cuh put 32 consecutive SITES on the lanes of a warp.  With one character per call
// -- the reference's literal usage (sumstatMCMC on one trait, src/phylomap.cpp:891) -- 31 of 32 lanes idle and a sweep is a
// chain of dependent L2 / DRAM latencies across five launches (80 us per sweep on a 100-tip tree, against 34 us for a
// flat CPU port on one core).  Here a block owns ONE site and its threads spread over the NODES of a level (pruning :503,
// node draws :591) and over the BRANCHES (paths :264-410); the site's state -- jump counts, shape words, node states,
// partials -- lives in shared memory for the whole call, the sweeps of a fixed-Q chain run back to back inside the launch,
// and nothing is launched, read back or synchronised per sweep.  The read-only topology comes through the L1 cache.
//
// Every draw takes the Philox key, and every item runs the arithmetic, of the 32-sites-per-warp kernels (the node draws
// are keyed by the position of the node in the clade schedule: the `key` word of `SmallOut::down`; the paths run the same item routines,
// PathWorker), so a chain gives the same rows whichever set of kernels runs it -- tests/test_gpu_small.py compares node
// states, piece counts and transition counts bit for bit; dwell-time sums differ in their rounding (summation order).
#pragma once
#include "pm_kernels.cuh"

namespace pm {

// per-sweep output of k_small_chain (reduced over the sites by k_small_reduce, pm_setup_kernels.cuh)
struct SmallOut {
  double* part;              // [nsweeps][S][n] dwell-time sums of every site
  unsigned long long* cnt;   // [nsweeps][n*n]  transition counters, summed over the sites (integer atomics: order-free)
  int* root;                 // [nsweeps]       root state of global site 0 (written by the block that holds it)
  const int4* down;          // top-down draw list: v, parent, edge, key -- grouped by depth (down_off), tips last at their depth
  const int* down_off; int n_down_levels;
  int n_chunks;              // record chunks (rec_cursor rows)
  const int* br_order; int n_order;  // thread i takes branch br_order[i] (-1: none), i < n_order: see pm_host.cu (long branches dealt over the warps)
  // ONE site: the block writes the rows itself, in k_reduce's layout [R(n) | N(n*n) | root | .. | error flag] (device
  // memory or mapped host memory: a rate-updating sampler reads the row right after the launch); nullptr: part / cnt / root
  double* rows; int row_stride, err_slot;
  // PHYLOMAP_B200_SMALL_PROF=1: clock cycles block 0 spends in [prune, node draws, paths (until the slowest warp is through),
  // row] summed over the sweeps, and the per-warp cycles of the path phase [4 + warp] (nullptr: nothing is measured)
  long long* prof;
};

// shared-memory layout (bytes, every section 16-byte aligned)
template <typename Real, int NS>
struct SmallSmem {
  int pl, meta, model, dw, cnt, shape, state, tip, total;
  __host__ __device__ static int up16(int x) { return (x + 15) & ~15; }
  __host__ __device__ SmallSmem(int T) {
    const int E = 2 * T - 2;
    pl = 0;
    meta = up16(pl + (T - 1) * NS * (int)sizeof(Real));
    model = up16(meta + E * 4);
    // B | Bs | pid, scale_old, scale_new, rate_old, rate_new | P_k [PM_SMEM_POW] | P_k transposed [PM_SMEM_POW]
    dw = up16(model + (2 * NS * NS + 5 * NS + 2 * PM_SMEM_POW * NS * NS) * (int)sizeof(Real));
    cnt = up16(dw + 8 * NS * (int)sizeof(double));
    shape = up16(cnt + NS * NS * 4);
    state = up16(shape + E * 2);
    tip = up16(state + 2 * T - 1);
    total = up16(tip + T);
  }
};

// MINB = 1: all the registers the item routine wants (one site: latency); MINB = 2: 128 registers, two blocks per SM (more
// sites than SMs: throughput)
template <typename Real, int NS, int MINB>
__global__ void __launch_bounds__(256, MINB) k_small_chain(ChainParams<Real> P, uint32_t iter0, int nsweeps, SmallOut out) {
  typedef Pin<Real> PN;
  constexpr int n = NS;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int T = P.T, E = P.E, NN = 2 * T - 1;
  const SmallSmem<Real, NS> lay(T);
  Real* const sPL = reinterpret_cast<Real*>(smem_raw + lay.pl);
  uint32_t* const sMeta = reinterpret_cast<uint32_t*>(smem_raw + lay.meta);
  Real* const sB = reinterpret_cast<Real*>(smem_raw + lay.model);
  Real* const sBs = sB + n * n;
  Real* const sVec = sBs + n * n;  // pid | scale_old | scale_new | rate_old | rate_new
  Real* const sPow = sVec + 5 * n;
  Real* const sPowT = sPow + PM_SMEM_POW * n * n;
  double* const s_dw = reinterpret_cast<double*>(smem_raw + lay.dw);  // [8 warps][n]
  unsigned* const s_cnt = reinterpret_cast<unsigned*>(smem_raw + lay.cnt);
  uint16_t* const sShape = reinterpret_cast<uint16_t*>(smem_raw + lay.shape);
  uint8_t* const sState = smem_raw + lay.state;
  uint8_t* const sTip = smem_raw + lay.tip;
  const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const long long S = P.S;
  const long long site = blockIdx.x;
  const uint32_t gsite = P.rng.site0 + (uint32_t)site;
  const bool parity = P.parity_tips != 0;
  const bool full = P.full_counts != 0;
  const int npow_s = min(PM_SMEM_POW, P.jcap);
  const uint32_t kslot = make_slot(K_NODEGRP, 0u);

  // ---- the site's state and the model, once per launch ----
  for (int i = tid; i < n * n; i += nthr) { sB[i] = P.model[i]; sBs[i] = P.model[n * n + i]; }
  for (int i = tid; i < 5 * n; i += nthr) sVec[i] = P.model[2 * n * n + i];
  for (int i = tid; i < npow_s * n * n; i += nthr) {
    const Real v = P.ppow[i];
    sPow[i] = v;
    const int k = i / (n * n), r = (i / n) % n, c = i % n;
    sPowT[k * n * n + c * n + r] = v;
  }
  for (int e = tid; e < E; e += nthr) { sMeta[e] = P.meta[(long long)e * S + site]; sShape[e] = P.shape[(long long)e * S + site]; }
  for (int v = tid; v < NN; v += nthr) sState[v] = P.node_state[(long long)v * S + site];
  for (int v = tid; v < T; v += nthr) sTip[v] = P.tipcode[(long long)v * P.TS + site];
  __syncthreads();
  const Real* const s_rate_old = sVec + 3 * n;
  const Real* const s_rate_new = sVec + 4 * n;

  // P_k times a child's message: the arithmetic of prune_clade_block (`contribution`, `product`), operand for operand
  auto contribution = [&](int k, int code, Real* v) {
    if (code >= 0 && !parity && k < npow_s) {
      VecIO<Real, NS>::load(sPowT + k * NS * NS + code * NS, NS, v);
    } else {
      if (code >= 0) tip_partial<Real, NS>(code, NS, parity, v);
      pow_times<Real, NS>(P, sPow, npow_s, k, v);
    }
  };
  auto product = [&](const Real* va, const Real* vb, Real* o) {
    Real sum = 0;
#pragma unroll
    for (int j = 0; j < NS; j++) { o[j] = vb[j] * va[j]; sum += o[j]; }
    if (sizeof(Real) == 4 && !(sum > (Real)1e-30)) {
      double d[NS], ds = 0;
#pragma unroll
      for (int j = 0; j < NS; j++) { d[j] = (double)vb[j] * (double)va[j]; ds += d[j]; }
      const double di = ds > 0 ? 1.0 / ds : 0.0;
#pragma unroll
      for (int j = 0; j < NS; j++) o[j] = (Real)(d[j] * di);
      return;
    }
    const Real inv = sum > (Real)0 ? fast_rcp<Real>(sum) : (Real)0;
#pragma unroll
    for (int j = 0; j < NS; j++) o[j] *= inv;
  };

  // A tree with at most as many internal nodes / drawn nodes / branches as the block has threads (the reference's
  // configs[0]: 99 / 98 / 198): every node and branch has a thread of its own, and its schedule entry stays in that
  // thread's registers for the whole launch -- a level then costs a compare and a barrier besides the node's arithmetic,
  // where the general loop reads the level's bounds and the entry again in every sweep (two thirds of a level's time).
  const int n_up = T - 1, n_down = __ldg(out.down_off + out.n_down_levels);
  // (only in the one-block-per-SM build: at the 128 registers of the two-per-SM build the entries would be spilled)
  const bool own_up = MINB == 1 && n_up <= nthr, own_down = MINB == 1 && n_down <= nthr, own_br = MINB == 1 && out.n_order <= nthr;
  int u_lv = -1, u_pn = 0, u_a = 0, u_ea = 0, u_b = 0, u_eb = 0;
  if (own_up && tid < n_up) {
    const int* en = P.up_entries + 5 * tid;
    u_pn = __ldg(en); u_a = __ldg(en + 1); u_ea = __ldg(en + 2); u_b = __ldg(en + 3); u_eb = __ldg(en + 4);
    for (int l = 0; l < P.n_up_levels; l++) if (tid >= __ldg(P.up_off + l)) u_lv = l;
  }
  int d_lv = -1;
  int4 d_en = make_int4(0, 0, 0, 0);
  if (own_down && tid < n_down) {
    d_en = __ldg(out.down + tid);
    for (int l = 0; l < out.n_down_levels; l++) if (tid >= __ldg(out.down_off + l)) d_lv = l;
  }
  int b_par = 0, b_chi = 0;
  Real b_len = 0;
  int b_e = -1;
  if (own_br && tid < out.n_order) {
    b_e = __ldg(out.br_order + tid);
    if (b_e >= 0) { b_par = __ldg(P.e_parent + b_e); b_chi = __ldg(P.e_child + b_e); b_len = __ldg(P.e_len + b_e); }
  }

  for (int sw = 0; sw < nsweeps; sw++) {
    const uint32_t iter = iter0 + (uint32_t)sw;
    const int first = iter == 0u ? 1 : 0;
    // the record cursors of this site's slices (per-site slices: rec_shift = 0 whenever this kernel is eligible)
    for (int ck = tid; ck < out.n_chunks; ck += nthr) P.rec_cursor[(long long)ck * P.rec_groups + (site >> P.rec_shift)] = 0;
    for (int i = tid; i < n * n; i += nthr) s_cnt[i] = 0;

    long long tk = 0;
    if (out.prof && blockIdx.x == 0) tk = clock64();
    auto lap = [&](int slot) {  // (after a barrier)
      if (out.prof && blockIdx.x == 0) { const long long t2 = clock64(); if (tid == 0) out.prof[slot] += t2 - tk; tk = t2; }
    };
    // ---- K1: pruning, level by level, one node per thread (makePLrcpp_bigtree :503-529) ----
    auto prune_node = [&](int pn, int a, int ea, int b, int eb) {
      const int ka = (int)(sMeta[ea] & 0xffffu) - 1, kb = (int)(sMeta[eb] & 0xffffu) - 1;
      Real va[NS], vb[NS], o[NS];
      int ca = -1, cb = -1;
      if (a < T) ca = sTip[a]; else VecIO<Real, NS>::load(sPL + (a - T) * NS, NS, va);
      if (b < T) cb = sTip[b]; else VecIO<Real, NS>::load(sPL + (b - T) * NS, NS, vb);
      contribution(kb, cb, vb);
      contribution(ka, ca, va);
      product(va, vb, o);
      VecIO<Real, NS>::store(sPL + (pn - T) * NS, NS, o);
    };
    if (own_up) {
      for (int l = 0; l < P.n_up_levels; l++) {
        if (u_lv == l) prune_node(u_pn, u_a, u_ea, u_b, u_eb);
        __syncthreads();
      }
    } else {
      for (int l = 0; l < P.n_up_levels; l++) {
        const int beg = __ldg(P.up_off + l), end = __ldg(P.up_off + l + 1);
        for (int idx = beg + tid; idx < end; idx += nthr) {
          const int* en = P.up_entries + 5 * idx;
          prune_node(__ldg(en), __ldg(en + 1), __ldg(en + 2), __ldg(en + 3), __ldg(en + 4));
        }
        __syncthreads();
      }
    }

    lap(0);
    // ---- K2: root (:618-627), then the nodes top-down by depth, redrawn tips at their depth (sampleinternalnodes* :591) ----
    if (tid == 0) {
      Real w[NS], pl[NS];
      VecIO<Real, NS>::load(sPL + (P.root - T) * NS, NS, pl);
#pragma unroll
      for (int j = 0; j < NS; j++) w[j] = sVec[j] * pl[j];
      uint32_t o[4];
      philox4x32_10_rk(0xffffffffu, kslot, iter, gsite, P.rng.rk, o);
      const int s = categorical<Real, NS, false>(w, NS, u01_from_word<Real>(o[0]), P.err_flag);
      sState[P.root] = (uint8_t)s;
      if (gsite == 0u && !out.rows) out.root[sw] = s;
    }
    __syncthreads();
    auto draw_node = [&](const int4 en) {  // v, parent, edge, key
      const int ps = sState[en.y];
      const int k = (int)(sMeta[en.z] & 0xffffu) - 1;
      Real pl[NS];
      if (en.x >= T) VecIO<Real, NS>::load(sPL + (en.x - T) * NS, NS, pl);
      // key: class (bits 30-31) | payload.  0: position i in the clade sequences -> block i >> 2, word i & 3;
      // 2: position i in the top list -> block 0x80000000 + i, word 0;  1: tip v -> block 0x40000000 + (v >> 2), word v & 3
      const uint32_t key = (uint32_t)en.w, cls = key >> 30, pay = key & 0x3fffffffu;
      const uint32_t ctr = cls == 2u ? key : (cls << 30) + (pay >> 2);
      const uint32_t wsel = cls == 2u ? 0u : (pay & 3u);
      uint32_t o[4];
      philox4x32_10_rk(ctr, kslot, iter, gsite, P.rng.rk, o);
      const uint32_t word = wsel == 0u ? o[0] : wsel == 1u ? o[1] : wsel == 2u ? o[2] : o[3];
      const int sn = en.x < T ? draw_tip_state<Real, NS>(P, sBs, sPow, npow_s, k, ps, sTip[en.x], parity, word)
                              : draw_node_state<Real, NS>(P, sBs, sPow, npow_s, k, ps, pl, word);
      sState[en.x] = (uint8_t)sn;
    };
    if (own_down) {
      for (int l = 0; l < out.n_down_levels; l++) {
        if (d_lv == l) draw_node(d_en);
        __syncthreads();
      }
    } else {
      for (int l = 0; l < out.n_down_levels; l++) {
        const int beg = __ldg(out.down_off + l), end = __ldg(out.down_off + l + 1);
        for (int idx = beg + tid; idx < end; idx += nthr) draw_node(__ldg(out.down + idx));
        __syncthreads();
      }
    }

    lap(1);
    // ---- K3: one branch per thread.  At most one jump point and count mode: the body of k_paths_easy; everything else:
    // the general item routine of k_paths_hard (which also reproduces what its short routine computes) ----
    PathWorker<Real, NS> pw(P, iter, first, n, sB, sBs, sPow, npow_s, s_cnt, s_dw, s_rate_old, s_rate_new);
    for (int i = tid; i < out.n_order; i += nthr) {
      const int e = own_br ? b_e : __ldg(out.br_order + i);
      if (e < 0) continue;
      const uint32_t mt = sMeta[e];
      const int ps = sState[own_br ? b_par : __ldg(P.e_parent + e)], cs = sState[own_br ? b_chi : __ldg(P.e_child + e)];
      const Real Le = own_br ? b_len : __ldg(P.e_len + e);
      const int m = (int)(mt & 0xffffu);
      const uint32_t q = mt >> 16;
      const bool two = (m == 2) && (ps != cs);
      const Real p1 = pos_dec<Real>(q, Le);
      const Real L0 = two ? p1 : Le;
      const int s0 = two ? ps : cs;
      const Real L1 = two ? PN::sub(Le, p1) : (Real)0;
      const Real lam = PN::add(PN::mul(rate_or_zero(s_rate_new[s0]), L0), PN::mul(rate_or_zero(s_rate_new[cs]), L1));
      const bool hard = (m > 2) || lam > (Real)PM_LAMBDA_INV;
      if (!hard) {
        uint32_t po[4];
        pair_block(P.rng, (uint32_t)site, iter, (uint32_t)e, po);
        const uint32_t wA = (e & 1) ? po[2] : po[0], wB = (e & 1) ? po[3] : po[1];
        const int k = poisson_inv<Real>(lam, wA);
        if (m == 2 && (full || two)) atomicAdd(&s_cnt[ps * n + cs], 1u);
        pw.add_dwell(s0, L0);
        if (two) pw.add_dwell(cs, L1);
        const uint32_t newq = (!two && k == 1) ? pos_rand(wB) : q;
        sMeta[e] = PM_META((two ? 2 : 1) + k, newq);
        sShape[e] = PM_SHAPE(two ? 1 : 0, s0, cs);
      } else {
        HardItem<Real> it;
        it.site = (uint32_t)site; it.e = (uint32_t)e; it.meta = mt;
        it.ends = (uint32_t)ps | ((uint32_t)cs << 8);
        it.shape = first ? 0u : (uint32_t)sShape[e];
        uint32_t mo; uint16_t so;
        pw.general_item(it, mo, so);
        sMeta[e] = mo;
        sShape[e] = so;
      }
    }
    if (pw.errbits) atomicOr(P.err_flag, pw.errbits);
    if (out.prof && blockIdx.x == 0 && lane == 0) out.prof[4 + warp] += clock64() - tk;

    // ---- K4: this site's share of the sweep's row ----
#pragma unroll
    for (int j = 0; j < NS; j++) {
      double v = pw.Rsum[j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
      if (lane == 0) s_dw[warp * n + j] = v;
    }
    __syncthreads();
    lap(2);
    if (out.rows) {  // one site: the row of this sweep is complete here
      double* const row = out.rows + (size_t)sw * out.row_stride;
      if (tid < n) {
        double v = 0;
        for (int w = 0; w < (nthr >> 5); w++) v += s_dw[w * n + tid];
        row[tid] = v;
      }
      for (int i = tid; i < n * n; i += nthr) row[n + i] = (double)s_cnt[i];
      if (tid == 0) {
        row[n + n * n] = gsite == 0u ? (double)sState[P.root] : 0.0;
        row[out.err_slot] = (double)atomicOr(P.err_flag, 0u);  // (every thread's flags were raised before the barrier above)
      }
    } else {
      if (tid < n) {
        double v = 0;
        for (int w = 0; w < (nthr >> 5); w++) v += s_dw[w * n + tid];
        out.part[((long long)sw * S + site) * n + tid] = v;
      }
      for (int i = tid; i < n * n; i += nthr) if (s_cnt[i]) atomicAdd(&out.cnt[(long long)sw * n * n + i], (unsigned long long)s_cnt[i]);
    }
    __syncthreads();
    lap(3);
  }

  // ---- the state goes back to where the other kernels (and export / read-back) expect it ----
  for (int e = tid; e < E; e += nthr) { P.meta[(long long)e * S + site] = sMeta[e]; P.shape[(long long)e * S + site] = sShape[e]; }
  for (int v = tid; v < NN; v += nthr) P.node_state[(long long)v * S + site] = sState[v];
}

}  // namespace pm

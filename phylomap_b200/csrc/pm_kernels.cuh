// The kernels of one MCMC sweep (SURVEY.md §2.3 / §8(a)).  The production arithmetic for n = 2 / 4 has kernels of its
// own; the deterministic mode and a run-time state count run the generic ones.
//   K1  pruning with P_e := B^(m_e - 1): replaces makePLrcpp* (src/phylomap.cpp:490-529, 1077-1088, 1938-1949) +
//       mmmmvFORpl (:446-450).  Production: k_prune_clade (every warp walks whole subtrees alone); generic: k_prune
//       (level by level).
//   K2  root draw + top-down node (and hidden-tip) draws: replaces sampleinternalnodes* (:535-738, 1091-1164, 1314-1403,
//       1952-2046) + updatenodestates (:460-475).  Production: k_nodes_clade (the same clades, pre-order); generic:
//       k_nodes.  k_prune_nodes_clade runs production K1 and K2 in one launch (the stand-alone pair serves the DIC
//       chains and PHYLOMAP_B200_FUSED=0).
//   K3  per (site, branch): regenerate the virtual jumps of the previous sweep, redraw the segment states
//       (resamplebranchstates :264-308), merge + count (shortener :44-73 / shortenerbf :997-1028), draw the new virtual
//       jumps (:391-410), accumulate dwell times (:745-757).  Production (any n): k_paths_easy streams over every branch
//       and completes the paths of at most one jump point, k_paths_hard takes the rest (short shapes first, then the
//       general routine); deterministic mode: k_paths.
//   K4  k_reduce (pm_setup_kernels.cuh): deterministic reduction of the per-block partial sums into one row.
// Few sites on a small tree: k_small_chain (pm_small.cuh) runs whole sweeps in one block per site.
// Data layout in HBM, and how the production and the deterministic mode encode meta and the path records: DESIGN.md §2.
#pragma once
#include <type_traits>
#include "pm_device.cuh"

namespace pm {

template <typename Real>
struct ChainParams {
  int n, T, E;
  const int* cap_off;  // [n_chunks+1] prefix sums of the record capacities of the branch chunks (see k_paths)
  long long S;
  const Real* model;  // [B n*n | Bs n*n | pid n | scale_old n | scale_new n | rate_old n | rate_new n], matrices row-major
  const Real* ppow;   // [jcap][n*n] P_j = Bs * P_{j-1}
  int jcap;
  const int* up_entries; const int* up_off; int n_up_levels;        // 5 ints per internal node: parent, a, ea, b, eb
  // (rec_cursor sits here so that every field below keeps its offset modulo 16: the kernels' parameter loads are
  // scheduled by it, and with the fields shifted by 8 bytes k_loglik<float, 2> takes 35 registers instead of 32)
  int* rec_cursor;  // [n_chunks][rec_groups] records appended so far to the slice of (chunk, site group) in this sweep
  // clade schedule of k_prune_clade (pm_tree.hpp): 8 ints per node, per-warp sequences then the top levels
  const int* cl_entries; const int* cl_warp_off; const int* cl_top_entries; const int* cl_top_off; int n_cl_top_levels;
  // ... and of k_nodes_clade: top part by depth (4 ints per node: v, parent, edge, -), then per-warp pre-order sequences (16 ints)
  const int* cd_top; const int* cd_top_off; int n_cd_top_levels; const int* cd_entries; const int* cd_warp_off;
  // tips to redraw (ks / mt samplers: all of them, entry v = tip v), 2 offsets per tip: the parent's node-state row
  // (parent x S) and the jump-count row of the tip's branch in bytes (edge x S x 4)
  const long long* cd_tips; int n_cd_tips;
  const int* down_entries; const int* down_off; int n_down_levels;  // 3 ints per drawn node: v, parent, edge
  const int* e_parent; const int* e_child; const Real* e_len;
  const long long* maps_off; const double* maps_len;
  int root;
  const uint8_t* tipcode; long long TS;  // tip codes [T][TS]: rows padded to a multiple of 16 sites (4-byte aligned cp.async)
  uint8_t* node_state; uint32_t* meta; Real* PL;
  // PL holds pl_S sites per node row.  Production (n = 2, 4): the fused prune + node-draw kernel keeps the partials of
  // the 32 sites of a block in the slot the block claimed (pl_S = 32 x slots: the partials are per-sweep scratch between
  // K1 and K2); everywhere else pl_S = S and column = site (tile_base = 0: first site of a stand-alone launch).
  long long tile_base, pl_S;
  // production path records: the slice of a branch chunk is shared by the 2^rec_shift consecutive sites of a group
  // (rec_groups groups per chunk): layout [chunk][group][cap], cursor [chunk][group]
  int rec_shift; long long rec_groups;
  // CUDA-graph replay of a sweep (small problems, where launch overhead dominates): the sweep index is read from device
  // memory instead of the kernel argument, so one instantiated graph serves every sweep.  ctl[0] = index of the sweep to
  // run, ctl[1] = row of the statistics block it fills; k_reduce advances both.  nullptr: the arguments hold.
  const uint32_t* ctl;
  // production: branches left to k_paths_hard, one bit per site: hard_ballot[e * W + w] covers sites 32 w .. 32 w + 31.
  // k_paths_hard walks them as wk_total work items, each a run of consecutive ballot words of one branch (sized on the
  // host so that an item holds ~100 set bits whatever the branch length), flattened by k_build_items: item i = branch
  // (bits 32-63) | first ballot word (5-31) | words - 1 (0-4), so that a warp finds its next item with ONE load, issued an
  // item ahead
  uint32_t* hard_ballot; int W;
  long long wk_total;
  long long pad0;  // unused: keeps every field below at its offset modulo 16 (see rec_cursor)
  const unsigned long long* wk_item;
  int chunk;        // branches per record chunk
  long long easy_blocks;  // blocks of k_paths_easy: k_paths_hard's dwell partials follow theirs in dw_partial
  // production: meta[e][s] = m | q << 16, q = 16-bit position (pos_dec) of the jump point of a path with one jump point
  // or one real jump, or the offset of the records of a path with two or more real jumps; shape[e][s] = PM_SHAPE(nj, s0, s1)
  uint16_t* shape;
  Real* rec_len[2]; uint8_t* rec_st[2];  // double-buffered path records: written by sweep i into [i & 1], read by sweep i + 1
  int normalize, full_counts, parity_tips;
  double* dw_partial; unsigned long long* cnt; int* root_out;
  unsigned* err_flag;
  RngDesc rng;
};

template <typename Real, int NC>
__device__ __forceinline__ void tip_partial(int code, int n, bool parity, Real* v) {
#pragma unroll
  for (int j = 0; j < n; j++) v[j] = parity ? (Real)((j & 1) != code) : (Real)(j == code);
}

// v <- Bs^k v
template <typename Real, int NC, bool EXACT>
__device__ __forceinline__ void apply_power(const ChainParams<Real>& P, const Real* sBs, int n, int k, Real* v) {
  if (k <= 0) return;
  if (!EXACT && k < P.jcap) { matvec<Real, NC, false>(P.ppow + (size_t)k * n * n, n, v); return; }
  for (int r = 0; r < k; r++) matvec<Real, NC, EXACT>(sBs, n, v);
}

template <typename Real>
__device__ __forceinline__ void load_model_smem(const ChainParams<Real>& P, int n, Real* sB, Real* sBs, Real* sVec /*3n*/) {
  for (int i = threadIdx.x; i < n * n; i += blockDim.x) { if (sB) sB[i] = P.model[i]; sBs[i] = P.model[n * n + i]; }
  if (sVec) for (int i = threadIdx.x; i < 3 * n; i += blockDim.x) sVec[i] = P.model[2 * n * n + i];
}

// ------------------------------------------------------------------------------------------------
// K1: pruning.  Block = one tile of 32 sites x (blockDim/32) warps; warps stride over the nodes of a level,
// levels are separated by __syncthreads (children written by sibling warps of the same block).
// ------------------------------------------------------------------------------------------------
template <typename Real, int NS, bool EXACT>
__global__ void __launch_bounds__(256) k_prune(ChainParams<Real> P) {
  constexpr int NC = NS > 0 ? NS : PM_NMAX;
  const int n = NS > 0 ? NS : P.n;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Real* sBs = reinterpret_cast<Real*>(smem_raw);
  load_model_smem<Real>(P, n, nullptr, sBs, nullptr);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const long long S = P.S;
  const long long site = (long long)blockIdx.x * 32 + lane;
  const bool active = site < S;
  const bool parity = P.parity_tips != 0;
  for (int l = 0; l < P.n_up_levels; l++) {
    const int beg = __ldg(P.up_off + l), end = __ldg(P.up_off + l + 1);
    for (int idx = beg + warp; idx < end; idx += nw) {
      const int* en = P.up_entries + 5 * idx;
      const int pn = __ldg(en), a = __ldg(en + 1), ea = __ldg(en + 2), b = __ldg(en + 3), eb = __ldg(en + 4);
      if (active) {
        const int ka = (int)(P.meta[(long long)ea * S + site] & 0xffffu) - 1;
        const int kb = (int)(P.meta[(long long)eb * S + site] & 0xffffu) - 1;
        Real va[NC], vb[NC];
        if (a < P.T) tip_partial<Real, NC>(P.tipcode[(long long)a * P.TS + site], n, parity, va);
        else VecIO<Real, NS>::load(P.PL + ((long long)(a - P.T) * S + site) * n, n, va);
        if (b < P.T) tip_partial<Real, NC>(P.tipcode[(long long)b * P.TS + site], n, parity, vb);
        else VecIO<Real, NS>::load(P.PL + ((long long)(b - P.T) * S + site) * n, n, vb);
        apply_power<Real, NC, EXACT>(P, sBs, n, kb, vb);
        apply_power<Real, NC, EXACT>(P, sBs, n, ka, va);
        Real out[NC];
#pragma unroll
        for (int j = 0; j < n; j++) out[j] = Ar<Real, EXACT>::mul(vb[j], va[j]);
        if (P.normalize) {
          if (EXACT) {  // arma::accu order on a row view: two interleaved accumulators
            Real a1 = 0, a2 = 0;
#pragma unroll
            for (int j = 0; j < n; j++) { if (j & 1) a2 = Ar<Real, true>::add(a2, out[j]); else a1 = Ar<Real, true>::add(a1, out[j]); }
            const Real s = Ar<Real, true>::add(a1, a2);
#pragma unroll
            for (int j = 0; j < n; j++) out[j] = Ar<Real, true>::div(out[j], s);
          } else {
            Real s = 0;
#pragma unroll
            for (int j = 0; j < n; j++) s += out[j];
            // structural zeros must stay zeros (no floor); a product that underflowed altogether becomes the zero
            // vector and surfaces in the draw as "Not enough positive probabilities", like a NaN would in the reference
            const Real inv = s > (Real)0 ? (Real)1 / s : (Real)0;
#pragma unroll
            for (int j = 0; j < n; j++) out[j] *= inv;
          }
        }
        VecIO<Real, NS>::store(P.PL + ((long long)(pn - P.T) * S + site) * n, n, out);
      }
    }
    __syncthreads();
  }
}

// v <- P_k v with the tabulated power P_k = B^k (production arithmetic, 2 or 4 states): from shared memory for the
// first PM_SMEM_POW powers (k = 0 is the identity, so lanes with different jump counts do not diverge), from the global
// table up to jcap, repeated mat-vecs beyond.
template <typename Real, int NS>
__device__ __forceinline__ void pow_times(const ChainParams<Real>& P, const Real* sPow, int npow_s, int k, Real* v) {
  if (k < npow_s) {
    const Real* M = sPow + k * NS * NS;
    Real y[NS];
#pragma unroll
    for (int i = 0; i < NS; i++) {
      Real acc = 0;
#pragma unroll
      for (int j = 0; j < NS; j++) acc += M[i * NS + j] * v[j];
      y[i] = acc;
    }
#pragma unroll
    for (int i = 0; i < NS; i++) v[i] = y[i];
  } else if (k < P.jcap) {
    matvec<Real, NS, false>(P.ppow + (size_t)k * NS * NS, NS, v);
  } else {
    for (int r = 0; r < k; r++) matvec<Real, NS, false>(sPow + NS * NS, NS, v);  // P_1 = B
  }
}

// ------------------------------------------------------------------------------------------------
// K1, production arithmetic (2 or 4 states), clade order.  Same tiling as k_prune.  A walk level by level would read
// every partial back from HBM a whole level after writing it (40 % of the 410 KB of traffic per site).  Here every warp
// walks complete subtrees ("clades", pm_tree.hpp) alone, in post-order with the larger child first:
//   * a parent follows its last child immediately -> that child's partial is taken from registers;
//   * its other internal child was finished a few nodes earlier by the same lane -> an L2 hit (same thread, same
//     address: program order makes the store visible to the load);
//   * jump counts, tip codes and the schedule never depend on the kernel's own output, so they are fetched DEPTH nodes
//     ahead with cp.async into a per-warp shared-memory ring;
//   * no block-wide barrier until the clades are done; the few hundred nodes above them go level by level.
// A tip child contributes a COLUMN of P_k, read as one vector from a transposed copy of the table, instead of a mat-vec
// with a one-hot vector; the normalisation uses the hardware reciprocal.
// ------------------------------------------------------------------------------------------------
template <typename Real> __device__ __forceinline__ Real fast_rcp(Real x) { return (Real)1 / x; }
template <> __device__ __forceinline__ float fast_rcp<float>(float x) {  // one MUFU: the result only rescales a partial
  float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r;
}

template <typename Real, int NS>
struct PruneNode {  // one node above the clades: what was loaded for it
  int pn; uint32_t ma, mb;
  int ca, cb;        // tip codes (or -1 for an internal child)
  Real va[NS], vb[NS];
};

// ---- shared-memory ring helpers (32-bit shared addresses, no generic-pointer arithmetic in the loop) ----
__device__ __forceinline__ void cp_async4(unsigned dst, const void* gsrc, bool pred) {
  const int sz = pred ? 4 : 0;  // src-size 0: the destination is zero-filled, nothing is read
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async4(unsigned dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async16(unsigned dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ int lds_u16(unsigned a) { unsigned short v; asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a)); return (int)v; }
__device__ __forceinline__ int lds_u8(unsigned a) { unsigned v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return (int)v; }
__device__ __forceinline__ int4 lds_v4(unsigned a) {
  int4 v; asm volatile("ld.shared.v4.s32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a)); return v;
}
template <typename Real, int NS> __device__ __forceinline__ void lds_vec(unsigned a, Real* v);
template <> __device__ __forceinline__ void lds_vec<float, 4>(unsigned a, float* v) {
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(a));
}
template <> __device__ __forceinline__ void lds_vec<float, 2>(unsigned a, float* v) {
  asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v[0]), "=f"(v[1]) : "r"(a));
}
template <> __device__ __forceinline__ void lds_vec<double, 2>(unsigned a, double* v) {
  asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v[0]), "=d"(v[1]) : "r"(a));
}
template <> __device__ __forceinline__ void lds_vec<double, 4>(unsigned a, double* v) {
  asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v[0]), "=d"(v[1]) : "r"(a));
  asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v[2]), "=d"(v[3]) : "r"(a + 16));
}
__device__ __forceinline__ int lds_s32(unsigned a) { int v; asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }

// One slot of a warp's prefetch ring: what a node needs that does not depend on this kernel's output.
//   [0,128) jump-count words of branch a per site   [128,256) of branch b   [256,288) tip codes of child a   [288,320) of b
//   [320,336) byte offsets of the parent's and of the loaded child's partial (or -1)   [336,340) flags
//   [352,384) schedule words 4..11 (branch and tip offsets) of the node that will take this slot next
#define PM_CLADE_SLOT 384
#define PM_CLADE_ENTRY_INTS 16  // host schedule entry (pm_host.cu): pn_off, x_off | ma_off, mb_off | ta_off, tb_off | flags (64 bytes)

// (the work of one block on the 32 sites [site0, site0 + 32), whose partials live at columns [pl0, pl0 + 32) of the
// partials buffer: called by the stand-alone kernel and by the fused prune + node-draw kernel below)
template <typename Real, int NS, int DEPTH>
__device__ __forceinline__ void prune_clade_block(const ChainParams<Real>& P, const long long site0, const long long pl0) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Real* sPow = reinterpret_cast<Real*>(smem_raw + PM_CLADE_SLOT * 8 * DEPTH);  // [PM_SMEM_POW][NS*NS]  P_k, row-major
  Real* sPowT = sPow + PM_SMEM_POW * NS * NS;                                  // [PM_SMEM_POW][NS*NS]  P_k transposed
  const int npow_s = min(PM_SMEM_POW, P.jcap);
  for (int i = threadIdx.x; i < npow_s * NS * NS; i += blockDim.x) {
    const Real v = P.ppow[i];
    sPow[i] = v;
    const int k = i / (NS * NS), r = (i / NS) % NS, c = i % NS;
    sPowT[k * NS * NS + c * NS + r] = v;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const long long S = P.S;
  const long long site_raw = site0 + lane;
  const bool active = site_raw < S;
  const long long site = active ? site_raw : S - 1;
  const bool parity = P.parity_tips != 0;
  const int T = P.T;
  const uint32_t* __restrict__ meta = P.meta + site;
  const uint8_t* __restrict__ tip = P.tipcode + site;
  Real* PLs = P.PL + (pl0 + (site - site0)) * NS;  // read and written by this thread: no __restrict__, no read-only loads
  const long long rowPL = P.pl_S * NS;

  auto contribution = [&](int k, int code, Real* v) {
    if (code >= 0 && !parity && k < npow_s) {
      VecIO<Real, NS>::load(sPowT + k * NS * NS + code * NS, NS, v);
    } else {
      if (code >= 0) tip_partial<Real, NS>(code, NS, parity, v);
      pow_times<Real, NS>(P, sPow, npow_s, k, v);
    }
  };
  // out = normalised va * vb (production arithmetic always rescales; no floor: structural zeros stay zeros)
  auto product = [&](const Real* va, const Real* vb, Real* out) {
    Real sum = 0;
#pragma unroll
    for (int j = 0; j < NS; j++) { out[j] = vb[j] * va[j]; sum += out[j]; }
    if (sizeof(Real) == 4 && !(sum > (Real)1e-30)) {
      // FP32 only, rare: two clades that each all but settle a DIFFERENT state (1e-20 x 1e-20): the products underflow
      // although both factors are representable.  Redo this node in double, where they cannot.
      double d[NS], ds = 0;
#pragma unroll
      for (int j = 0; j < NS; j++) { d[j] = (double)vb[j] * (double)va[j]; ds += d[j]; }
      const double di = ds > 0 ? 1.0 / ds : 0.0;
#pragma unroll
      for (int j = 0; j < NS; j++) out[j] = (Real)(d[j] * di);
      return;
    }
    const Real inv = sum > (Real)0 ? fast_rcp<Real>(sum) : (Real)0;
#pragma unroll
    for (int j = 0; j < NS; j++) out[j] *= inv;
  };

  // ---- phase 1: this warp's clades ----
  {
    const int i0 = __ldg(P.cl_warp_off + warp), i1 = __ldg(P.cl_warp_off + warp + 1);
    unsigned ring = (unsigned)__cvta_generic_to_shared(smem_raw) + warp * (DEPTH * PM_CLADE_SLOT);
    asm volatile("" : "+r"(ring));  // kept in a register: the compiler would rebuild it from %tid and the window base per node
    char* const plb = reinterpret_cast<char*>(PLs);
    const char* const mtb = reinterpret_cast<const char*>(meta);
    const char* const tpb = reinterpret_cast<const char*>(P.tipcode) + site0 + 4 * (lane & 7);  // lanes 0..7: four tip codes each
    const bool tip_in = site0 + 4 * (lane & 7) < S;
    const int4* ep = reinterpret_cast<const int4*>(P.cl_entries) + 4 * (long long)i0;  // entry of the next node to issue
    // keep the per-lane bases in registers: recomputing them from blockIdx / S every iteration costs more than they do
    unsigned long long plb_u = reinterpret_cast<unsigned long long>(plb), mtb_u = reinterpret_cast<unsigned long long>(mtb),
                       tpb_u = reinterpret_cast<unsigned long long>(tpb);
    int act = active ? 1 : 0;
    asm volatile("" : "+l"(plb_u), "+l"(mtb_u), "+l"(tpb_u), "+r"(act));
    auto off64 = [](int lo, int hi) { return (long long)(((unsigned long long)(unsigned)hi << 32) | (unsigned)lo); };
    // start the asynchronous copies of the node with entry *e (q1, q2 = its second and third quarter) into the slot:
    // two instructions for the jump-count words (every lane, one word per branch) and ONE for the rest, by lane role:
    // lanes 0..7 four tip codes of child a each, 8..15 of child b, 16..20 the five header words, 21..28 the eight
    // offset words of the node DEPTH further on (read back from the slot when that node is issued into it).  A child
    // that is not a tip copies nothing (source size 0 zero-fills).
    // Branch-free by per-lane constants: source = cbase + X with X = the entry pointer (entry roles) or the tip-row
    // offset of child a / b (tip roles; negative = not a tip -> nothing to copy).
    const bool role_b = (lane >> 3) == 1, role_nxt = lane >= 21, role_ent = lane >= 16;
    unsigned long long cbase = role_ent ? (unsigned long long)(role_nxt ? (long long)DEPTH * 64 + 16 + 4 * (lane - 21)  // words 4..11 of entry e + DEPTH
                                                                        : (lane == 20 ? 48 : 4 * (lane - 16)))           // words 0..3 and 12 of entry e
                                        : tpb_u;
    // lanes 29..31 copy nothing: their zero-fill lands in the unused words [340, 352) of the slot
    unsigned dst_off = lane >= 29 ? 340 + 4 * (lane - 29) : role_nxt ? 352 + 4 * (lane - 21) : 256 + 4 * lane;
    // bit 0: this lane copies at all; 1: only while there is a node DEPTH further on; 2: role b; 3: entry role
    int lrole = ((lane < 29 && (role_ent || tip_in)) ? 1 : 0) | (role_nxt ? 2 : 0) | (role_b ? 4 : 0) | (role_ent ? 8 : 0);
    unsigned lane4 = 4 * lane;
    // fast path only with the full shared-memory table (a power of two, so one OR tests both counts) and one-hot tips
    unsigned fast_pow = ((!parity || NS == 4) && npow_s == PM_SMEM_POW) ? (unsigned)PM_SMEM_POW : 0u;
    int lane_v = lane;
    asm volatile("" : "+l"(cbase), "+r"(dst_off), "+r"(lrole), "+r"(lane4), "+r"(fast_pow), "+r"(lane_v));
    auto issue = [&](unsigned slot, const int4* e, const int4& q1, const int4& q2, bool more) {
      cp_async4(slot + lane4, reinterpret_cast<const char*>(mtb_u) + off64(q1.x, q1.y));
      cp_async4(slot + 128 + lane4, reinterpret_cast<const char*>(mtb_u) + off64(q1.z, q1.w));
      const long long tipoff = (lrole & 4) ? off64(q2.z, q2.w) : off64(q2.x, q2.y);
      const long long X = (lrole & 8) ? reinterpret_cast<long long>(e) : tipoff;
      const bool on = (lrole & 1) && X >= 0 && (more || !(lrole & 2));
      cp_async4(slot + dst_off, reinterpret_cast<const char*>(cbase + (unsigned long long)(X >= 0 ? X : 0LL)), on);
    };
#pragma unroll 1
    for (int u = 0; u < DEPTH; u++) {
      if (i0 + u < i1) { issue(ring + u * PM_CLADE_SLOT, ep, __ldg(ep + 1), __ldg(ep + 2), i0 + u + DEPTH < i1); ep += 4; }
      cp_async_commit();
    }
    Real prev[NS], xA[NS], xB[NS];  // xA / xB: the loaded child of the current / next node, roles alternate
#pragma unroll
    for (int j = 0; j < NS; j++) { prev[j] = 0; xA[j] = 0; xB[j] = 0; }
    long long pnA = 0, pnB = 0;
    int flA = 0, flB = 0;
    if (i0 < i1) {
      cp_async_wait<DEPTH - 1>();
      __syncwarp();
      const int4 h = lds_v4(ring + 320);
      pnA = off64(h.x, h.y);
      flA = lds_s32(ring + 336);
    }
    unsigned slot = ring;
    unsigned ring_end = ring + DEPTH * PM_CLADE_SLOT;
    asm volatile("" : "+r"(ring_end));
    // one node: (pn_off, fl, xcur) describe it, (pn_off_n, fl_n, xnext) receive the next node's
    // P_k times a tip's partial: one column of P_k for a one-hot tip; for the hidden-rate models' parity tips
    // (1,0,1,0) / (0,1,0,1) the sum of the two columns whose state has the observed parity -- the same additions, in the
    // same order, as the mat-vec with that 0/1 vector
    auto tip_column = [&](int k, int code, Real* v) {
      if (!parity) { VecIO<Real, NS>::load(sPowT + (k * NS + code) * NS, NS, v); return; }
      Real c0[NS], c1[NS];
      const int j0 = 1 - code;
      VecIO<Real, NS>::load(sPowT + (k * NS + j0) * NS, NS, c0);
      VecIO<Real, NS>::load(sPowT + (k * NS + (j0 + 2 < NS ? j0 + 2 : j0)) * NS, NS, c1);
#pragma unroll
      for (int j = 0; j < NS; j++) v[j] = c0[j] + c1[j];
    };
    auto step = [&](int idx, long long pn_off, int fl, const Real* xcur, long long& pn_off_n, int& fl_n, Real* xnext) {
      const unsigned slot_n = (slot + PM_CLADE_SLOT == ring_end) ? ring : slot + PM_CLADE_SLOT;
      // the group of node idx + 1 has landed as well (DEPTH - 2 younger ones may still be in flight): its header tells
      // which internal child to fetch.  That child is not the node computed now, so it was stored at least one node ago.
      cp_async_wait<DEPTH - 2>();
      __syncwarp();
      if (idx + 1 < i1) {
        const int4 h = lds_v4(slot_n + 320);
        fl_n = lds_s32(slot_n + 336);
        pn_off_n = off64(h.x, h.y);
        if (h.w >= 0) VecIO<Real, NS>::load(reinterpret_cast<const Real*>(plb_u + (unsigned long long)off64(h.z, h.w)), NS, xnext);
      }
      const int ma = lds_u16(slot + lane4), mb = lds_u16(slot + 128 + lane4);
      Real va[NS], vb[NS];
      // fast path (warp-uniform): one-hot tips and every jump count inside the shared-memory table -> straight-line code,
      // a tip child is one column of P_k, an internal child one 4 x 4 (2 x 2) product with P_k
      const bool fast = __all_sync(0xffffffffu, ((unsigned)(ma - 1) | (unsigned)(mb - 1)) < fast_pow);
      if (fast) {
        if (fl & 16) tip_column(ma - 1, lds_u8(slot + 256 + lane_v), va);
        else {
          const Real* Ma = sPow + (ma - 1) * NS * NS;
          Real src[NS];
#pragma unroll
          for (int j = 0; j < NS; j++) src[j] = (fl & 1) ? prev[j] : xcur[j];
#pragma unroll
          for (int r = 0; r < NS; r++) {
            Real row[NS];
            VecIO<Real, NS>::load(Ma + r * NS, NS, row);
            Real acc = 0;
#pragma unroll
            for (int c = 0; c < NS; c++) acc += row[c] * src[c];
            va[r] = acc;
          }
        }
        if (fl & 32) tip_column(mb - 1, lds_u8(slot + 288 + lane_v), vb);
        else {
          const Real* Mb = sPow + (mb - 1) * NS * NS;
          Real src[NS];
#pragma unroll
          for (int j = 0; j < NS; j++) src[j] = (fl & 2) ? prev[j] : xcur[j];
#pragma unroll
          for (int r = 0; r < NS; r++) {
            Real row[NS];
            VecIO<Real, NS>::load(Mb + r * NS, NS, row);
            Real acc = 0;
#pragma unroll
            for (int c = 0; c < NS; c++) acc += row[c] * src[c];
            vb[r] = acc;
          }
        }
      } else {
        const int ca = (fl & 16) ? lds_u8(slot + 256 + lane_v) : -1, cb = (fl & 32) ? lds_u8(slot + 288 + lane_v) : -1;
#pragma unroll
        for (int j = 0; j < NS; j++) {
          va[j] = (fl & 1) ? prev[j] : xcur[j];
          vb[j] = (fl & 2) ? prev[j] : xcur[j];
        }
        contribution(mb - 1, cb, vb);
        contribution(ma - 1, ca, va);
      }
      product(va, vb, prev);
      if (act) VecIO<Real, NS>::store(reinterpret_cast<Real*>(plb_u + (unsigned long long)pn_off), NS, prev);
      __syncwarp();  // every lane has read the slot before it is refilled
      if (idx + DEPTH < i1) {  // the slot just consumed also carried this node's offset words
        const int4 q1 = lds_v4(slot + 352), q2 = lds_v4(slot + 368);
        __syncwarp();
        issue(slot, ep, q1, q2, idx + 2 * DEPTH < i1);
        ep += 4;
      }
      cp_async_commit();
      slot = slot_n;
    };
#pragma unroll 1
    for (int idx = i0; idx < i1; idx += 2) {
      step(idx, pnA, flA, xA, pnB, flB, xB);
      if (idx + 1 < i1) step(idx + 1, pnB, flB, xB, pnA, flA, xA);
    }
    cp_async_wait<0>();
  }
  __syncthreads();

  // ---- phase 2: the nodes above the clades, level by level (children come from memory) ----
  const int4* __restrict__ ent = reinterpret_cast<const int4*>(P.cl_top_entries);  // 8 ints per node: pn a ea b | eb - - -
  auto load = [&](PruneNode<Real, NS>& nd, int id) {
    const int4 e0 = __ldg(ent + 2 * id), e1 = __ldg(ent + 2 * id + 1);
    nd.pn = e0.x;
    nd.ma = meta[(long long)e0.z * S];
    nd.mb = meta[(long long)e1.x * S];
    nd.ca = -1; nd.cb = -1;
    if (e0.y < T) nd.ca = tip[(long long)e0.y * P.TS];
    else VecIO<Real, NS>::load(PLs + (long long)(e0.y - T) * rowPL, NS, nd.va);
    if (e0.w < T) nd.cb = tip[(long long)e0.w * P.TS];
    else VecIO<Real, NS>::load(PLs + (long long)(e0.w - T) * rowPL, NS, nd.vb);
  };
  auto compute = [&](PruneNode<Real, NS>& nd) {
    contribution((int)(nd.mb & 0xffffu) - 1, nd.cb, nd.vb);
    contribution((int)(nd.ma & 0xffffu) - 1, nd.ca, nd.va);
    Real out[NS];
    product(nd.va, nd.vb, out);
    if (active) VecIO<Real, NS>::store(PLs + (long long)(nd.pn - T) * rowPL, NS, out);
  };
  PruneNode<Real, NS> A, B;
  for (int l = 0; l < P.n_cl_top_levels; l++) {
    const int beg = __ldg(P.cl_top_off + l), end = __ldg(P.cl_top_off + l + 1);
    int idx = beg + warp;
    if (idx < end) load(A, idx);
    while (idx < end) {
      if (idx + nw < end) load(B, idx + nw);
      compute(A);
      idx += nw;
      if (idx >= end) break;
      if (idx + nw < end) load(A, idx + nw);
      compute(B);
      idx += nw;
    }
    __syncthreads();
  }
}

template <typename Real, int NS, int DEPTH, int MINB>
__global__ void __launch_bounds__(256, MINB) k_prune_clade(ChainParams<Real> P) {
  prune_clade_block<Real, NS, DEPTH>(P, P.tile_base + (long long)blockIdx.x * 32, (long long)blockIdx.x * 32);
}

// ------------------------------------------------------------------------------------------------
// K2: node states, top-down.
// ------------------------------------------------------------------------------------------------
template <typename Real, int NS, bool EXACT>
__global__ void __launch_bounds__(256) k_nodes(ChainParams<Real> P, uint32_t iter) {
  if (P.ctl) iter = P.ctl[0];
  constexpr int NC = NS > 0 ? NS : PM_NMAX;
  typedef typename StreamSel<Real, EXACT>::type Stream;
  const int n = NS > 0 ? NS : P.n;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Real* sBs = reinterpret_cast<Real*>(smem_raw);
  Real* sVec = sBs + n * n;  // pid, scale_old, scale_new
  load_model_smem<Real>(P, n, nullptr, sBs, sVec);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const long long S = P.S;
  const long long site = (long long)blockIdx.x * 32 + lane;
  const bool active = site < S;
  const bool parity = P.parity_tips != 0;
  if (warp == 0 && active) {  // root :618-627
    Real w[NC], pl[NC];
    VecIO<Real, NS>::load(P.PL + ((long long)(P.root - P.T) * S + site) * n, n, pl);
#pragma unroll
    for (int j = 0; j < n; j++) w[j] = Ar<Real, EXACT>::mul(sVec[j], pl[j]);
    Stream g; g.open(P.rng, (uint32_t)site, iter, K_NODE, (uint32_t)P.root, P.err_flag);
    const int s = categorical<Real, NC, EXACT>(w, n, g.next(), P.err_flag);
    P.node_state[(long long)P.root * S + site] = (uint8_t)s;
    if (P.rng.site0 + (uint32_t)site == 0u) *P.root_out = s;
  }
  __syncthreads();
  for (int l = 0; l < P.n_down_levels; l++) {
    const int beg = __ldg(P.down_off + l), end = __ldg(P.down_off + l + 1);
    for (int idx = beg + warp; idx < end; idx += nw) {
      const int* en = P.down_entries + 3 * idx;
      const int v = __ldg(en), pn = __ldg(en + 1), e = __ldg(en + 2);
      if (active) {
        const int ps = P.node_state[(long long)pn * S + site];
        const int k = (int)(P.meta[(long long)e * S + site] & 0xffffu) - 1;
        Real w[NC], pl[NC];
        bool done = false;
        if (!EXACT && k > 0) {  // row ps of B^k from the table
          const Real* M = k < P.jcap ? P.ppow + (size_t)k * n * n : nullptr;
          if (M) {
#pragma unroll
            for (int j = 0; j < n; j++) w[j] = M[ps * n + j];
            done = true;
          }
        }
        if (!done) {  // (B^T)^k e_ps as k mat-vecs, Tvmmp :431-436
#pragma unroll
          for (int j = 0; j < n; j++) w[j] = (Real)(j == ps);
          for (int r = 0; r < k; r++) matvec_t<Real, NC, EXACT>(sBs, n, w);
        }
        if (v < P.T) tip_partial<Real, NC>(P.tipcode[(long long)v * P.TS + site], n, parity, pl);
        else VecIO<Real, NS>::load(P.PL + ((long long)(v - P.T) * S + site) * n, n, pl);
#pragma unroll
        for (int j = 0; j < n; j++) w[j] = Ar<Real, EXACT>::mul(w[j], pl[j]);
        Stream g; g.open(P.rng, (uint32_t)site, iter, K_NODE, (uint32_t)v, P.err_flag);
        const int s = categorical<Real, NC, EXACT>(w, n, g.next(), P.err_flag);
        P.node_state[(long long)v * S + site] = (uint8_t)s;
      }
    }
    __syncthreads();
  }
}

// uniform in (0, 1) from one Philox word (production node draws: one block feeds four nodes, which cuts the dominant
// cost of a draw -- ten Philox rounds -- by four)
template <typename Real> __device__ __forceinline__ Real u01_from_word(uint32_t x);
template <> __device__ __forceinline__ float u01_from_word<float>(uint32_t x) { return ((float)(x >> 8) + 0.5f) * (1.0f / 16777216.0f); }
template <> __device__ __forceinline__ double u01_from_word<double>(uint32_t x) { return ((double)x + 0.5) * (1.0 / 4294967296.0); }

// ------------------------------------------------------------------------------------------------
// K3, deterministic mode (FP64, the reference's order of operations).  Thread = one site x a chunk of branches; block =
// 128 consecutive sites.  Per (site, branch): regenerate the virtual jumps of the previous sweep, redraw the segment
// states (resamplebranchstates :264-308), merge + count (shortener :44-73 / shortenerbf :997-1028), draw the new virtual
// jumps (:391-410), accumulate dwell times (:745-757); then a block-level reduction.  meta = m | real jumps nj << 16 |
// first state << 24, and every path keeps its nj + 1 runs as records.
// ------------------------------------------------------------------------------------------------
template <int NS>
__global__ void __launch_bounds__(128) k_paths(ChainParams<double> P, uint32_t iter, int first, int chunk) {
  if (P.ctl) { iter = P.ctl[0]; first = iter == 0u; }
  constexpr int NC = NS > 0 ? NS : PM_NMAX;
  typedef Ar<double, true> A;
  const int n = NS > 0 ? NS : P.n;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* s_dw = reinterpret_cast<double*>(smem_raw);                     // [4 warps][n] (NS>0) or [n] atomics (NS==0)
  unsigned* s_cnt = reinterpret_cast<unsigned*>(s_dw + 4 * n);           // [n*n]
  double* sB = reinterpret_cast<double*>(s_cnt + n * n + ((n * n) & 1));  // dense B (forward row)
  double* sBs = sB + n * n;
  double* sVec = sBs + n * n;
  load_model_smem<double>(P, n, sB, sBs, sVec);
  for (int i = threadIdx.x; i < n * n; i += blockDim.x) s_cnt[i] = 0;
  for (int i = threadIdx.x; i < 4 * n; i += blockDim.x) s_dw[i] = 0.0;
  __syncthreads();
  const double* s_scale_old = sVec + n;
  const double* s_scale_new = sVec + 2 * n;
  const long long S = P.S;
  const long long site = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = site < S;
  const int e0 = blockIdx.y * chunk, e1 = min(P.E, e0 + chunk);
  const int cap0 = __ldg(P.cap_off + blockIdx.y), cap_c = __ldg(P.cap_off + blockIdx.y + 1) - cap0;
  const long long abase = (long long)cap0 * S + (active ? site : 0) * (long long)cap_c;
  const double* __restrict__ rd_len = P.rec_len[(iter & 1u) ^ 1u] + abase;
  const uint8_t* __restrict__ rd_st = P.rec_st[(iter & 1u) ^ 1u] + abase;
  double* __restrict__ wr_len = P.rec_len[iter & 1u] + abase;
  uint8_t* __restrict__ wr_st = P.rec_st[iter & 1u] + abase;
  int rd = 0, wr = 0;
  const bool full = P.full_counts != 0;
  double Racc[NS > 0 ? NS : 1];
#pragma unroll
  for (int j = 0; j < (NS > 0 ? NS : 1); j++) Racc[j] = 0;
  unsigned errbits = 0;

  if (active) for (int e = e0; e < e1; e++) {
    const long long pe = (long long)e * S + site;
    const uint32_t mt = P.meta[pe];
    const int m = (int)(mt & 0xffffu), nj = (int)((mt >> 16) & 0xffu);
    const int ps = P.node_state[(long long)__ldg(P.e_parent + e) * S + site];
    const int cs = P.node_state[(long long)__ldg(P.e_child + e) * S + site];
    int nout = 0, newm = 0, sfirst = 0;
    StreamD gnew; gnew.open(P.rng, (uint32_t)site, iter, K_BREXP, (uint32_t)e, P.err_flag);

    // emit one merged run: store it, add its dwell time, draw its new virtual jumps (count only)
    auto emit = [&](double L, int s) {
      if (nout == 0) sfirst = s;
      if (wr < cap_c && nout < PM_LOCAL_PATH_MAX) { wr_len[wr] = L; wr_st[wr] = (uint8_t)s; wr++; }
      else errbits |= (nout >= PM_LOCAL_PATH_MAX) ? PM_DE_JUMP_LIMIT : PM_DE_PATH_CAP;
      if (NS > 0) {
#pragma unroll
        for (int j = 0; j < (NS > 0 ? NS : 1); j++) Racc[j] += (s == j) ? L : 0.0;
      } else atomicAdd(&s_dw[s], L);
      const double sc = s_scale_new[s];
      if (isfinite(sc) && sc > 0.0) {
        double tot = 0;
        for (;;) {
          const double g = A::mul(sc, exp_rand_R(gnew));
          const double t2 = A::add(tot, g);
          if (t2 < L) { tot = t2; newm++; if (newm > 70000) break; } else break;
        }
      }
      newm++;
      nout++;
    };

    double in_len[PM_LOCAL_PATH_MAX]; uint8_t in_st[PM_LOCAL_PATH_MAX];
    int nin = 0;
    if (!first) {
      nin = min(nj + 1, PM_LOCAL_PATH_MAX);
      for (int c = 0; c < nin; c++) { const int q = min(rd + c, cap_c - 1); in_len[c] = rd_len[q]; in_st[c] = rd_st[q]; }
      rd += nj + 1;
    }
    StreamD gold;  // the stream that drew the virtual jumps of the previous sweep (none before the first one)
    gold.open(P.rng, (uint32_t)site, first ? iter : iter - 1u, K_BREXP, (uint32_t)e, P.err_flag);
    StreamD gst; gst.open(P.rng, (uint32_t)site, iter, K_BRSTATE, (uint32_t)e, P.err_flag);
    int j = 0; double tot = 0; long long cp = first ? P.maps_off[e] : 0;
    auto next_piece = [&]() -> double {
      if (first) return P.maps_len[cp++];
      if (j >= nin) { errbits |= PM_DE_INCONSISTENT; return 0.0; }
      const double L = in_len[j];
      const double sc = s_scale_old[in_st[j]];
      if (isfinite(sc) && sc > 0.0) {
        const double g = A::mul(sc, exp_rand_R(gold));
        const double t2 = A::add(tot, g);
        if (t2 < L) { tot = t2; return g; }
      }
      const double r = A::sub(L, tot);
      j++; tot = 0;
      return r;
    };
    int cur_state = (m == 1) ? cs : ps;
    double cur_len = next_piece();
    int prev = cur_state;
    for (int p = 1; p < m; p++) {
      int st;
      if (p == m - 1) st = cs;
      else {
        const int jd = m - p - 1;  // beta_jd = Bs^jd e_cs: column cs of the host's power table (built bit for bit as the
                                   // reference's backward vectors), repeated mat-vecs beyond it
        double w[NC];
        if (jd < P.jcap) {
          const double* M = P.ppow + (size_t)jd * n * n;
#pragma unroll
          for (int c = 0; c < n; c++) w[c] = M[c * n + cs];
        } else {
#pragma unroll
          for (int c = 0; c < n; c++) w[c] = (double)(c == cs);
          for (int r = 0; r < jd; r++) matvec<double, NC, true>(sBs, n, w);
        }
#pragma unroll
        for (int c = 0; c < n; c++) w[c] = A::mul(sB[prev * n + c], w[c]);
        st = categorical<double, NC, true>(w, n, gst.next(), P.err_flag);
      }
      const double len = next_piece();
      if (full) atomicAdd(&s_cnt[prev * n + st], 1u);
      if (st == cur_state) cur_len = A::add(cur_len, len);
      else {
        emit(cur_len, cur_state);
        if (!full) atomicAdd(&s_cnt[cur_state * n + st], 1u);
        cur_state = st; cur_len = len;
      }
      prev = st;
    }
    emit(cur_len, cur_state);
    if (newm > 65535) { errbits |= PM_DE_M_OVERFLOW; newm = 65535; }
    if (nout > PM_LOCAL_PATH_MAX) nout = PM_LOCAL_PATH_MAX;  // flagged in emit
    P.meta[pe] = (uint32_t)newm | ((uint32_t)(nout - 1) << 16) | ((uint32_t)sfirst << 24);
  }
  if (errbits) atomicOr(P.err_flag, errbits);

  // block reduction: dwell times through a fixed-order shuffle tree + per-warp slots, counts through shared atomics
  if (NS > 0) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < (NS > 0 ? NS : 1); j++) {
      double v = Racc[j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
      if (lane == 0) s_dw[warp * n + j] = v;
    }
  }
  __syncthreads();
  const long long blk = (long long)blockIdx.y * gridDim.x + blockIdx.x;
  if ((int)threadIdx.x < n) {
    double v;
    if (NS > 0) { v = 0; for (int w = 0; w < (int)(blockDim.x >> 5); w++) v += s_dw[w * n + threadIdx.x]; }
    else v = s_dw[threadIdx.x];
    P.dw_partial[blk * n + threadIdx.x] = v;
  }
  for (int i = threadIdx.x; i < n * n; i += blockDim.x) if (s_cnt[i]) atomicAdd(&P.cnt[i], (unsigned long long)s_cnt[i]);
}

// ------------------------------------------------------------------------------------------------
// K2, production arithmetic, clade order (the top-down twin of k_prune_clade, same clades).  The root, then the nodes
// above the clades by depth, then every warp walks its clades alone in pre-order: a node's parent is either the node
// drawn just before (state in a register) or an ancestor drawn earlier by the same lane (one byte from L2, fetched one
// node ahead); the node's partial and jump count come through a cp.async ring 8 nodes deep.  One Philox block serves
// four consecutive nodes of a sequence.  Tips (ks / mt samplers) are redrawn at the end, four per Philox block.
//   slot: [0, PLB) partial per site   [PLB, +128) jump-count words   [+128, +144) v_off, parent_off (or -1: previous node)
//         [+144, +160) partial / jump-count offsets of the node that takes this slot next      (PLB = 32 * NS * sizeof(Real))
//   entry (host, 16 ints): pl_off, meta_off | v_off, parent_off | pad
// ------------------------------------------------------------------------------------------------
template <typename Real, int NS>
__device__ __forceinline__ int draw_node_state(const ChainParams<Real>& P, const Real* sBs, const Real* sPow, int npow_s, int k, int ps,
                                               const Real* pl, uint32_t word) {
  Real w[NS];
  if (k < npow_s) VecIO<Real, NS>::load(sPow + (k * NS + ps) * NS, NS, w);
  else if (k < P.jcap) {
#pragma unroll
    for (int j = 0; j < NS; j++) w[j] = P.ppow[(size_t)k * NS * NS + ps * NS + j];
  } else {
#pragma unroll
    for (int j = 0; j < NS; j++) w[j] = (Real)(j == ps);
    for (int r = 0; r < k; r++) matvec_t<Real, NS, false>(sBs, NS, w);
  }
#pragma unroll
  for (int j = 0; j < NS; j++) w[j] *= pl[j];
  // inverse-cdf draw, the same pick as categorical<.., false> for non-negative weights, without its per-state tests:
  // the first state whose running sum exceeds t is the number of running sums t has reached (a state of weight zero
  // repeats its predecessor's sum and cannot be the first)
  Real c[NS];
  c[0] = w[0];
#pragma unroll
  for (int j = 1; j < NS; j++) c[j] = c[j - 1] + w[j];
  const Real tot = c[NS - 1];
  if (!(tot > (Real)0) || !isfinite(tot)) { atomicOr(P.err_flag, tot > (Real)0 ? PM_DE_SAMPLE_NA : PM_DE_SAMPLE_ZERO); return 0; }
  const Real t = u01_from_word<Real>(word) * tot;
  int pick = 0;
#pragma unroll
  for (int j = 0; j < NS - 1; j++) pick += (t >= c[j]) ? 1 : 0;
  if (!(t < tot)) {  // rounding put t on the total: the last state with positive weight, as categorical does
#pragma unroll
    for (int j = 0; j < NS; j++) if (w[j] > (Real)0) pick = j;
  }
  return pick;
}

// The redraw of a tip of the hidden-rate samplers (ks / ksmt: the observed trait is the PARITY of the state, `code`): only
// the two states a = 1 - code and b = a + 2 carry weight, so the draw is between two entries of the row of P_k.  The same
// pick, bit for bit, as draw_node_state() with the 0/1 partial of tip_partial(): there the zero entries add nothing to
// the running sums (c = ra, ra, ra + rb, ra + rb for code 1; 0, ra, ra, ra + rb for code 0), t = u (ra + rb) falls below ra
// or not, and a t that rounding put on the total takes the last state with positive weight.
template <typename Real>
__device__ __forceinline__ int draw_parity_tip4(const ChainParams<Real>& P, const Real* sBs, const Real* sPow, int npow_s, int k, int ps,
                                                int code, uint32_t word) {
  Real w[4];
  if (k < npow_s) VecIO<Real, 4>::load(sPow + (k * 4 + ps) * 4, 4, w);
  else if (k < P.jcap) {
#pragma unroll
    for (int j = 0; j < 4; j++) w[j] = P.ppow[(size_t)k * 16 + ps * 4 + j];
  } else {
#pragma unroll
    for (int j = 0; j < 4; j++) w[j] = (Real)(j == ps);
    for (int r = 0; r < k; r++) matvec_t<Real, 4, false>(sBs, 4, w);
  }
  const Real ra = code ? w[0] : w[1], rb = code ? w[2] : w[3];
  const Real tot = ra + rb;
  if (!(tot > (Real)0) || !isfinite(tot)) { atomicOr(P.err_flag, tot > (Real)0 ? PM_DE_SAMPLE_NA : PM_DE_SAMPLE_ZERO); return 0; }
  const Real t = u01_from_word<Real>(word) * tot;
  const int a = 1 - code;
  int pick = (t < ra) ? a : a + 2;
  if (!(t < tot)) pick = (rb > (Real)0) ? a + 2 : a;
  return pick;
}
// a redrawn tip: the two-state draw above for parity tips of a 4-state model, the general draw otherwise
template <typename Real, int NS>
__device__ __forceinline__ int draw_tip_state(const ChainParams<Real>& P, const Real* sBs, const Real* sPow, int npow_s, int k, int ps, int code,
                                              bool parity, uint32_t word) {
  if (NS == 4 && parity) return draw_parity_tip4<Real>(P, sBs, sPow, npow_s, k, ps, code, word);
  Real pl[NS];
  tip_partial<Real, NS>(code, NS, parity, pl);
  return draw_node_state<Real, NS>(P, sBs, sPow, npow_s, k, ps, pl, word);
}

template <typename Real, int NS, int DEPTH>
__device__ __forceinline__ void nodes_clade_block(const ChainParams<Real>& P, const uint32_t iter, const long long site0, const long long pl0) {
  constexpr int PB = NS * (int)sizeof(Real);  // bytes of one partial
  constexpr int PLB = 32 * PB;
  constexpr int SLOT = PLB + 160;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Real* sBs = reinterpret_cast<Real*>(smem_raw + SLOT * 8 * DEPTH);
  Real* sVec = sBs + NS * NS;  // pid, scale_old, scale_new
  Real* sPow = sVec + 3 * NS;
  const int npow_s = min(PM_SMEM_POW, P.jcap);
  load_model_smem<Real>(P, NS, nullptr, sBs, sVec);
  for (int i = threadIdx.x; i < npow_s * NS * NS; i += blockDim.x) sPow[i] = P.ppow[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const long long S = P.S;
  const long long site_raw = site0 + lane;
  const bool active = site_raw < S;
  const long long site = active ? site_raw : S - 1;
  const long long lsite = pl0 + (site - site0);  // column of the site in the partials buffer
  const bool parity = P.parity_tips != 0;
  const int T = P.T;
  const uint32_t gsite = P.rng.site0 + (uint32_t)site;
  const uint32_t kslot = make_slot(K_NODEGRP, 0u);
  uint8_t* const nst = P.node_state + site;  // read and written by this thread
  if (warp == 0) {  // root :618-627
    Real w[NS], pl[NS];
    VecIO<Real, NS>::load(P.PL + ((long long)(P.root - T) * P.pl_S + lsite) * NS, NS, pl);
#pragma unroll
    for (int j = 0; j < NS; j++) w[j] = sVec[j] * pl[j];
    uint32_t o[4];
    philox4x32_10_rk(0xffffffffu, kslot, iter, gsite, P.rng.rk, o);
    const int s = categorical<Real, NS, false>(w, NS, u01_from_word<Real>(o[0]), P.err_flag);
    if (active) {
      nst[(long long)P.root * S] = (uint8_t)s;
      if (gsite == 0u) *P.root_out = s;
    }
  }
  __syncthreads();
  // ---- the nodes above the clades, by depth (a few hundred): one node per warp at a time, Philox block 0x80000000 + index
  for (int l = 0; l < P.n_cd_top_levels; l++) {
    const int beg = __ldg(P.cd_top_off + l), end = __ldg(P.cd_top_off + l + 1);
    for (int idx = beg + warp; idx < end; idx += nw) {
      const int4 en = __ldg(reinterpret_cast<const int4*>(P.cd_top) + idx);
      const int ps = nst[(long long)en.y * S];
      const int k = (int)(P.meta[(long long)en.z * S + site] & 0xffffu) - 1;
      Real pl[NS];
      VecIO<Real, NS>::load(P.PL + ((long long)(en.x - T) * P.pl_S + lsite) * NS, NS, pl);
      uint32_t o[4];
      philox4x32_10_rk(0x80000000u + (uint32_t)idx, kslot, iter, gsite, P.rng.rk, o);
      const int s = draw_node_state<Real, NS>(P, sBs, sPow, npow_s, k, ps, pl, o[0]);
      if (active) nst[(long long)en.x * S] = (uint8_t)s;
    }
    __syncthreads();
  }
  // ---- this warp's clades, pre-order ----
  {
    const int i0 = __ldg(P.cd_warp_off + warp), i1 = __ldg(P.cd_warp_off + warp + 1);
    unsigned ring = (unsigned)__cvta_generic_to_shared(smem_raw) + warp * (DEPTH * SLOT);
    asm volatile("" : "+r"(ring));  // kept in a register (see k_prune_clade)
    unsigned long long plb_u = reinterpret_cast<unsigned long long>(P.PL + lsite * NS),
                       mtb_u = reinterpret_cast<unsigned long long>(P.meta + site),
                       nsb_u = reinterpret_cast<unsigned long long>(nst);
    int act = active ? 1 : 0;
    unsigned lane4 = 4 * lane, lanePB = PB * lane;
    // lanes 0..3 copy the header words (entry words 4..7), lanes 4..7 the offsets of the node DEPTH further on (words 0..3)
    unsigned long long hsrc = lane < 4 ? 16 + 4 * lane : (unsigned long long)DEPTH * 64 + 4 * (lane - 4);
    unsigned hdst = PLB + 128 + 4 * lane;
    asm volatile("" : "+l"(plb_u), "+l"(mtb_u), "+l"(nsb_u), "+r"(act), "+r"(lane4), "+r"(lanePB), "+l"(hsrc), "+r"(hdst));
    auto off64 = [](int lo, int hi) { return (long long)(((unsigned long long)(unsigned)hi << 32) | (unsigned)lo); };
    const int4* ep = reinterpret_cast<const int4*>(P.cd_entries) + 4 * (long long)i0;
    auto issue = [&](unsigned slot, const int4* e, const int4& q0, bool more) {
      const char* src = reinterpret_cast<const char*>(plb_u) + off64(q0.x, q0.y);
      if (PB == 8) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(slot + lanePB), "l"(src) : "memory");
      else {
        cp_async16(slot + lanePB, src);
        if (PB == 32) cp_async16(slot + lanePB + 16, src + 16);
      }
      cp_async4(slot + PLB + lane4, reinterpret_cast<const char*>(mtb_u) + off64(q0.z, q0.w));
      if (lane < 8) cp_async4(slot + hdst, reinterpret_cast<const char*>(e) + hsrc, lane < 4 || more);
    };
#pragma unroll 1
    for (int u = 0; u < DEPTH; u++) {
      if (i0 + u < i1) { issue(ring + u * SLOT, ep, __ldg(ep), i0 + u + DEPTH < i1); ep += 4; }
      cp_async_commit();
    }
    long long vA = 0, vB = 0, pA = -1, pB = -1;  // node_state offsets of the node and of its parent (-1: previous node)
    int psA = 0, psB = 0;                       // parent state fetched from memory
    if (i0 < i1) {
      cp_async_wait<DEPTH - 1>();
      __syncwarp();
      const int4 h = lds_v4(ring + PLB + 128);
      vA = off64(h.x, h.y); pA = off64(h.z, h.w);
      if (pA >= 0) psA = *reinterpret_cast<const uint8_t*>(nsb_u + (unsigned long long)pA);
    }
    unsigned slot = ring;
    unsigned ring_end = ring + DEPTH * SLOT;
    asm volatile("" : "+r"(ring_end));
    int sprev = 0;
    uint32_t o[4] = {0, 0, 0, 0};
    auto step = [&](int idx, long long v_off, long long p_off, int ps_mem, long long& v_off_n, long long& p_off_n, int& ps_mem_n) {
      const unsigned slot_n = (slot + SLOT == ring_end) ? ring : slot + SLOT;
      cp_async_wait<DEPTH - 2>();
      __syncwarp();
      if (idx + 1 < i1) {
        const int4 h = lds_v4(slot_n + PLB + 128);
        v_off_n = off64(h.x, h.y); p_off_n = off64(h.z, h.w);
        // the parent of the next node, unless it is the node drawn now: stored at least one node ago by this lane
        if (h.w >= 0) ps_mem_n = *reinterpret_cast<const uint8_t*>(nsb_u + (unsigned long long)p_off_n);
      }
      if ((idx & 3) == 0 || idx == i0) philox4x32_10_rk((uint32_t)idx >> 2, kslot, iter, gsite, P.rng.rk, o);
      const uint32_t word = (idx & 3) == 0 ? o[0] : (idx & 3) == 1 ? o[1] : (idx & 3) == 2 ? o[2] : o[3];
      Real pl[NS];
      lds_vec<Real, NS>(slot + lanePB, pl);  // the partial of this node, copied by this lane
      const int k = lds_u16(slot + PLB + lane4) - 1;
      const int ps = p_off < 0 ? sprev : ps_mem;
      const int sn = draw_node_state<Real, NS>(P, sBs, sPow, npow_s, k, ps, pl, word);
      if (act) *reinterpret_cast<uint8_t*>(nsb_u + (unsigned long long)v_off) = (uint8_t)sn;
      sprev = sn;
      __syncwarp();
      if (idx + DEPTH < i1) {
        const int4 q0 = lds_v4(slot + PLB + 144);
        __syncwarp();
        issue(slot, ep, q0, idx + 2 * DEPTH < i1);
        ep += 4;
      }
      cp_async_commit();
      slot = slot_n;
    };
#pragma unroll 1
    for (int idx = i0; idx < i1; idx += 2) {
      step(idx, vA, pA, psA, vB, pB, psB);
      if (idx + 1 < i1) step(idx + 1, vB, pB, psB, vA, pA, psA);
    }
    cp_async_wait<0>();
  }
  // ---- tips (samplers that redraw them): four consecutive list entries share a Philox block 0x40000000 + group.  Software
  // pipeline: the twelve loads of a warp's NEXT group are in flight while it draws the current one.
  if (P.n_cd_tips > 0) {
    __syncthreads();
    const int ntip = P.n_cd_tips, ngrp = (ntip + 3) >> 2;
    const uint8_t* const tipb = P.tipcode + site;
    const char* const mtb = reinterpret_cast<const char*>(P.meta + site);
    struct TipLoad { int ps, k, cd; };
    auto load = [&](int grp, TipLoad (&L)[4]) {
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const int v = min(4 * grp + q, ntip - 1);
        const longlong2 en = __ldg(reinterpret_cast<const longlong2*>(P.cd_tips) + v);
        L[q].ps = nst[en.x];
        L[q].k = (int)(*reinterpret_cast<const uint32_t*>(mtb + en.y) & 0xffffu) - 1;
        L[q].cd = tipb[(long long)v * P.TS];
      }
    };
    auto draw = [&](int grp, const TipLoad (&L)[4]) {
      uint32_t o[4];
      philox4x32_10_rk(0x40000000u + (uint32_t)grp, kslot, iter, gsite, P.rng.rk, o);
#pragma unroll
      for (int q = 0; q < 4; q++) {
        if (4 * grp + q < ntip) {  // warp-uniform
          const uint32_t word = q == 0 ? o[0] : q == 1 ? o[1] : q == 2 ? o[2] : o[3];
          const int sn = draw_tip_state<Real, NS>(P, sBs, sPow, npow_s, L[q].k, L[q].ps, L[q].cd, parity, word);
          if (active) nst[(long long)(4 * grp + q) * S] = (uint8_t)sn;
        }
      }
    };
    TipLoad A[4], B[4];
    int grp = warp;
    if (grp < ngrp) load(grp, A);
    while (grp < ngrp) {
      if (grp + nw < ngrp) load(grp + nw, B);
      draw(grp, A);
      grp += nw;
      if (grp >= ngrp) break;
      if (grp + nw < ngrp) load(grp + nw, A);
      draw(grp, B);
      grp += nw;
    }
  }
}

template <typename Real, int NS, int DEPTH, int MINB>
__global__ void __launch_bounds__(256, MINB) k_nodes_clade(ChainParams<Real> P, uint32_t iter) {
  if (P.ctl) iter = P.ctl[0];
  nodes_clade_block<Real, NS, DEPTH>(P, iter, P.tile_base + (long long)blockIdx.x * 32, (long long)blockIdx.x * 32);
}

// ------------------------------------------------------------------------------------------------
// K1 + K2 fused (production, n = 2 / 4).  A block's partials are read by nobody but the same block's node draws, so a
// block prunes its 32 sites and draws their node states straight away.  The partials of the whole sweep then live in one
// SLOT of 32 sites per block that is RESIDENT at a time -- slots_per_sm per SM, claimed at block start and released at
// block end (a block keeps its SM) -- (T - 1) x 32 x n reals per slot: 2.3 GB at 10 000 tips instead of 20 GB for
// 125 000 sites, and the two passes share one launch with no tail between them.  The schedules' byte offsets are built
// for a row of 32 x slots sites (ChainParams::pl_S).
//   phases: 1 = prune only (timing, partials read-back), 3 = both.   phase_ns (optional): block-time spent in each pass.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long global_ns() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ unsigned sm_id() { unsigned v; asm volatile("mov.u32 %0, %%smid;" : "=r"(v)); return v; }

template <typename Real, int NS, int DEPTH, int MINB>
__global__ void __launch_bounds__(256, MINB) k_prune_nodes_clade(ChainParams<Real> P, uint32_t iter, long long b0, int phases, int* slot_busy,
                                                                 int slots_per_sm, unsigned long long* phase_ns) {
  if (P.ctl) iter = P.ctl[0];
  __shared__ unsigned long long s_t[2];
  __shared__ int s_slot;
  if (threadIdx.x == 0) {
    // claim a slot of this SM: at most slots_per_sm blocks are resident on it (occupancy), and a block that leaves has
    // released its slot before the next one can start here
    // (slot_busy == nullptr: slot = block index, for a launch of at most as many blocks as there are slots)
    int slot = (int)blockIdx.x;
    if (slot_busy) {
      const int base = (int)sm_id() * slots_per_sm;
      int k = 0;
      while (atomicCAS(slot_busy + base + k, 0, 1) != 0) k = (k + 1 == slots_per_sm) ? 0 : k + 1;
      slot = base + k;
    }
    s_slot = slot;
    if (phase_ns) s_t[0] = global_ns();
  }
  __syncthreads();
  const int slot = s_slot;
  const long long site0 = (b0 + blockIdx.x) * 32, pl0 = (long long)slot * 32;
  prune_clade_block<Real, NS, DEPTH>(P, site0, pl0);
  __syncthreads();  // every partial of these sites is written (and visible to the block) before the draws read them
  if (phases & 2) {
    if (phase_ns && threadIdx.x == 0) s_t[1] = global_ns();
    nodes_clade_block<Real, NS, DEPTH>(P, iter, site0, pl0);
    __syncthreads();
    if (phase_ns && threadIdx.x == 0) {
      const unsigned long long t2 = global_ns();
      atomicAdd(phase_ns, s_t[1] - s_t[0]);
      atomicAdd(phase_ns + 1, t2 - s_t[1]);
    }
  }
  if (threadIdx.x == 0 && slot_busy) atomicExch(slot_busy + slot, 0);  // (after a barrier: nobody reads the slot any more)
}

// ------------------------------------------------------------------------------------------------
// K3, production arithmetic: two kernels (virtual-jump model: see pm_device.cuh).
//
// State a sweep leaves per (branch, site):  meta = m (bits 0-15) | real jumps nj (16-21) | state of run 0 (22-26) |
// state of run 1 (27-31);  pos1 = length of the first piece when m == 2 or nj == 1 (the position of the only jump point,
// respectively of the only real jump);  paths with nj >= 2 (a fraction of a percent) keep all their runs as records and
// pos1 holds their offset in the site's record slice; nj = 63 stands for "63 or more": such a path starts with a header
// record holding its run count.  The first sweep finds m and (for two-piece maps) pos1 seeded from the caller's maps.
//
//   k_paths_easy  every branch whose previous path has at most one jump point (m <= 2: ~98 % here).  No
//                 regeneration and no record is needed: the pieces are (pos1, t - pos1), the new states are the two
//                 node states, the new virtual-jump counts take one uniform per run from a Philox block shared by two
//                 branches.  Coalesced streaming over the chunk, straight-line code; everything else gets a bit in the
//                 branch-major ballot array (one warp vote and one 4-byte store per warp and branch).
//   k_paths_hard  persistent warps over branch-major work items (a run of ballot words of ONE branch, sized on the host to
//                 ~100 set bits).  A warp turns the set bits into (site, branch) items, reads their meta word and sorts
//                 them into two per-warp shared-memory queues; whenever a queue holds 32 items they are processed, one per
//                 lane: [short] three pieces with at most one real jump (~3/4 of the items here) by straight-line code,
//                 [general] everything else: regenerate the virtual jumps of the previous sweep run by run, redraw the
//                 interior states (resamplebranchstates :264-308), merge and count (shortener :44-73 / shortenerbf
//                 :997-1028), draw the new counts; a path too long for the local buffer is walked a second time to write
//                 its records in place.  No block barrier; lanes of a round run the same code on items of like shape.
// ------------------------------------------------------------------------------------------------
#define PM_META(m, q) ((uint32_t)(m) | ((uint32_t)(q) << 16))

template <typename Real>
__device__ __forceinline__ bool rate_ok(Real r) { return isfinite(r) && r > (Real)0; }

__device__ __forceinline__ float lds_real(unsigned a, float) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v; }
__device__ __forceinline__ double lds_real(unsigned a, double) { double v; asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a)); return v; }
__device__ __forceinline__ unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

// Shared-memory layout of k_paths_easy, in bytes from the start of the dynamic window (offsets up to topo multiples of 16):
//   [0, dw) dwell partials [4 warps][n] f64 | cnt: transition counters [n*n] u32 | rate [n] | acc: every thread's dwell
//   sums, [NS][128 threads] of Real (the current stretch of 32 branch pairs), then [NS][128] of f64 (the flushed
//   stretches; NS > 0 only) | topo: the chunk's topology, parent and child node (int2) per branch | len: its branch lengths
// With a compile-time state count every offset but the entry index is an immediate, so the kernel keeps ONE base address
// in a register (formed from several pointers, the compiler rebuilds the shared window base at every use: ~10 % of the
// loop's instructions).
template <typename Real, int NS>
struct EasySmem {
  int cnt, rate, acc, sum, topo;
  __host__ __device__ static int up16(int x) { return (x + 15) & ~15; }
  __host__ __device__ explicit EasySmem(int n) {
    cnt = up16(4 * n * (int)sizeof(double));
    rate = up16(cnt + n * n * (int)sizeof(unsigned));
    acc = up16(rate + n * (int)sizeof(Real));
    sum = acc + (NS > 0 ? NS * 128 * (int)sizeof(Real) : 0);
    topo = sum + (NS > 0 ? NS * 128 * (int)sizeof(double) : 0);
  }
  __host__ __device__ int len(int chunk) const { return topo + chunk * 8; }
  __host__ __device__ size_t bytes(int chunk) const { return (size_t)len(chunk) + (size_t)chunk * sizeof(Real); }
};
__device__ __forceinline__ void lds_v2s32(unsigned a, int& x, int& y) { asm volatile("ld.shared.v2.s32 {%0,%1}, [%2];" : "=r"(x), "=r"(y) : "r"(a)); }
// Predicated forms (one set-predicate, then @p instructions): guarded by an `if`, the compiler branches around them.
__device__ __forceinline__ void red_shared_inc_if(bool p, unsigned a) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %1, 0;\n\t@q red.shared.add.u32 [%0], 1;\n\t}" ::"r"(a), "r"((unsigned)p) : "memory");
}
// *a += x in shared memory, rounded once (the same bits as a register sum: fma(1, x, s) = s + x)
__device__ __forceinline__ void sts_add_if(bool p, unsigned a, float x) {
  asm volatile("{\n\t.reg .pred q;\n\t.reg .f32 v;\n\tsetp.ne.b32 q, %2, 0;\n\t@q ld.shared.f32 v, [%0];\n\t@q add.rn.f32 v, v, %1;\n\t"
               "@q st.shared.f32 [%0], v;\n\t}" ::"r"(a), "f"(x), "r"((unsigned)p));
}
__device__ __forceinline__ void sts_add_if(bool p, unsigned a, double x) {
  asm volatile("{\n\t.reg .pred q;\n\t.reg .f64 v;\n\tsetp.ne.b32 q, %2, 0;\n\t@q ld.shared.f64 v, [%0];\n\t@q add.rn.f64 v, v, %1;\n\t"
               "@q st.shared.f64 [%0], v;\n\t}" ::"r"(a), "d"(x), "r"((unsigned)p));
}
__device__ __forceinline__ void sts_real(unsigned a, float x) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(x)); }
__device__ __forceinline__ void sts_real(unsigned a, double x) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(x)); }
// global loads and stores through pointers the kernel keeps in registers (asm outputs): the compiler no longer knows
// they point to global memory and would emit generic accesses
__device__ __forceinline__ uint32_t ldg_u32(const uint32_t* a) { uint32_t v; asm volatile("ld.global.u32 %0, [%1];" : "=r"(v) : "l"(a)); return v; }
__device__ __forceinline__ int ldg_u8(const uint8_t* a) { uint32_t v; asm volatile("ld.global.u8 %0, [%1];" : "=r"(v) : "l"(a)); return (int)v; }
__device__ __forceinline__ void stg_u32_if(bool p, uint32_t* a, uint32_t x) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q st.global.u32 [%0], %1;\n\t}" ::"l"(a), "r"(x), "r"((unsigned)p));
}
__device__ __forceinline__ void stg_u16_if(bool p, uint16_t* a, uint16_t x) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q st.global.u16 [%0], %1;\n\t}" ::"l"(a), "h"(x), "r"((unsigned)p));
}

template <typename Real, int NS>
__global__ void __launch_bounds__(128, (sizeof(Real) == 8 ? 6 : 8)) k_paths_easy(ChainParams<Real> P, uint32_t iter, int chunk) {
  if (P.ctl) iter = P.ctl[0];
  constexpr int NR = NS > 0 ? NS : 1;
  typedef Pin<Real> PN;
  const int n = NS > 0 ? NS : P.n;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const EasySmem<Real, NS> lay(n);
  double* s_dw = reinterpret_cast<double*>(smem_raw);                       // [4 warps][n] (NS>0) or [n] atomics (NS==0)
  unsigned* s_cnt = reinterpret_cast<unsigned*>(smem_raw + lay.cnt);       // [n*n] (a copy per warp was tried: +2 % time)
  Real* s_rate = reinterpret_cast<Real*>(smem_raw + lay.rate);             // [n] Omega + Q_ss of this sweep
  // dwell of state s: the thread's running sum acc[s][thread] += L in shared memory (address = state * 128 * sizeof(Real)
  // + the thread's own column: conflict-free, one load / add / store per run, skipped where the lane has nothing to add);
  // every 32 branch pairs it is added to sum[s][thread] in double.  Neither takes registers in the loop.
  Real* s_acc = reinterpret_cast<Real*>(smem_raw + lay.acc);               // [NS][128]
  double* s_sum = reinterpret_cast<double*>(smem_raw + lay.sum);           // [NS][128]
  // topology of the chunk (the same for every thread of the block): parent / child node and branch length per branch
  int2* s_topo = reinterpret_cast<int2*>(smem_raw + lay.topo);
  Real* s_len = reinterpret_cast<Real*>(smem_raw + lay.len(chunk));
  const int e0 = blockIdx.y * chunk, e1 = min(P.E, e0 + chunk);
  for (int i = threadIdx.x; i < n * n; i += blockDim.x) s_cnt[i] = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {  // a state without a valid rate draws no virtual jumps
    const Real r = P.model[2 * n * n + 4 * n + i];
    s_rate[i] = rate_ok(r) ? r : (Real)0;
  }
  for (int i = threadIdx.x; i < 4 * n; i += blockDim.x) s_dw[i] = 0.0;
  if (NS > 0) for (int j = 0; j < NS; j++) { s_acc[j * 128 + threadIdx.x] = 0; s_sum[j * 128 + threadIdx.x] = 0.0; }
  for (int i = threadIdx.x; i < e1 - e0; i += blockDim.x) {
    s_topo[i] = make_int2(P.e_parent[e0 + i], P.e_child[e0 + i]);
    s_len[i] = P.e_len[e0 + i];
  }
  __syncthreads();
  // ONE 32-bit shared-memory base, kept in a register; everything else is base + immediate (+ scaled index)
  unsigned a_base = smem_addr(smem_raw);
  asm volatile("" : "+r"(a_base));
  const unsigned a_cnt = a_base + (unsigned)lay.cnt, a_rate = a_base + (unsigned)lay.rate, a_topo = a_base + (unsigned)lay.topo,
                 a_len = a_base + (unsigned)lay.len(chunk);
  const unsigned a_acc = a_base + (unsigned)lay.acc + (unsigned)sizeof(Real) * threadIdx.x,
                 a_sum = a_base + (unsigned)lay.sum + (unsigned)sizeof(double) * threadIdx.x;
  const long long S = P.S;
  uint32_t Su = (uint32_t)S;  // S < 2^31 (checked by the host): 32 x 32 -> 64-bit offsets are one instruction
  const long long site_raw = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long site = site_raw < S ? site_raw : S - 1;
  const bool full = P.full_counts != 0;
  const long long wglob = site_raw >> 5;  // ballot word of this warp (the same for its 32 lanes)
  // Rows of the chunk are addressed as base + 32-bit element index (the host keeps chunk x S below 2^32): one wide
  // multiply-add per access and one add per branch, instead of a 64-bit pointer bump per array
  uint32_t* __restrict__ bal_b = P.hard_ballot + (long long)e0 * P.W + wglob;
  unsigned bal_writer = (threadIdx.x & 31) == 0 && wglob < (long long)P.W;
  uint32_t Wu = (uint32_t)P.W;
  uint32_t* __restrict__ meta_b = P.meta + (long long)e0 * S + site;   // row i of the chunk: meta_b[i * S]
  uint16_t* __restrict__ shape_b = P.shape + (long long)e0 * S + site;
  uint32_t row = 0, rowf = 0, rowb = 0;  // i * S of the store cursor and of the fetch cursor, i * W of the ballot cursor
  const uint8_t* __restrict__ nstate = P.node_state + site;
  // kept in registers for the whole loop (left to itself, the compiler reloads them from the parameter bank and redoes
  // the 64-bit additions at every use; the FP64 kernel has no registers to spare for them: it would spill)
  if (sizeof(Real) == 4) asm volatile("" : "+l"(bal_b), "+l"(meta_b), "+l"(shape_b), "+l"(nstate), "+r"(Wu), "+r"(Su), "+r"(bal_writer));
  auto add_dwell = [&](int s, Real L, bool p) {
    if (NS > 0) sts_add_if(p, a_acc + (unsigned)s * (unsigned)(128 * sizeof(Real)), L);
    else if (p && L != (Real)0) atomicAdd(&s_dw[s], (double)L);
  };
  auto flush_dwell = [&]() {
    if (NS > 0) {
#pragma unroll
      for (int j = 0; j < NR; j++) {
        const unsigned a = a_acc + (unsigned)j * (unsigned)(128 * sizeof(Real)), b = a_sum + (unsigned)j * (128u * 8u);
        sts_real(b, lds_real(b, 0.0) + (double)lds_real(a, (Real)0));
        sts_real(a, (Real)0);
      }
    }
  };
  // Software pipeline over pairs of branches (2j, 2j + 1: they share a Philox block): at the top of a trip the state
  // words and node states of the NEXT pair are requested (three independent loads per branch: the position of a lone
  // jump point travels inside the state word), so no load is waited for inside a trip.
  const int nb = e1 - e0;
  struct Ahead { uint32_t mt; int ps, cs; };
  Ahead X = {0, 0, 0}, Y = {0, 0, 0};
  auto fetch = [&](int i, Ahead& a) {
    a.mt = ldg_u32(meta_b + rowf); rowf += Su;
    int par, chi;
    lds_v2s32(a_topo + 8u * (unsigned)i, par, chi);
    a.ps = ldg_u8(nstate + (uint64_t)(uint32_t)par * Su);
    a.cs = ldg_u8(nstate + (uint64_t)(uint32_t)chi * Su);
  };
  uint32_t po[4] = {0, 0, 0, 0};
  const PairBlocks pb(P.rng, iter);
  const uint32_t gsite = P.rng.site0 + (uint32_t)site;
  // one branch, from what was fetched for it.  ODD: second branch of its Philox pair (the block was drawn by the first,
  // unless NEWBLK: it opens the chunk).  TAIL: the block may hold sites past the end.  Straight-line code: lanes that
  // leave their branch to the general kernels compute along and contribute zeros; only the stores are predicated.
  auto body = [&](int i, auto odd_c, auto newblk_c, auto tail_c, const Ahead cur) {
    constexpr bool ODD = decltype(odd_c)::value, NEWBLK = decltype(newblk_c)::value, TAIL = decltype(tail_c)::value;
    const int e = e0 + i;
    const uint32_t mt = cur.mt; const int ps = cur.ps, cs = cur.cs;
    if (NEWBLK) pb.block(P.rng, (uint32_t)e >> 1, gsite, po);
    const uint32_t wA = ODD ? po[2] : po[0], wB = ODD ? po[3] : po[1];
    const int m = (int)(mt & 0xffffu);
    const uint32_t q = mt >> 16;
    const Real Le = lds_real(a_len + (unsigned)sizeof(Real) * (unsigned)i, (Real)0);
    // pieces: (Le) or (p1, Le - p1); states ps | cs (a one-piece branch carries the child state, :460-475).  The
    // virtual jumps of a two-run path are counted together: K ~ Poisson(lam0 + lam1) from the A word (their positions,
    // if a later sweep needs them, are regenerated by the general kernels, see RunPieces)
    const bool two = (m == 2) && (ps != cs);
    const Real p1 = pos_dec<Real>(q, Le);
    const Real L0 = two ? p1 : Le;
    const int s0 = two ? ps : cs;
    const Real L1 = two ? PN::sub(Le, p1) : (Real)0;
    // rates are clamped to >= 0 when staged; x + 0 = x: a single run has lam = rate * t_e exactly
    const Real lam = PN::add(PN::mul(lds_real(a_rate + (unsigned)sizeof(Real) * (unsigned)s0, (Real)0), L0),
                             PN::mul(lds_real(a_rate + (unsigned)sizeof(Real) * (unsigned)cs, (Real)0), L1));
    const bool hard = (m > 2) || lam > (Real)PM_LAMBDA_INV;
    const bool ok = TAIL ? (!hard && site_raw < S) : !hard;
    const int k = poisson_inv<Real>(lam, wA);
    red_shared_inc_if(ok && m == 2 && (full || two), a_cnt + 4u * (unsigned)(ps * n + cs));
    add_dwell(s0, L0, ok);
    add_dwell(cs, L1, ok && two);  // (a single run adds nothing here)
    // a path that ends up with a single jump point keeps that point in the state word: the real jump stays where it
    // was; a lone new virtual jump is uniform on the branch -- its 16-bit position comes from the B word
    const uint32_t newq = (!two && k == 1) ? pos_rand(wB) : q;
    stg_u32_if(ok, meta_b + row, (newq << 16) + (uint32_t)((two ? 2 : 1) + k));  // = PM_META (k <= 64)
    stg_u16_if(ok, shape_b + row, (uint16_t)(((uint32_t)cs << 11) + ((uint32_t)s0 << 6) + (two ? 1u : 0u)));  // = PM_SHAPE
    row += Su;
    const unsigned bal = __ballot_sync(0xffffffffu, TAIL ? (hard && site_raw < S) : hard);
    stg_u32_if(bal_writer != 0, bal_b + rowb, bal);
    rowb += Wu;
  };
  auto run = [&](auto tail_c) {
    const std::true_type T{}; const std::false_type F{};
    int i = 0;
    if (nb > 0 && (e0 & 1)) {  // the chunk opens on the second branch of a pair: on its own, unpipelined
      fetch(0, X);
      body(0, T, T, tail_c, X);
      i = 1;
    }
    if (i < nb) fetch(i, X);
    if (i + 1 < nb) fetch(i + 1, Y);
    while (i + 3 < nb) {  // 32 pairs, then the FP32 dwell sums of the stretch go to the double accumulators
      const int stop = min(nb - 4, i + 62);
      for (; i <= stop; i += 2) {
        const Ahead cx = X, cy = Y;
        fetch(i + 2, X); fetch(i + 3, Y);
        body(i, F, T, tail_c, cx);
        body(i + 1, T, F, tail_c, cy);
      }
      flush_dwell();
    }
    for (; i + 1 < nb; i += 2) {  // the last pair(s): nothing, or not everything, left to prefetch
      const Ahead cx = X, cy = Y;
      if (i + 2 < nb) fetch(i + 2, X);
      if (i + 3 < nb) fetch(i + 3, Y);
      body(i, F, T, tail_c, cx);
      body(i + 1, T, F, tail_c, cy);
    }
    if (i < nb) body(i, F, T, tail_c, X);
    flush_dwell();
  };
  if ((long long)(blockIdx.x + 1) * blockDim.x <= S) run(std::false_type()); else run(std::true_type());
  if (NS > 0) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < NR; j++) {
      double v = lds_real(a_sum + (unsigned)j * (128u * 8u), 0.0);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
      if (lane == 0) s_dw[warp * n + j] = v;
    }
  }
  __syncthreads();
  const long long blk = (long long)blockIdx.y * gridDim.x + blockIdx.x;
  if ((int)threadIdx.x < n) {
    double v;
    if (NS > 0) { v = 0; for (int w = 0; w < (int)(blockDim.x >> 5); w++) v += s_dw[w * n + threadIdx.x]; }
    else v = s_dw[threadIdx.x];
    P.dw_partial[blk * n + threadIdx.x] = v;
  }
  for (int i = threadIdx.x; i < n * n; i += blockDim.x) if (s_cnt[i]) atomicAdd(&P.cnt[i], (unsigned long long)s_cnt[i]);
}

// rate of the virtual jumps in a state, 0 where the model has none (a state without a valid rate draws no virtual jumps)
template <typename Real>
__device__ __forceinline__ Real rate_or_zero(Real r) { return rate_ok(r) ? r : (Real)0; }

// The pieces of one run of the previous path, in order (regenerated, never stored).
// Joint mode: a two-run path (one real jump, at p1) whose virtual jumps were COUNTED TOGETHER -- K ~ Poisson(lam0 + lam1)
// from one uniform (pm_device.cuh).  Their positions are K independent draws from the piecewise-constant intensity,
// generated in increasing order: order statistics v_1 < ... < v_K of uniforms on (0, 1), v < q = lam0 / (lam0 + lam1)
// falls on run 0 at v * (lamT / r0), the rest on run 1 at (v - q) * (lamT / r1) past the real jump.  By the splitting
// property of the Poisson process this is the law of two independent Poisson(lam_i) sets of uniform positions.
template <typename Real>
struct RunPieces {
  Real L, x, rate;  // joint mode: `rate` holds q, the share of run 0 in the branch's intensity
  int left;       // count mode: jumps not yet emitted
  bool gaps;      // lambda > PM_LAMBDA_INV
  bool firstB;    // the first position uniform is the pair block's B word (single-run path, joint two-run path)
  uint32_t wB;
  WordStream ws;  // positions (count mode) or gaps
  bool joint, pend, run0;
  Real v, sc;     // joint mode: last order statistic drawn on (0, 1); branch length per unit of v on the current run
  __device__ __forceinline__ void begin(const RngDesc& d, uint32_t site, uint32_t it, uint32_t e, int run, Real len, Real r,
                                       uint32_t cnt_word, bool single_run, uint32_t wordB) {
    L = len; x = 0; rate = r; left = 0; gaps = false; firstB = single_run; wB = wordB; joint = false;
    if (!rate_ok(r)) return;
    const Real lam = Pin<Real>::mul(r, len);
    if (lam > (Real)PM_LAMBDA_INV) { gaps = true; ws.open(d, site, it, K_BRGAP, e, (uint32_t)run); }
    else { left = poisson_inv<Real>(lam, cnt_word); ws.open(d, site, it, K_BRPOS, e, (uint32_t)run); }
  }
  // joint mode, run 0 of length len0 and (clamped) rate r0; K virtual jumps on the whole branch
  __device__ __forceinline__ void begin_joint(const RngDesc& d, uint32_t site, uint32_t it, uint32_t e, Real len0, int K, Real lam0,
                                             Real lamT, Real r0, uint32_t wordB) {
    typedef Pin<Real> PN;
    L = len0; x = 0; left = K; gaps = false; firstB = true; wB = wordB; joint = true; pend = false; run0 = true;
    v = 0; rate = PN::div(lam0, lamT); sc = PN::div(lamT, r0);
    ws.open(d, site, it, K_BRPOS, e, 0u);
  }
  __device__ __forceinline__ void second_run(Real len1, Real lamT, Real r1) { L = len1; x = 0; run0 = false; sc = Pin<Real>::div(lamT, r1); }
  // returns the next piece; `last` tells whether it closes the run
  __device__ __forceinline__ Real next(bool& last) {
    typedef Pin<Real> PN;
    if (joint) {
      if (!pend && left > 0) {
        uint32_t w;
        if (firstB) { w = wB; firstB = false; } else w = ws.next();
        v = next_order_stat<Real>(v, (Real)1, left, w);
        left--; pend = true;
      }
      if (pend && (!run0 || v < rate)) {
        const Real t2 = min(PN::mul(run0 ? v : PN::sub(v, rate), sc), L);
        const Real piece = max(PN::sub(t2, x), (Real)0);
        x = max(t2, x); pend = false; last = false;
        return piece;
      }
      last = true;
      return PN::sub(L, x);
    }
    if (gaps) {
      const Real g = PN::div(PN::neglog(PN::u01(ws.next())), rate);
      const Real t2 = PN::add(x, g);
      if (t2 < L) { x = t2; last = false; return g; }
      last = true;
      return PN::sub(L, x);
    }
    if (left > 0) {
      uint32_t w;
      if (firstB) { w = wB; firstB = false; } else w = ws.next();
      const Real t2 = next_order_stat<Real>(x, L, left, w);
      const Real piece = PN::sub(t2, x);
      x = t2; left--; last = false;
      return piece;
    }
    last = true;
    return PN::sub(L, x);
  }
};

// number of exponential gaps of the given rate that fit into a run of length L (a run too long for the count mode);
// *first = the first gap.  Rare: kept out of line.
template <typename Real>
__device__ __noinline__ int count_gaps(RngDesc d, uint32_t site, uint32_t it, uint32_t e, uint32_t run, Real L, Real rate, Real* first) {
  typedef Pin<Real> PN;
  WordStream g; g.open(d, site, it, K_BRGAP, e, run);
  Real x = 0; int k = 0;
  for (;;) {
    const Real gp = PN::div(PN::neglog(PN::u01(g.next())), rate);
    const Real t2 = PN::add(x, gp);
    if (!(t2 < L) || k > 70000) break;
    x = t2; k++;
    if (k == 1) *first = gp;
  }
  return k;
}

// One (site, branch) item of the general path kernel, as queued per warp: everything the item reads from the sweep's
// state is fetched when it is queued (four independent loads per lane in flight), so that processing it later waits
// for no memory.
template <typename Real>
struct HardItem { uint32_t site, e, meta, ends, shape; };  // ends = parent state | child state << 8

// The two item routines of the general path kernels, as methods of a per-thread context (so that the persistent kernels
// below and the one-block-per-site chain kernel of small trees, pm_small.cuh, run the SAME code on an item).  They return
// the item's new state word and shape word; the caller stores them.
template <typename Real, int NS>
struct PathWorker {
  static constexpr int NC = NS > 0 ? NS : PM_NMAX;
  static constexpr int NR = NS > 0 ? NS : 1;
  typedef typename StreamSel<Real, false>::type Stream;
  typedef Pin<Real> PN;
  const ChainParams<Real>& P;
  const uint32_t iter; const int first; const int n; const bool full;
  const Real* const sB; const Real* const sBs; const Real* const sPow; const int npow_s;
  unsigned* const s_cnt; double* const s_dw;
  const Real* const s_rate_old; const Real* const s_rate_new;
  const Real* __restrict__ rd_len; const uint8_t* __restrict__ rd_st;
  Real* __restrict__ wr_len; uint8_t* __restrict__ wr_st;
  double Rsum[NR];
  unsigned errbits;
  __device__ __forceinline__ PathWorker(const ChainParams<Real>& P_, uint32_t iter_, int first_, int n_, const Real* sB_, const Real* sBs_,
                                        const Real* sPow_, int npow_s_, unsigned* s_cnt_, double* s_dw_, const Real* rate_old_,
                                        const Real* rate_new_)
      : P(P_), iter(iter_), first(first_), n(n_), full(P_.full_counts != 0), sB(sB_), sBs(sBs_), sPow(sPow_), npow_s(npow_s_),
        s_cnt(s_cnt_), s_dw(s_dw_), s_rate_old(rate_old_), s_rate_new(rate_new_), rd_len(P_.rec_len[(iter_ & 1u) ^ 1u]),
        rd_st(P_.rec_st[(iter_ & 1u) ^ 1u]), wr_len(P_.rec_len[iter_ & 1u]), wr_st(P_.rec_st[iter_ & 1u]), errbits(0) {
#pragma unroll
    for (int j = 0; j < NR; j++) Rsum[j] = 0;
  }
  __device__ __forceinline__ void add_dwell(int s, Real L) {
    if (NS > 0) {
#pragma unroll
      for (int j = 0; j < NR; j++) Rsum[j] += (s == j) ? (double)L : 0.0;
    } else atomicAdd(&s_dw[s], (double)L);
  }

  // ---- the common short shapes: three or four pieces (two or three jump points), at most one of them a real jump, every
  // run in count mode.  Unrolled, register-only restatement of what the general code below does for such an item: same
  // streams, same words, same pinned arithmetic, so a path may be written by one and regenerated by the other.
  __device__ __forceinline__ void short_item(const HardItem<Real> it, uint32_t& meta_out, uint16_t& shape_out) {
    const long long site = it.site;
    const int eb = (int)it.e;
    const uint32_t mt = it.meta;
    const int m = (int)(mt & 0xffffu);  // 3 or 4
    const int nj = (int)(it.shape & 0x3fu);
    const int so0 = (int)((it.shape >> 6) & 0x1fu), so1 = (int)((it.shape >> 11) & 0x1fu);
    const int ps = (int)(it.ends & 0xffu), cs = (int)(it.ends >> 8);
    const Real Le = __ldg(P.e_len + eb);
    const uint32_t gsite = P.rng.site0 + (uint32_t)site;
    uint32_t po_old[4], po_new[4];
    pair_block(P.rng, (uint32_t)site, iter, (uint32_t)eb, po_new);
    if (nj < 2) pair_block(P.rng, (uint32_t)site, iter - 1u, (uint32_t)eb, po_old);
    const uint32_t nA = (eb & 1) ? po_new[2] : po_new[0], nB = (eb & 1) ? po_new[3] : po_new[1];
    // ---- the m - 1 jump points of the previous path, in order.  nj <= 1: K = m - 1 - nj virtual ones (one to three) and,
    // if nj == 1, the real one at p1.  The virtual ones are order statistics of K uniforms on (0, 1) -- words: the pair
    // block's B, then the (K_BRPOS, e; run 0) block -- mapped through the inverse of the normalised intensity: all of
    // (0, 1) onto the single run, or (0, q) onto run 0 and (q, 1) onto run 1 (joint count, see RunPieces).
    // nj == m - 1 (two or three real jumps, no virtual one): the path's records.
    Real J0, J1, J2;
    if (nj >= 2) {
      const int ck = eb / P.chunk;
      const int cap0 = __ldg(P.cap_off + ck), cap_c = __ldg(P.cap_off + ck + 1) - cap0;
      const long long sl = ((long long)cap0 * P.rec_groups) + (site >> P.rec_shift) * (long long)cap_c;
      const int rd0 = (int)(mt >> 16);
      J0 = rd_len[sl + min(rd0, cap_c - 1)];
      J1 = PN::add(J0, rd_len[sl + min(rd0 + 1, cap_c - 1)]);
      J2 = m == 4 ? PN::add(J1, rd_len[sl + min(rd0 + 2, cap_c - 1)]) : J1;
    } else {
      const int K = m - 1 - nj;
      const Real p1 = nj == 0 ? Le : pos_dec<Real>(mt >> 16, Le);          // length of run 0
      const Real L1r = PN::sub(Le, p1);              // length of run 1 (nj == 1)
      Real qq = (Real)2, sc0 = Le, sc1 = 0;
      if (nj == 1) {
        const Real ro0 = rate_or_zero(s_rate_old[so0]), ro1 = rate_or_zero(s_rate_old[so1]);
        const Real lam0 = PN::mul(ro0, p1), lamT = PN::add(lam0, PN::mul(ro1, L1r));
        qq = PN::div(lam0, lamT); sc0 = PN::div(lamT, ro0); sc1 = PN::div(lamT, ro1);
      }
      const uint32_t oB = (eb & 1) ? po_old[3] : po_old[1];
      uint32_t pw[4] = {0, 0, 0, 0};
      if (K > 1) philox4x32_10(0u, make_slot(K_BRPOS, (uint32_t)eb), iter - 1u, gsite, P.rng.k0, P.rng.k1, pw);
      Real vt0 = 0, vt1 = 0, vt2 = 0;
      int k0o = 0;  // virtual jumps on run 0
      {
        Real v = 0;
#pragma unroll
        for (int j = 0; j < 3; j++) {
          if (j < K) {
            v = next_order_stat<Real>(v, (Real)1, K - j, j == 0 ? oB : pw[j - 1 < 0 ? 0 : j - 1]);
            const bool on0 = v < qq;
            const Real t = on0 ? min(PN::mul(v, sc0), p1) : PN::add(p1, min(PN::mul(PN::sub(v, qq), sc1), L1r));
            k0o += on0 ? 1 : 0;
            if (j == 0) vt0 = t; else if (j == 1) vt1 = t; else vt2 = t;
          }
        }
      }
      // the jump points with the real one in its place (after the k0o virtual jumps of run 0)
      J0 = vt0; J1 = vt1; J2 = vt2;
      if (nj == 1) {
        J2 = k0o == 2 ? p1 : vt1;
        J1 = k0o == 0 ? vt0 : k0o == 1 ? p1 : vt1;
        J0 = k0o == 0 ? p1 : vt0;
      }
    }
    // piece j of the path lies between jump points j - 1 and j (0 and Le at the ends); m = 3 or 4
    auto piece_len = [&](int jx) -> Real {
      const Real hi = jx == 0 ? J0 : jx == 1 ? J1 : (jx == 2 && m == 4) ? J2 : Le;
      const Real lo = jx == 0 ? (Real)0 : jx == 1 ? J0 : jx == 2 ? J1 : J2;
      return PN::sub(hi, lo);
    };
    // ---- the new path ----
    int nout = 0, S0 = 0, S1 = 0, S2 = 0, S3 = 0;
    Real L0 = 0, L1 = 0, L2 = 0, L3 = 0;
    auto emit = [&](Real L, int sst) {
      const int r = nout;
      if (r == 0) { L0 = L; S0 = sst; } else if (r == 1) { L1 = L; S1 = sst; } else if (r == 2) { L2 = L; S2 = sst; } else { L3 = L; S3 = sst; }
      if (r >= 2) add_dwell(sst, L);  // (runs 0 and 1: when the path is complete -- a two-run path is quantised first)
      nout++;
    };
    Stream gst; gst.open(P.rng, (uint32_t)site, iter, K_BRSTATE, (uint32_t)eb, P.err_flag);
    int cur_state = ps, prev = ps;
    Real cur_len = piece_len(0);
#pragma unroll
    for (int pp = 1; pp < 4; pp++) {
      if (pp < m) {
        int st;
        if (pp == m - 1) st = cs;
        else {
          const int jd = m - pp - 1;  // 1 or 2
          Real wv[NC];
          const Real* M = (jd < npow_s) ? (sPow + jd * n * n) : (P.ppow + (size_t)jd * n * n);
#pragma unroll
          for (int q = 0; q < n; q++) wv[q] = sB[prev * n + q] * M[q * n + cs];
          st = categorical<Real, NC, false>(wv, n, gst.next(), P.err_flag);
        }
        const Real len = piece_len(pp);
        if (full) atomicAdd(&s_cnt[prev * n + st], 1u);
        if (st == cur_state) cur_len = cur_len + len;
        else {
          emit(cur_len, cur_state);
          if (!full) atomicAdd(&s_cnt[cur_state * n + st], 1u);
          cur_state = st; cur_len = len;
        }
        prev = st;
      }
    }
    emit(nout == 0 ? Le : nout == 1 ? PN::sub(Le, L0) : cur_len, cur_state);
    // ---- the new virtual jumps: one run, or two runs counted together, from the pair block's A word; three or four
    // runs one by one (A, B, then the K_BRCNT block).  lam <= rate_max t_e < PM_LAMBDA_INV here: always count mode
    int newm = nout;
    uint32_t newq = 0;
    const Real rn0 = rate_or_zero(s_rate_new[S0]);
    if (nout == 1) {
      add_dwell(S0, L0);
      const int k0n = poisson_inv<Real>(PN::mul(rn0, L0), nA);
      newm += k0n;
      newq = pos_rand(nB);  // position of a lone virtual jump (used if k0n == 1): uniform on the branch
    } else {
      const Real rn1 = rate_or_zero(s_rate_new[S1]);
      if (nout == 2) {  // the jump point moves to its 16-bit lattice: everything below sees the stored path
        newq = pos_enc<Real>(L0, Le);
        L0 = pos_dec<Real>(newq, Le); L1 = PN::sub(Le, L0);
      }
      add_dwell(S0, L0); add_dwell(S1, L1);
      const Real lam0 = PN::mul(rn0, L0), lam1 = PN::mul(rn1, L1);
      if (nout == 2) newm += poisson_inv<Real>(PN::add(lam0, lam1), nA);
      else {
        uint32_t cw[4];
        philox4x32_10(0u, make_slot(K_BRCNT, (uint32_t)eb), iter, gsite, P.rng.k0, P.rng.k1, cw);
        newm += poisson_inv<Real>(lam0, nA) + poisson_inv<Real>(lam1, nB) +
                poisson_inv<Real>(PN::mul(rate_or_zero(s_rate_new[S2]), L2), cw[0]);
        if (nout == 4) newm += poisson_inv<Real>(PN::mul(rate_or_zero(s_rate_new[S3]), L3), cw[1]);
        const int ck = eb / P.chunk;
        const int cap0 = __ldg(P.cap_off + ck), cap_c = __ldg(P.cap_off + ck + 1) - cap0;
        const long long sl = ((long long)cap0 * P.rec_groups) + (site >> P.rec_shift) * (long long)cap_c;
        const int base = atomicAdd(P.rec_cursor + (long long)ck * P.rec_groups + (site >> P.rec_shift), nout);
        newq = (uint32_t)base;
        if (base + nout > cap_c) errbits |= PM_DE_PATH_CAP;
        else {
          wr_len[sl + base] = L0; wr_st[sl + base] = (uint8_t)S0;
          wr_len[sl + base + 1] = L1; wr_st[sl + base + 1] = (uint8_t)S1;
          wr_len[sl + base + 2] = L2; wr_st[sl + base + 2] = (uint8_t)S2;
          if (nout == 4) { wr_len[sl + base + 3] = L3; wr_st[sl + base + 3] = (uint8_t)S3; }
        }
      }
    }
    meta_out = PM_META(newm, newq);
    shape_out = PM_SHAPE(nout - 1, S0, S1);
  }

  // ---- any item: regenerate the pieces run by run, redraw the interior states, merge, count, emit ----
  __device__ __forceinline__ void general_item(const HardItem<Real> it, uint32_t& meta_out, uint16_t& shape_out) {
    const long long site = it.site;
    const int eb = (int)it.e;
    const uint32_t mt = it.meta;
    const int ck = eb / P.chunk;
    const int cap0 = __ldg(P.cap_off + ck), cap_c = __ldg(P.cap_off + ck + 1) - cap0;
    const long long sbase = ((long long)cap0 * P.rec_groups) + (site >> P.rec_shift) * (long long)cap_c;  // record slice of the site's group
    int* cursor = P.rec_cursor + (long long)ck * P.rec_groups + (site >> P.rec_shift);

    const int m = (int)(mt & 0xffffu);
    const int njf = first ? 0 : (int)(it.shape & 0x3fu);  // real jumps; 63 = "63 or more, see the record header"
    const int ps = (int)(it.ends & 0xffu), cs = (int)(it.ends >> 8);
    const Real Le = __ldg(P.e_len + eb);
    uint32_t po_old[4], po_new[4];
    pair_block(P.rng, (uint32_t)site, iter, (uint32_t)eb, po_new);
    if (!first) pair_block(P.rng, (uint32_t)site, iter - 1u, (uint32_t)eb, po_old);
    const uint32_t oA = (eb & 1) ? po_old[2] : po_old[0], oB = (eb & 1) ? po_old[3] : po_old[1];
    const uint32_t nA = (eb & 1) ? po_new[2] : po_new[0], nB = (eb & 1) ? po_new[3] : po_new[1];
    // nj == 1: pos1 = length of run 0; nj >= 2: pos1 = offset of the path's records in the site's slice.  A path with 64
    // or more runs starts with a header record holding its run count.
    const Real p1 = (!first && njf == 1) ? pos_dec<Real>(mt >> 16, Le) : (Real)0;
    int rd0 = (njf >= 2) ? (int)(mt >> 16) : 0;
    int nj = njf;
    if (njf == 63) {
      const int q = min(rd0, cap_c - 1);
      nj = max(63, (int)rd_len[sbase + q] - 1);
      rd0 += 1;
    }
    const int nrun = nj + 1;
    // a two-run path in joint count mode (the rule of the sweep that wrote it, evaluated with that sweep's rates)
    bool joint_old = false;
    if (!first && nj == 1) {
      const Real jr0 = rate_or_zero(s_rate_old[(it.shape >> 6) & 0x1fu]), jr1 = rate_or_zero(s_rate_old[(it.shape >> 11) & 0x1fu]);
      joint_old = !(PN::add(PN::mul(jr0, p1), PN::mul(jr1, PN::sub(Le, p1))) > (Real)PM_LAMBDA_INV);
    }

    // ---- the new path ----
    // Runs are emitted in order; the first two are held in registers until a third one shows up (a path with at most
    // one real jump lives in meta + pos1, only longer ones go to the record slice).
    int nout = 0, newm = 0, S0 = 0, S1 = 0, k0 = 0;
    Real L0 = 0, L1 = 0, gap0 = 0;
    bool gaps0 = false;
    Real bufL[PM_LOCAL_PATH_MAX]; uint8_t bufS[PM_LOCAL_PATH_MAX];  // runs 2.. of a long path (local memory, rarely touched)

    // One pass over the branch: regenerate the previous path piece by piece, redraw the interior states, merge, emit the
    // runs.  All uniforms come from keyed streams opened here, so a second pass reproduces the first: a path with more
    // runs than the local buffer holds (a saturated branch) is walked again with `replay` set, and this time its runs go
    // straight to the records reserved at `wbase` -- nothing else is done twice (no counts, dwell times or draws of new
    // virtual jumps).
    int wbase = 0;
    uint32_t newq = 0;  // position field of the new state word
#pragma unroll 1
    for (int pass = 0; pass < 2; pass++) {  // pass 1 only for a path longer than the local buffer (see below)
      const bool replay = pass != 0;
      WordStream cnt_old; cnt_old.open(P.rng, (uint32_t)site, first ? iter : iter - 1u, K_BRCNT, (uint32_t)eb, 0u);
      WordStream cnt_new; cnt_new.open(P.rng, (uint32_t)site, iter, K_BRCNT, (uint32_t)eb, 0u);
      Stream gst; gst.open(P.rng, (uint32_t)site, iter, K_BRSTATE, (uint32_t)eb, P.err_flag);
      int jrun = 0;
      RunPieces<Real> rp;
      long long cp = first ? P.maps_off[eb] : 0;
      auto open_run = [&](int r) {
        Real len; int st;
        if (joint_old) {  // two runs whose virtual jumps were counted together (A word); positions: B, then (K_BRPOS; run 0)
          const Real jr0 = rate_or_zero(s_rate_old[(it.shape >> 6) & 0x1fu]), jr1 = rate_or_zero(s_rate_old[(it.shape >> 11) & 0x1fu]);
          const Real L1o = PN::sub(Le, p1);
          const Real jlam0 = PN::mul(jr0, p1), jlamT = PN::add(jlam0, PN::mul(jr1, L1o));
          if (r == 0) rp.begin_joint(P.rng, (uint32_t)site, iter - 1u, (uint32_t)eb, p1, poisson_inv<Real>(jlamT, oA), jlam0, jlamT, jr0, oB);
          else rp.second_run(L1o, jlamT, jr1);
          return;
        }
        if (nj == 0) { len = Le; st = (int)((it.shape >> 6) & 0x1fu); }
        else if (nj == 1) { len = r == 0 ? p1 : PN::sub(Le, p1); st = (int)((it.shape >> (r == 0 ? 6 : 11)) & 0x1fu); }
        else { const int q = min(rd0 + r, cap_c - 1); len = rd_len[sbase + q]; st = rd_st[sbase + q]; }
        const uint32_t cw = r == 0 ? oA : r == 1 ? oB : cnt_old.next();
        rp.begin(P.rng, (uint32_t)site, iter - 1u, (uint32_t)eb, r, len, s_rate_old[st], cw, nj == 0, oB);
      };
      if (!first) open_run(0);
      auto next_piece = [&]() -> Real {
        if (first) return (Real)P.maps_len[cp++];
        if (jrun >= nrun) { errbits |= PM_DE_INCONSISTENT; return (Real)0; }
        bool last;
        const Real piece = rp.next(last);
        if (last) { jrun++; if (jrun < nrun) open_run(jrun); }
        return piece;
      };
      nout = 0;
      // new virtual jumps of run r (length L, clamped rate): their count, by inversion or, above PM_LAMBDA_INV, by gaps
      auto draw_run = [&](int r, Real L, Real rate, uint32_t cw) -> int {
        if (!(rate > (Real)0)) return 0;
        const Real lam = PN::mul(rate, L);
        if (!(lam > (Real)PM_LAMBDA_INV)) return poisson_inv<Real>(lam, cw);
        Real g1 = 0;
        const int k = count_gaps<Real>(P.rng, (uint32_t)site, iter, (uint32_t)eb, (uint32_t)r, L, rate, &g1);
        if (r == 0) { gaps0 = true; gap0 = g1; }
        return k;
      };
      auto emit = [&](Real L, int s) {
        const int r = nout;
        if (replay) {  // records only; the header sits at wbase
          wr_len[sbase + wbase + 1 + r] = L; wr_st[sbase + wbase + 1 + r] = (uint8_t)s;
          nout++;
          return;
        }
        if (r == 0) { L0 = L; S0 = s; }
        else if (r == 1) { L1 = L; S1 = s; }
        else if (r < PM_LOCAL_PATH_MAX) { bufL[r] = L; bufS[r] = (uint8_t)s; }
        if (r >= 2) add_dwell(s, L);
        // the count word of run r >= 2 is consumed whether or not the run uses it (gap mode, zero rate): the next sweep's
        // open_run() takes one word per run when it regenerates this path.  Runs 0 and 1 draw when the path is complete
        // (a path of two runs counts its virtual jumps together)
        newm += 1;
        if (r >= 2) newm += draw_run(r, L, rate_or_zero(s_rate_new[s]), cnt_new.next());
        nout++;
      };

      int cur_state = (m == 1) ? cs : ps;
      Real cur_len = next_piece();
      int prev = cur_state;
      for (int p = 1; p < m; p++) {
        int st;
        if (p == m - 1) st = cs;
        else {
          const int jd = m - p - 1;  // beta_jd = Bs^jd e_cs
          Real wv[NC];
          const Real* M = (jd < npow_s) ? (sPow + jd * n * n) : (jd < P.jcap ? P.ppow + (size_t)jd * n * n : nullptr);
          if (M) {
#pragma unroll
            for (int c = 0; c < n; c++) wv[c] = M[c * n + cs];
          } else {
#pragma unroll
            for (int c = 0; c < n; c++) wv[c] = (Real)(c == cs);
            for (int r = 0; r < jd; r++) matvec<Real, NC, false>(sBs, n, wv);
          }
#pragma unroll
          for (int c = 0; c < n; c++) wv[c] = sB[prev * n + c] * wv[c];
          st = categorical<Real, NC, false>(wv, n, gst.next(), P.err_flag);
        }
        const Real len = next_piece();
        if (full && !replay) atomicAdd(&s_cnt[prev * n + st], 1u);
        if (st == cur_state) cur_len = cur_len + len;
        else {
          emit(cur_len, cur_state);
          if (!full && !replay) atomicAdd(&s_cnt[cur_state * n + st], 1u);
          cur_state = st; cur_len = len;
        }
        prev = st;
      }
      if (!first && (jrun != nrun)) errbits |= PM_DE_INCONSISTENT;  // the regenerated pieces must add up to m
      // a single-run path spans the whole branch: take its length from the tree, not from the sum of its pieces
      // ... and the second run of a two-run path is what is left after the first (the form the next sweep rebuilds it in)
      emit(nout == 0 ? Le : nout == 1 ? PN::sub(Le, L0) : cur_len, cur_state);
      if (replay) {
        if (nout != (int)wr_len[sbase + wbase]) errbits |= PM_DE_INCONSISTENT;  // the header holds the count of pass 0
        break;
      }
      {  // runs 0 and 1: dwell times and new virtual jumps, now that the path is complete
        if (nout == 2) {  // the jump point moves to its 16-bit lattice: everything below sees the stored path
          newq = pos_enc<Real>(L0, Le);
          L0 = pos_dec<Real>(newq, Le); L1 = PN::sub(Le, L0);
        }
        add_dwell(S0, L0);
        if (nout >= 2) add_dwell(S1, L1);
        const Real rn0 = rate_or_zero(s_rate_new[S0]), rn1 = nout >= 2 ? rate_or_zero(s_rate_new[S1]) : (Real)0;
        const bool together = nout == 2 && !(PN::add(PN::mul(rn0, L0), PN::mul(rn1, L1)) > (Real)PM_LAMBDA_INV);
        if (together) newm += poisson_inv<Real>(PN::add(PN::mul(rn0, L0), PN::mul(rn1, L1)), nA);
        else {
#pragma unroll 1
          for (int r = 0; r < min(nout, 2); r++) {
            const int k = draw_run(r, r == 0 ? L0 : L1, r == 0 ? rn0 : rn1, r == 0 ? nA : nB);
            if (r == 0) k0 = k;
            newm += k;
          }
        }
      }
      if (newm > 65535) { errbits |= PM_DE_M_OVERFLOW; newm = 65535; }
      if (nout == 1) {  // a lone virtual jump: uniform on the branch (count mode), or where the first gap put it
        newq = (k0 == 1 && gaps0) ? pos_enc<Real>(gap0, Le) : pos_rand(nB);
        break;
      }
      if (nout == 2) break;
      // three or more runs: a contiguous block of records in the site's slice; its offset goes where a shorter path
      // keeps the position of its jump point.  64 runs or more: a header record with the count comes first.
      const bool longp = nout >= 64;
      const int need = nout + (longp ? 1 : 0);
      const int base = atomicAdd(cursor, need);
      newq = (uint32_t)min(base, 65535);
      if (base + need > cap_c || base > 65535) { errbits |= PM_DE_PATH_CAP; break; }
      if (longp) { wr_len[sbase + base] = (Real)nout; wr_st[sbase + base] = 0; }
      if (nout > PM_LOCAL_PATH_MAX) {  // not all runs were kept: walk the branch once more, writing them in place
        wbase = base;
        continue;
      }
      const int o = base + (longp ? 1 : 0);
      wr_len[sbase + o] = L0; wr_st[sbase + o] = (uint8_t)S0;
      wr_len[sbase + o + 1] = L1; wr_st[sbase + o + 1] = (uint8_t)S1;
      for (int r = 2; r < nout; r++) { wr_len[sbase + o + r] = bufL[r]; wr_st[sbase + o + r] = bufS[r]; }
      break;
    }
    meta_out = PM_META(newm, newq);
    shape_out = PM_SHAPE(min(nout - 1, 63), S0, S1);
  }
};

// WHICH = 0: the short items only (small code, half the registers: twice the resident warps), launched first: it clears
// the ballot bits of the items it takes.  WHICH = 1: whatever is left.
template <typename Real, int NS, int MINB, int WHICH>
__global__ void __launch_bounds__(128, MINB) k_paths_hard(ChainParams<Real> P, uint32_t iter, int first) {
  if (P.ctl) { iter = P.ctl[0]; first = iter == 0u; }
  constexpr int NR = NS > 0 ? NS : 1;
  typedef typename StreamSel<Real, false>::type Stream;
  typedef Pin<Real> PN;
  const int n = NS > 0 ? NS : P.n;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* s_dw = reinterpret_cast<double*>(smem_raw);                 // [4 warps][n] (NS>0) or [n] atomics (NS==0)
  unsigned* s_cnt = reinterpret_cast<unsigned*>(s_dw + 4 * n);       // [n*n]
  Real* sB = reinterpret_cast<Real*>(s_cnt + n * n + ((n * n) & 1));  // dense B (forward row)
  Real* sBs = sB + n * n;
  Real* sVec = sBs + n * n;  // pid | scale_old | scale_new | rate_old | rate_new
  Real* sPow = sVec + 5 * n;
  const int npow_s = min(NS > 0 ? PM_SMEM_POW : 0, P.jcap);  // the first powers of B in shared memory (n = 2, 4)
  for (int i = threadIdx.x; i < n * n; i += blockDim.x) { sB[i] = P.model[i]; sBs[i] = P.model[n * n + i]; s_cnt[i] = 0; }
  for (int i = threadIdx.x; i < 5 * n; i += blockDim.x) sVec[i] = P.model[2 * n * n + i];
  for (int i = threadIdx.x; i < npow_s * n * n; i += blockDim.x) sPow[i] = P.ppow[i];
  for (int i = threadIdx.x; i < 4 * n; i += blockDim.x) s_dw[i] = 0.0;
  // per-warp queues of classified items: [0] the common short shape (processed by straight-line code), [1] everything else
  __shared__ HardItem<Real> s_q[4][64];
  __shared__ unsigned short s_stage[4][1024];  // site offsets of the set bits of the warp's current work item (<= 32 words)
  __syncthreads();
  const Real* s_rate_old = sVec + 3 * n;
  const Real* s_rate_new = sVec + 4 * n;
  Real rate_max = 0;  // largest virtual-jump rate of the previous and of this sweep: bounds every run's lambda by rate_max * t_e
  for (int s = 0; s < n; s++) {
    const Real a = s_rate_old[s], b = s_rate_new[s];
    if (rate_ok(a)) rate_max = max(rate_max, a);
    if (rate_ok(b)) rate_max = max(rate_max, b);
  }
  const long long S = P.S;
  const int W = P.W;
  PathWorker<Real, NS> pw(P, iter, first, n, sB, sBs, sPow, npow_s, s_cnt, s_dw, s_rate_old, s_rate_new);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned FULL = 0xffffffffu;

  // ---- the warp walks its work items; items are classified, queued and processed 32 at a time ----
  // One loop, one place where items are processed (the kernel stalls mostly on instruction fetch: branchy code, few
  // resident warps -- every extra inlined copy of an item routine costs).
  int nq = 0;  // queue fill (warp-uniform)
  const long long gw = (long long)blockIdx.x * (blockDim.x >> 5) + warp, NW = (long long)gridDim.x * (blockDim.x >> 5);
  long long wi = gw;
  unsigned long long en_next = wi < P.wk_total ? __ldg(P.wk_item + wi) : 0ull;  // the entry of the NEXT work item, in flight
  int e = 0, base = 0, total = 0, c = 0, inc = 0;
  long long w0 = 0, prow = 0, crow = 0, erow = 0;
  uint32_t bits = 0;
  bool short_ok = false, finishing = false;
  for (;;) {
    const bool room = nq < 32;  // a round queues up to 32 items, the queue holds 64
    if (room && base >= total && !finishing) {  // next work item
      if (wi >= P.wk_total) finishing = true;
      else {
        const unsigned long long en = en_next;
        e = (int)(en >> 32);
        w0 = (long long)((en >> 5) & 0x7ffffffull);
        const int nw = (int)(en & 31ull) + 1;
        wi += NW;
        en_next = wi < P.wk_total ? __ldg(P.wk_item + wi) : 0ull;
        bits = lane < nw ? P.hard_ballot[(long long)e * W + w0 + lane] : 0u;
        c = __popc(bits);
        inc = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(FULL, inc, o); if (lane >= o) inc += v; }
        total = __shfl_sync(FULL, inc, 31);
        base = 0;
        if (total == 0) continue;
        // every lane lists the set bits of its own word: site offsets inside the work item, in site order
        __syncwarp();
        {
          int pos = inc - c;
          uint32_t b2 = bits;
          while (b2) { s_stage[warp][pos++] = (unsigned short)(lane * 32 + __ffs((int)b2) - 1); b2 &= b2 - 1u; }
        }
        __syncwarp();
        short_ok = !first && PN::mul(rate_max, __ldg(P.e_len + e)) <= (Real)(PM_LAMBDA_INV - 0.5);  // (sums of two products stay below PM_LAMBDA_INV)
        prow = (long long)__ldg(P.e_parent + e) * S; crow = (long long)__ldg(P.e_child + e) * S; erow = (long long)e * S;
      }
    }
    if (room && !finishing) {  // queue the next 32 items of the work item
      const int k = base + lane;
      const bool have = k < total;
      HardItem<Real> it;
      it.e = (uint32_t)e;
      it.site = have ? (uint32_t)(w0 * 32 + s_stage[warp][k]) : 0u;
      it.meta = 0u; it.ends = 0u; it.shape = 0u;
      if (have) {  // four independent loads
        it.meta = P.meta[erow + it.site];
        const uint32_t a = P.node_state[prow + it.site], b = P.node_state[crow + it.site];
        if (!first) it.shape = P.shape[erow + it.site];
        it.ends = a | (b << 8);
      }
      bool is_short = false;
      if (WHICH == 0 && have && short_ok) {
        const int m = (int)(it.meta & 0xffffu), njq = (int)(it.shape & 0x3fu);
        // three or four pieces; at most one real jump (the virtual ones are regenerated) or nothing but real jumps (records)
        is_short = (m == 3 || m == 4) && (njq <= 1 || njq == m - 1);
      }
      // the short launch (first) takes its items out of the ballot array; the general launch takes whatever is left
      const bool mine = have && (WHICH == 1 || is_short);
      if (WHICH == 0 && mine) atomicAnd(P.hard_ballot + (long long)e * W + (it.site >> 5), ~(1u << (it.site & 31u)));
      const unsigned bq = __ballot_sync(FULL, mine);
      if (mine) s_q[warp][nq + __popc(bq & ((1u << lane) - 1u))] = it;
      nq += __popc(bq);
      base += 32;
      __syncwarp();
    }
    if (nq >= 32 || (finishing && nq > 0)) {
      const int take = min(nq, 32);
      nq -= take;
      if (lane < take) {
        const HardItem<Real> it = s_q[warp][nq + lane];
        uint32_t mo; uint16_t so;
        if (WHICH == 0) pw.short_item(it, mo, so);
        else pw.general_item(it, mo, so);
        const long long pe = (long long)it.e * S + it.site;
        P.meta[pe] = mo;
        P.shape[pe] = so;
      }
      __syncwarp();
    } else if (finishing) break;
  }
  if (pw.errbits) atomicOr(P.err_flag, pw.errbits);

  if (NS > 0) {
#pragma unroll
    for (int j = 0; j < NR; j++) {
      double v = pw.Rsum[j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
      if (lane == 0) s_dw[warp * n + j] = v;
    }
  }
  __syncthreads();
  if ((int)threadIdx.x < n) {
    double v;
    if (NS > 0) { v = 0; for (int ww = 0; ww < (int)(blockDim.x >> 5); ww++) v += s_dw[ww * n + threadIdx.x]; }
    else v = s_dw[threadIdx.x];
    P.dw_partial[((long long)P.easy_blocks + (WHICH ? 2LL * gridDim.x : 0LL) + blockIdx.x) * n + threadIdx.x] = v;
  }
  for (int i = threadIdx.x; i < n * n; i += blockDim.x) if (s_cnt[i]) atomicAdd(&P.cnt[i], (unsigned long long)s_cnt[i]);
}

}  // namespace pm

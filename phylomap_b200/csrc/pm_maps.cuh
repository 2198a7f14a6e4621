// Stochastic maps of the current chain state, decoded on the device (pm_chain_get_maps).
//   k_maps_count  run count of every (selected site, branch): production nj + 1 from the shape word (or the header record
//                 when nj = 63), deterministic mode nj + 1 from the meta word
//   (an exclusive scan of the counts, cub::DeviceScan, gives the CSR offsets)
//   k_maps_write  the runs of every (selected site, branch) at its offset, lengths widened to double exactly as
//                 pm_chain_get_path does: a one-run path is (t_e, s0), a two-run path is (pos_dec(q, t_e), s0),
//                 (t_e - that, s1), longer paths are copied from the record slice the last sweep wrote
// Unit of work: a tile of 32 selected sites x 32 branches per block of 32 x 8 threads.  The state words are read with the
// site on the lane (a contiguous selection reads the branch-major rows coalesced), transposed through shared memory, and
// the outputs written with the branch on the lane (site-major: one warp writes consecutive offsets).  Neither kernel
// writes to a chain buffer.
#pragma once
#include "pm_kernels.cuh"

namespace pm {

// device scratch of one batch of selected sites: counts and offsets, and the runs of a range of the batch's sites
constexpr size_t kMapsScratchBytes = (size_t)512 << 20;

template <typename Real>
struct MapsSrc {
  const uint32_t* meta; const uint16_t* shape;   // [E][S]; shape: production only
  const Real* e_len;
  const Real* rec_len; const uint8_t* rec_st;    // the record buffer the last sweep wrote
  const int* cap_off;                            // [chunks + 1]
  long long S, rec_groups;
  int E, chunk, rec_shift, exact;
};

// slice of (branch chunk of e, site group of `site`) in the record buffer
template <typename Real>
__device__ __forceinline__ long long maps_slice(const MapsSrc<Real>& M, long long site, int e) {
  const int c = e / M.chunk;
  const int c0 = __ldg(M.cap_off + c), cap_c = __ldg(M.cap_off + c + 1) - c0;
  return (long long)c0 * M.rec_groups + (site >> M.rec_shift) * (long long)cap_c;
}

template <typename Real>
__device__ __forceinline__ void maps_load_tile(const MapsSrc<Real>& M, const long long* __restrict__ sel, long long i0, long long i1,
                                               int e0, uint32_t (*sm)[33], uint32_t (*ss)[33], long long* ssite) {
  const int tx = threadIdx.x, ty = threadIdx.y;
  const long long i = i0 + tx;
  const long long site = i < i1 ? __ldg(sel + i) : 0;
  if (ty == 0) ssite[tx] = site;
  for (int r = ty; r < 32; r += 8) {
    const int e = e0 + r;
    if (e < M.E && i < i1) {
      const size_t k = (size_t)e * M.S + site;
      sm[r][tx] = __ldg(M.meta + k);
      ss[r][tx] = M.exact ? 0u : (uint32_t)__ldg(M.shape + k);
    }
  }
  __syncthreads();
}

template <typename Real>
__global__ void __launch_bounds__(256) k_maps_count(MapsSrc<Real> M, const long long* __restrict__ sel, long long nb, int* __restrict__ cnt) {
  __shared__ uint32_t sm[32][33], ss[32][33];
  __shared__ long long ssite[32];
  const int e0 = blockIdx.x * 32;
  const long long i0 = (long long)blockIdx.y * 32;
  maps_load_tile(M, sel, i0, nb, e0, sm, ss, ssite);
  const int e = e0 + threadIdx.x;
  if (e >= M.E) return;
  for (int r = threadIdx.y; r < 32 && i0 + r < nb; r += 8) {
    const uint32_t m = sm[threadIdx.x][r], sh = ss[threadIdx.x][r];
    int runs;
    if (M.exact) runs = (int)((m >> 16) & 0xffu) + 1;
    else {
      const int nj = (int)(sh & 0x3fu);
      runs = nj + 1;
      if (nj == 63) runs = (int)__ldg(M.rec_len + maps_slice(M, ssite[r], e) + (m >> 16));  // header record: the run count
    }
    cnt[(i0 + r) * M.E + e] = runs;
  }
}

// sites [j0, j1) of the batch; off: the batch's offsets, rbase: the offset of site j0's first run (index 0 of len / st)
template <typename Real>
__global__ void __launch_bounds__(256) k_maps_write(MapsSrc<Real> M, const long long* __restrict__ sel, long long j0, long long j1,
                                                   const long long* __restrict__ off, long long rbase, double* __restrict__ len,
                                                   int32_t* __restrict__ st) {
  typedef Pin<Real> PN;
  __shared__ uint32_t sm[32][33], ss[32][33];
  __shared__ long long ssite[32];
  const int e0 = blockIdx.x * 32;
  const long long i0 = j0 + (long long)blockIdx.y * 32;
  maps_load_tile(M, sel, i0, j1, e0, sm, ss, ssite);
  const int e = e0 + threadIdx.x;
  if (e >= M.E) return;
  for (int r = threadIdx.y; r < 32 && i0 + r < j1; r += 8) {
    const uint32_t m = sm[threadIdx.x][r], sh = ss[threadIdx.x][r];
    const long long site = ssite[r];
    const long long* o = off + (i0 + r) * M.E;
    const long long p = o[e] - rbase;
    const int runs = (int)(o[e + 1] - o[e]);
    long long pos;
    if (M.exact) {
      // every path keeps its runs as records, the paths of a chunk one after the other
      pos = o[e] - o[(e / M.chunk) * M.chunk];
    } else {
      const int nj = (int)(sh & 0x3fu);
      const int s0 = (int)((sh >> 6) & 0x1fu);
      const Real Le = __ldg(M.e_len + e);
      if (nj == 0) { len[p] = (double)Le; st[p] = s0; continue; }
      if (nj == 1) {
        const Real p1 = pos_dec<Real>(m >> 16, Le);
        len[p] = (double)p1; st[p] = s0;
        len[p + 1] = (double)PN::sub(Le, p1); st[p + 1] = (int)((sh >> 11) & 0x1fu);
        continue;
      }
      pos = (long long)(m >> 16) + (nj == 63 ? 1 : 0);
    }
    const long long b = maps_slice(M, site, e) + pos;
    for (int k = 0; k < runs; k++) { len[p + k] = (double)__ldg(M.rec_len + b + k); st[p + k] = (int32_t)__ldg(M.rec_st + b + k); }
  }
}

}  // namespace pm

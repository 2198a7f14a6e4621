// Launch interface between the host (pm_host.cu) and the sweep kernels, which are instantiated in separate
// translation units (pm_sweep_*.cu) so that they compile in parallel.
#pragma once
#include "pm_kernels.cuh"
#include "pm_small.cuh"

namespace pm {

template <typename Real, int NS, bool EXACT>
struct Sweep {
  // the production arithmetic for n = 2 / 4 has kernels of its own (the clade kernels, the one-block-per-site kernel);
  // run-time n and the deterministic mode run the generic ones
  static constexpr bool production = !EXACT && (NS == 2 || NS == 4);
  // K1 and K2 as two launches over all sites: the stand-alone clade kernels (production: the DIC chains and
  // PHYLOMAP_B200_FUSED=0) or k_prune / k_nodes
  static void prune(const ChainParams<Real>& P, int grid, size_t smem, cudaStream_t st);
  static void nodes(const ChainParams<Real>& P, int grid, size_t smem, cudaStream_t st, uint32_t iter);
  // production: the fused prune + node-draw kernel over the site blocks [b0, b0 + grid); phases 1 = prune only.
  // slot_busy: slots_per_sm flags per SM (nullptr: block i uses slot i).  fused_blocks_per_sm: resident blocks per SM.
  static int fused_blocks_per_sm(size_t smem_nodes);
  static void prune_nodes(const ChainParams<Real>& P, int grid, size_t smem_nodes, cudaStream_t st, uint32_t iter, long long b0,
                          int phases, int* slot_busy, int slots_per_sm, unsigned long long* phase_ns);
  static void paths(const ChainParams<Real>& P, dim3 grid, size_t smem, cudaStream_t st, uint32_t iter, int first, int chunk,
                    int hard_blocks);
  // production, few sites on a tree whose per-site state fits shared memory: `nsweeps` sweeps of every site in
  // ONE launch, a block per site (pm_small.cuh).  small_smem: the dynamic shared memory it needs for T tips.
  static size_t small_smem(int T);
  static void small_chain(const ChainParams<Real>& P, int sites, cudaStream_t st, uint32_t iter0, int nsweeps, const SmallOut& out,
                          bool two_per_sm);
};

}  // namespace pm

#pragma once
#include "pm_launch.cuh"

namespace pm {

template <typename Real, int NS, bool EXACT>
void Sweep<Real, NS, EXACT>::prune(const ChainParams<Real>& P, int grid, size_t smem, cudaStream_t st) {
  if constexpr (!EXACT && (NS == 2 || NS == 4)) {
    constexpr int D = 8, MB = sizeof(Real) == 8 ? 2 : 3;  // FP64 needs the registers of 2 blocks / SM
    const size_t spow = 2 * PM_SMEM_POW * NS * NS * sizeof(Real);  // the power table and its transpose
    const size_t sm = spow + (size_t)PM_CLADE_SLOT * 8 * D;
    auto kern = k_prune_clade<Real, NS, D, MB>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    kern<<<grid, 256, sm, st>>>(P);
  }
  else k_prune<Real, NS, EXACT><<<grid, 256, smem, st>>>(P);
}
template <typename Real, int NS, bool EXACT>
void Sweep<Real, NS, EXACT>::nodes(const ChainParams<Real>& P, int grid, size_t smem, cudaStream_t st, uint32_t iter) {
  if constexpr (!EXACT && (NS == 2 || NS == 4)) {
    constexpr int D = 8, MB = sizeof(Real) == 8 ? 2 : 3;
    const size_t sm = smem + (size_t)(32 * NS * sizeof(Real) + 160) * 8 * D;
    auto kern = k_nodes_clade<Real, NS, D, MB>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    kern<<<grid, 256, sm, st>>>(P, iter);
  }
  else k_nodes<Real, NS, EXACT><<<grid, 256, smem, st>>>(P, iter);
}
template <typename Real, int NS, bool EXACT>
struct FusedCfg {
  static constexpr int D = 8, MB = sizeof(Real) == 8 ? 2 : 3;  // FP64 needs the registers of 2 blocks / SM
  static size_t smem(size_t smem_nodes) {
    const size_t sm_prune = 2 * PM_SMEM_POW * (NS > 0 ? NS : 1) * (NS > 0 ? NS : 1) * sizeof(Real) + (size_t)PM_CLADE_SLOT * 8 * D;
    const size_t sm_nodes = smem_nodes + (size_t)(32 * (NS > 0 ? NS : 1) * sizeof(Real) + 160) * 8 * D;
    return sm_prune > sm_nodes ? sm_prune : sm_nodes;
  }
};
template <typename Real, int NS, bool EXACT>
int Sweep<Real, NS, EXACT>::fused_blocks_per_sm(size_t smem_nodes) {
  if constexpr (!EXACT && (NS == 2 || NS == 4)) {
    typedef FusedCfg<Real, NS, EXACT> C;
    auto kern = k_prune_nodes_clade<Real, NS, C::D, C::MB>;
    const size_t sm = C::smem(smem_nodes);
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, 256, sm) != cudaSuccess) return 0;
    return nb;
  }
  return 0;
}
template <typename Real, int NS, bool EXACT>
void Sweep<Real, NS, EXACT>::prune_nodes(const ChainParams<Real>& P, int grid, size_t smem_nodes, cudaStream_t st, uint32_t iter,
                                         long long b0, int phases, int* slot_busy, int slots_per_sm, unsigned long long* phase_ns) {
  if constexpr (!EXACT && (NS == 2 || NS == 4)) {
    typedef FusedCfg<Real, NS, EXACT> C;
    auto kern = k_prune_nodes_clade<Real, NS, C::D, C::MB>;
    const size_t sm = C::smem(smem_nodes);
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    kern<<<grid, 256, sm, st>>>(P, iter, b0, phases, slot_busy, slots_per_sm, phase_ns);
  }
}
template <typename Real, int NS, bool EXACT>
void Sweep<Real, NS, EXACT>::paths(const ChainParams<Real>& P, dim3 grid, size_t smem, cudaStream_t st, uint32_t iter,
                                   int first, int chunk, int hard_blocks) {
  if constexpr (EXACT) k_paths<Real, NS, true><<<grid, 128, smem, st>>>(P, iter, first, chunk);
  else {
    // the easy kernel also serves the first sweep: a map of one or two pieces is a path like any other (pos1 was
    // seeded from it), only longer maps are walked piece by piece by the general kernel
    const size_t smem_easy = EasySmem<Real, NS>(P.n).bytes(chunk);
    k_paths_easy<Real, NS><<<grid, 128, smem_easy, st>>>(P, iter, chunk);
    // (the short shape does not occur in the first sweep: the caller's maps are walked by the general routine)
    if (!first) k_paths_hard<Real, NS, 8, 0><<<2 * hard_blocks, 128, smem, st>>>(P, iter, first);
    k_paths_hard<Real, NS, 4, 1><<<hard_blocks, 128, smem, st>>>(P, iter, first);
  }
}
template <typename Real, int NS, bool EXACT>
size_t Sweep<Real, NS, EXACT>::small_smem(int T) {
  if constexpr (!EXACT && (NS == 2 || NS == 4)) return (size_t)SmallSmem<Real, NS>(T).total;
  return (size_t)1 << 40;  // no such kernel
}
template <typename Real, int NS, bool EXACT>
void Sweep<Real, NS, EXACT>::small_chain(const ChainParams<Real>& P, int sites, cudaStream_t st, uint32_t iter0, int nsweeps,
                                         const SmallOut& out, bool two_per_sm) {
  if constexpr (!EXACT && (NS == 2 || NS == 4)) {
    const size_t sm = (size_t)SmallSmem<Real, NS>(P.T).total;
    auto kern = two_per_sm ? k_small_chain<Real, NS, 2> : k_small_chain<Real, NS, 1>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    kern<<<sites, 256, sm, st>>>(P, iter0, nsweeps, out);
  }
}

}  // namespace pm

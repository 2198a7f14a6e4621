"""phylomap_b200: B200-native stochastic-mapping MCMC core (the uniformization sampler of vnminin/phylomap).

Only the hot path lives here: the CUDA kernels and C ABI (csrc/, include/phylomap_b200.h), the ctypes binding
(capi), the host-side mirror of the reference's R functions (api), and synthetic-input generators (synth).
"""
from . import capi  # noqa: F401
from .api import (Chain, ExpectedSumstats, SPARSEmaketreelistMCMC, SPARSEsumstatMCMC, colnames, expected_sumstats, loglik, make2stateDIC, make2stateDICbig, make4stateDIC,  # noqa: F401
                  make4stateDICbig, makenodelist, maketreelistEXP, maketreelistMCMC,  # noqa: F401
                  maketreelistMCMC2sDICt, maketreelistMCMC_bigtree, maketreelistMCMCbf, maketreelistMCMCks,
                  maketreelistMCMCksDICt, maketreelistMCMCksmt, maketreelistMCMCmt, myreorder, pruningwiseedgeorder,
                  sumstatEXP, sumstatMCMC, sumstatMCMC2sDICt, sumstatMCMC_bigtree, sumstatMCMCbf, sumstatMCMCks, sumstatMCMCksDICt,
                  sumstatMCMCksmt, sumstatMCMCmt)
from .simmap import StochasticMaps, multi_simmap  # noqa: F401
from .tree import PhyloTree  # noqa: F401

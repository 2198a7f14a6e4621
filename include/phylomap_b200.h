/*
 * phylomap_b200 — C ABI of the B200-native stochastic-mapping MCMC core.
 *
 * This is the drop-in boundary for the hot path of vnminin/phylomap: the seven uniformization samplers that
 * the reference exports to R through Rcpp (`.Call('phylomap_<fn>', ...)`, reference src/RcppExports.cpp).
 * Every pm_maketreelist* entry below replaces exactly one `[[Rcpp::export]]` function of the reference
 * src/phylomap.cpp; arguments keep the reference's meaning, order and 1-based conventions, flattened from
 * R objects to plain pointers (INTEGRATION.md shows the Rcpp shim that does the flattening).
 *
 *   pm_SPARSEmaketreelistMCMC   <- SPARSEmaketreelistMCMC   src/phylomap.cpp:822  (src/RcppExports.cpp:11)
 *   pm_maketreelistMCMC         <- maketreelistMCMC         src/phylomap.cpp:891  (src/RcppExports.cpp:34)
 *   pm_maketreelistMCMC_bigtree <- maketreelistMCMC_bigtree src/phylomap.cpp:942  (src/RcppExports.cpp:57)
 *   pm_maketreelistMCMCbf       <- maketreelistMCMCbf       src/phylomap.cpp:1258 (src/RcppExports.cpp:106)
 *   pm_maketreelistMCMCks       <- maketreelistMCMCks       src/phylomap.cpp:1802 (src/RcppExports.cpp:132)
 *   pm_maketreelistMCMCmt       <- maketreelistMCMCmt       src/phylomap.cpp:2267 (src/RcppExports.cpp:159)
 *   pm_maketreelistMCMCksmt     <- maketreelistMCMCksmt     src/phylomap.cpp:2722 (src/RcppExports.cpp:185)
 *   pm_maketreelistEXP          <- maketreelistEXP          src/phylomap.cpp:3001 (src/RcppExports.cpp:80)
 *   pm_maketreelistMCMC2sDICt   <- maketreelistMCMC2sDICt   src/phylomap.cpp:3183 (src/RcppExports.cpp:211)
 *   pm_maketreelistMCMCksDICt   <- maketreelistMCMCksDICt   src/phylomap.cpp:3300 (src/RcppExports.cpp:237)
 *   pm_loglik                   <- the pruning loop of make2stateDIC / make4stateDIC(big), R/sourceme.R:141-177, 248-284, 445-516
 *   pm_expected_sumstats        (no counterpart: the exact posterior expectations the fixed-Q samplers estimate)
 *   pm_tree_order               <- pruningwiseedgeorder / makenodelist / myreorder, R/sumstatMCMC.R:1-18 (O(E) here)
 *
 * There is no CPU fallback: every entry fails with PM_ERR_CUDA when no sm_100 device is usable.
 *
 * New with respect to the reference: a data-parallel SITE axis.  `states` may hold n_sites tip-state vectors
 * (site-major).  All sites share the tree, the initial segmentation (`maps`) and Q; each site is an independent
 * copy of the reference's chain; row i of the result holds the SUM over sites of the per-site statistics
 * (this is what the conjugate rate updates consume); per-site columns (root state) report global site 0.
 * n_sites == 1 reproduces the reference's call.
 */
#ifndef PHYLOMAP_B200_H
#define PHYLOMAP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PM_OK 0
#define PM_ERR_ARG 1        /* malformed input (message in err) */
#define PM_ERR_CUDA 2       /* CUDA runtime failure / no usable device */
#define PM_ERR_SAMPLE 3     /* RcppArmadillo::sample would have thrown (NA / negative / all-zero weights) */
#define PM_ERR_CAPACITY 4   /* a capacity was exceeded: the run records of a branch chunk (pm_options.path_capacity), 65535 jump
                               points on one branch, or (deterministic mode only) 63 state changes on one branch at one site */
#define PM_ERR_REPLAY 5     /* replay table exhausted */

/* precision of the device arithmetic */
#define PM_F64 0
#define PM_F32 1
/* arithmetic mode */
#define PM_MODE_PRODUCTION 0     /* fast: fused multiply-add allowed, B^k tables, -log(u) exponentials */
#define PM_MODE_DETERMINISTIC 1  /* reference order of operations, no FMA, R's exp_rand, sorted categorical draw */
/* source of uniforms for the device-side draws */
#define PM_RNG_PHILOX 0          /* Philox4x32-10 keyed by (seed, site, iteration, slot, k) */
#define PM_RNG_TABLE 1           /* replay of a uniform stream exported from a sequential (R-order) run */

/* One tree in the reference's tweaked ape/phytools layout (fields read at src/phylomap.cpp:896-910). */
typedef struct pm_tree {
  int32_t n_tips;            /* T = length(x$states); tips are nodes 1..T, internal nodes T+1..2T-1 */
  int32_t n_edges;           /* E = nrow(x$edge) = 2T-2 (binary trees only, as the reference: :508-510) */
  const int32_t* edge;       /* x$edge, column-major [2E]: E parents then E children, 1-based */
  const int32_t* nen;        /* [E] pruning-wise edge order, 1-based edge rows, sibling pairs adjacent */
  const int32_t* nodelist;   /* [T-2] internal nodes below the root, top-down, 1-based */
  int32_t root;              /* 1-based root node */
  const int64_t* maps_off;   /* [E+1] CSR offsets into maps_len / maps_state */
  const double* maps_len;    /* x$maps: initial segment lengths of every branch */
  const int32_t* maps_state; /* x$mapnames (1-based); validated only — every sweep redraws all segment states */
  const int32_t* states;     /* x$states, 1-based, [n_sites][T] site-major; may be NULL if states_u8 is given */
  const uint8_t* states_u8;  /* optional compact alternative to `states` (same values, same layout) */
  int64_t n_sites;           /* S (1 = the reference) */
  const double* edge_length; /* x$edge.length [E]: read by the DIC samplers only (src/phylomap.cpp:3225); NULL = sum of maps */
} pm_tree;

/* Site sharding over several processes (one per GPU).  Either give the library an NCCL clique (nccl_id / nccl_rank /
 * nccl_world below: it then calls ncclAllReduce itself on the chain's stream), or a callback of this type, which must sum
 * `count` doubles at DEVICE address `dev_buf` across all ranks in stream order on pm_options.cuda_stream (which is then
 * mandatory: the library cannot order a foreign collective on its private stream) and return 0.  The reduced row carries
 * one extra double, the sum of the ranks' device error flags, so every rank sees a failure in the same iteration and all
 * of them leave together instead of hanging in the next collective.  Called once per iteration by the rate-updating
 * samplers (bf/ks/mt/ksmt), once per pm_chain_run by the fixed-Q ones. */
typedef int (*pm_allreduce_fn)(void* ctx, double* dev_buf, int32_t count);

typedef struct pm_options {
  int32_t device;          /* CUDA device ordinal */
  int32_t precision;       /* PM_F64 | PM_F32 */
  int32_t mode;            /* PM_MODE_PRODUCTION | PM_MODE_DETERMINISTIC */
  int32_t rng;             /* PM_RNG_PHILOX | PM_RNG_TABLE */
  uint64_t seed;           /* Philox key; host-side rate-update draws use R's Mersenne-Twister set.seed((uint32)seed) */
  int64_t site_offset;     /* global index of local site 0 (site sharding); keys use global site indices */
  int32_t path_capacity;   /* stored path records per (site, branch) on average over a chunk of branches; 0 = sized from the
                              Poisson tail of the real-jump counts and the initial maps (PM_ERR_CAPACITY asks to raise it) */
  int32_t power_capacity;  /* number of tabulated powers of B; 0 = sized from Omega x the longest branch (>= 64); beyond
                              the table the kernels fall back to repeated mat-vecs */
  const int64_t* tab_off;  /* PM_RNG_TABLE: CSR over slots ((tree*S+site)*N+iter)*(2T-1+2E) + slot */
  const double* tab_u;     /*               the uniforms */
  const double* host_tab;  /*               uniforms consumed by the host-side rate updates, in order */
  int64_t host_tab_n;
  pm_allreduce_fn allreduce; /* NULL = single process */
  void* allreduce_ctx;
  void* cuda_stream;       /* cudaStream_t to launch on; NULL = a private stream */
  int32_t progress;        /* non-zero: print "%i \r" per iteration like the reference (:930) */
  int32_t nccl_world;      /* > 1: number of ranks of the NCCL clique the library joins at pm_chain_create (a collective call
                              the first time an id is seen; the communicator is then kept for the life of the process and
                              reused by every later call that passes the same id) */
  int32_t nccl_rank;       /* this process's rank in it */
  int32_t reserved;
  const void* nccl_id;     /* the clique's 128-byte ncclUniqueId: pm_nccl_unique_id() on one rank, handed to the others by the
                              caller (MPI, a file, torch.distributed.broadcast ...) */
} pm_options;

void pm_default_options(pm_options* o);
/* Writes a fresh ncclUniqueId (128 bytes) for pm_options.nccl_id.  NCCL is loaded at run time (libnccl.so.2; override
 * with PHYLOMAP_B200_NCCL=/path); PM_ERR_CUDA if it cannot be. */
int pm_nccl_unique_id(void* out128, char* err, size_t errlen);

/* Fixed-Q samplers.  out: caller-owned, column-major [N x (n + n(n-1))]:
 * [R_0..R_{n-1}, N_{0->1}, N_{0->2}, ... (diagonal skipped) ..., N_{n-1->n-2}]  (man/sumstatMCMC.Rd:18). */
int pm_maketreelistMCMC(const pm_tree* x, int32_t n, double* Q, const double* pid, double* B, double Omega,
                        int32_t N, const pm_options* opt, double* out, char* err, size_t errlen);
int pm_SPARSEmaketreelistMCMC(const pm_tree* x, int32_t n, double* Q, const double* pid, double* B, double Omega,
                              int32_t N, const pm_options* opt, double* out, char* err, size_t errlen);
int pm_maketreelistMCMC_bigtree(const pm_tree* x, int32_t n, double* Q, const double* pid, double* B, double Omega,
                                int32_t N, const pm_options* opt, double* out, char* err, size_t errlen);

/* Rate-updating samplers.  Q and B (column-major n x n) are updated IN PLACE like the reference does
 * (B2 aliases B: src/phylomap.cpp:1284).  out column layouts:
 *   bf   [N x 9]             t0 t1 n00 n01 n10 n11 l01 l10 root          (R/sumstatMCMCbf.R:33)
 *   ks   [N x n+n^2+2+3k+1]  R(n) N(n x n row-major) l01 l10 rk(k) lk(k) gamma(k) root   (src/phylomap.cpp:1789-1795)
 *   mt   [N x 9]             as bf, last column = 0-based index of the tree recorded    (R/sumstatMCMCmt.R:39)
 *   ksmt                     as ks, last column = tree index                             (src/phylomap.cpp:2828)
 * prior: bf/mt 4 values, ks 6, ksmt 8 (man/sumstatMCMCbf.Rd:16, man/sumstatMCMCks.Rd:16, man/sumstatMCMCksmt.Rd:16). */
int pm_maketreelistMCMCbf(const pm_tree* x, int32_t n, double* Q, const double* pid, double* B, double Omega,
                          int32_t N, const double* prior, int32_t nprior, const pm_options* opt, double* out,
                          char* err, size_t errlen);
int pm_maketreelistMCMCks(const pm_tree* x, int32_t n, double* Q, const double* pid, double* B, double Omega,
                          int32_t N, const double* prior, int32_t nprior, const pm_options* opt, double* out,
                          char* err, size_t errlen);
int pm_maketreelistMCMCmt(const pm_tree* trees, int32_t ntrees, int32_t n, double* Q, const double* pid, double* B,
                          double Omega, int32_t N, const double* prior, int32_t nprior, const pm_options* opt,
                          double* out, char* err, size_t errlen);
int pm_maketreelistMCMCksmt(const pm_tree* trees, int32_t ntrees, int32_t n, double* Q, const double* pid, double* B,
                            double Omega, int32_t N, const double* prior, int32_t nprior, const pm_options* opt,
                            double* out, char* err, size_t errlen);

/* DIC chains: the bf / ks samplers with one more column, log p(y | Q) of the current rates by matrix exponentiation
 * (summed over sites), computed after every sweep and before the rate update (src/phylomap.cpp:3242-3250, :3383-3390):
 *   2sDICt [N x 10]                  t0 t1 n00 n01 n10 n11 l01 l10 root loglik
 *   ksDICt [N x n+n^2+2+3k+2]        as ks, then loglik */
int pm_maketreelistMCMC2sDICt(const pm_tree* x, int32_t n, double* Q, const double* pid, double* B, double Omega, int32_t N,
                              const double* prior, int32_t nprior, const pm_options* opt, double* out, char* err,
                              size_t errlen);
int pm_maketreelistMCMCksDICt(const pm_tree* x, int32_t n, double* Q, const double* pid, double* B, double Omega, int32_t N,
                              const double* prior, int32_t nprior, const pm_options* opt, double* out, char* err,
                              size_t errlen);

/* log p(y | Q) alone, summed over sites (and over ranks when pm_options.allreduce is set): Felsenstein pruning with
 * P(t_e) = exp(Q edge_length[e]) (maps sums when edge_length is NULL), every node rescaled.  This is the D(Q-hat) term the
 * R helpers make2stateDIC / make4stateDIC / make{2,4}stateDICbig evaluate with expm() and an R loop over the nodes
 * (R/sourceme.R:141-177, 248-284, 445-516).  parity_tips != 0: the hidden-rate tip partials (1,0,1,0,..) / (0,1,0,1,..)
 * of make4stateDIC (:264-267); 0: one-hot tips.  Q column-major n x n, n <= 8; not modified. */
int pm_loglik(const pm_tree* x, int32_t n, const double* Q, const double* pid, int32_t parity_tips, const pm_options* opt,
              double* out, char* err, size_t errlen);

/* Exact posterior expectations under a fixed Q (no sampling, no random numbers): for every site, the expected dwell
 * times and transition counts given the tip data, in the fixed-Q sampler row layout (n + n(n-1) columns), and log p(y|Q);
 * for the selected LOCAL sites also per branch (edge-row order) and the marginal state probabilities of every node.
 *   stats          column-major [S x (n + n(n-1))] or NULL
 *   loglik         [S] or NULL
 *   branch_stats   [nsel][E][n + n(n-1)] or NULL        node_marginals  [nsel][2T-1][n] or NULL (0-based node ids)
 * parity_tips as in pm_loglik; Q column-major n x n, 2 <= n <= 8; not modified.  Branch lengths as in
 * pm_loglik (edge_length, or the sums of maps when it is NULL).  Sites may repeat and come in any order.  The simulation-free
 * stochastic mapping of Minin & Suchard (2008): branch integrals by Van Loan's block exponential, an inside and an
 * outside pruning pass on the device, in tiles of sites that change no output bit.  pm_options.precision and .device
 * apply; mode, seed and the collective options have no effect.  PM_ERR_ARG before any device work for a null tree, Q or
 * pid, n out of range, parity tips with an odd n or a site out of range; PM_ERR_SAMPLE when a site's data have zero
 * likelihood under Q (in FP32 also when its products underflow). */
int pm_expected_sumstats(const pm_tree* x, int32_t n, const double* Q, const double* pid, int32_t parity_tips,
                         const int64_t* sites, int64_t nsel, const pm_options* opt, double* stats, double* loglik,
                         double* branch_stats, double* node_marginals, char* err, size_t errlen);

/* The direct sampler with matrix exponentiation, maketreelistEXP (src/phylomap.cpp:3001, src/RcppExports.cpp:80): N
 * INDEPENDENT histories per site.  lefts / rights / d: eigenvectors, their inverse and diag(eigenvalues) of Q, column-major
 * n x n as R/sumstatEXP.R:26-31 passes them.  Omega := -min diag(Q) (:3008).  out: [N x (n + n(n-1))] like the fixed-Q samplers.
 * Production arithmetic only. */
int pm_maketreelistEXP(const pm_tree* x, int32_t n, double* Q, const double* pid, int32_t N, const double* lefts,
                       const double* rights, const double* d, const pm_options* opt, double* out, char* err, size_t errlen);

/* Number of result columns of a variant (PM_V_*) for n states. */
#define PM_V_PLAIN 0
#define PM_V_SPARSE 1
#define PM_V_BIGTREE 2
#define PM_V_BF 3
#define PM_V_KS 4
#define PM_V_MT 5
#define PM_V_KSMT 6
#define PM_V_DIC2S 7
#define PM_V_DICKS 8
#define PM_V_EXP 9
int32_t pm_ncols(int32_t variant, int32_t n);

/* O(E) replacement of the R helpers pruningwiseedgeorder / makenodelist / myreorder (R/sumstatMCMC.R:1-18):
 * a valid pruning-wise edge order (children before parents, sibling pairs adjacent), the top-down list of the
 * internal nodes below the root, and the root.  edge: column-major [2E], 1-based. */
int pm_tree_order(const int32_t* edge, int32_t n_edges, int32_t n_tips, int32_t* nen, int32_t* nodelist,
                  int32_t* root, char* err, size_t errlen);

/* ---- Resident-chain interface (what the one-call entries are built from; used by benchmarks and tests) ---- */
typedef struct pm_chain pm_chain;

int pm_chain_create(int32_t variant, const pm_tree* trees, int32_t ntrees, int32_t n, double* Q, const double* pid,
                    double* B, double Omega, const double* prior, int32_t nprior, int32_t N_total,
                    const pm_options* opt, pm_chain** out, char* err, size_t errlen);
/* Run `count` further iterations; rows [first .. first+count) of `out` (column-major, leading dimension ld)
 * are written.  first must equal the number of iterations already done. */
int pm_chain_run(pm_chain* c, int32_t count, double* out, int64_t ld, char* err, size_t errlen);
/* Test hook (host only, no device needed): builds the clade schedules the production pruning / node-draw kernels walk for
 * this tree (pm_tree.hpp) and verifies them -- every internal node once, children before parents inside a warp's
 * sequence, register / reload flags consistent, top-down order valid.  stats[8]: nodes in warp sequences, nodes above
 * the clades, levels above, lightest and heaviest warp, children handed over in registers, top-down sequence nodes,
 * top-down top nodes. */
int pm_debug_clade_schedule(const int32_t* edge, int32_t n_edges, int32_t n_tips, const int32_t* nen, const int32_t* nodelist,
                            int32_t root, int32_t nwarps, int32_t clade_max, int64_t* stats, char* err, size_t errlen);

/* Checkpoint / resume (the reference has none: its chain state is lost when the call returns, SURVEY.md §5).  The
 * exported blob holds what the next sweep reads and pm_chain_create does not rebuild: iteration counter, host generator,
 * current Q and B, node states, jump counts, first positions and run records.  Import into a chain created with the SAME
 * arguments (trees, sampler, precision, mode, seed, site block); Q and B are written back into the caller's arrays.  A
 * resumed run continues bit for bit like the uninterrupted one (device uniforms are keyed by (seed, site, sweep, slot)). */
int64_t pm_chain_state_bytes(pm_chain* c);
int pm_chain_export_state(pm_chain* c, void* buf, int64_t bytes, char* err, size_t errlen);
int pm_chain_import_state(pm_chain* c, const void* buf, int64_t bytes, char* err, size_t errlen);
/* Launch `reps` pruning passes (kernel K1 only) on the current chain state; returns the mean milliseconds per pass
 * measured with CUDA events on the chain's stream.  Does not modify the chain. */
int pm_chain_time_prune(pm_chain* c, int32_t tree, int32_t reps, float* ms_per_pass, char* err, size_t errlen);
/* Per-kernel CUDA-event times (ms) accumulated since creation: [prune, sample_nodes, resample_paths, reduce], and
 * the number of kernel launches issued. */
void pm_chain_kernel_times(pm_chain* c, double ms[4], int64_t* launches);
void pm_chain_enable_timing(pm_chain* c, int32_t on);
/* Rate-updating samplers, with timing enabled: ms[0] = device time of the per-sweep all-reduces (CUDA events around the
 * collective), ms[1] = host time of the replicated rate updates + model upload, both accumulated since creation. */
void pm_chain_overheads(pm_chain* c, double ms[2]);
/* State after the last sweep, copied to host (for parity tests). */
int pm_chain_get_node_states(pm_chain* c, int32_t tree, int32_t* out /* [S][2T-1] 0-based */);
int pm_chain_get_piece_counts(pm_chain* c, int32_t tree, int32_t* out /* [S][E] */);
int pm_chain_get_path(pm_chain* c, int32_t tree, int64_t site, int32_t e, double* len, int32_t* st, int32_t cap);
/* Stochastic maps of the current chain state: the merged history of every branch of the selected LOCAL sites of tree
 * `tree`, as stored after the last sweep.  Output is CSR, site-major in the order of `sites`, branches in edge-row order
 * (x$edge), runs from the parent end to the child end:
 *   off[i*E + e] .. off[i*E + e + 1]  -> len[], st[] (0-based states), i = position in `sites`;  off has nsel*E + 1 entries.
 * off is always written.  len / st are written when non-NULL and cap >= off[nsel*E]; when non-NULL with a smaller cap the
 * call returns PM_ERR_CAPACITY having written off (and nothing beyond len[cap - 1] / st[cap - 1]).  Sites may repeat and
 * come in any order.  Every run equals what pm_chain_get_path returns for the same (site, branch).  Decoded on the device
 * in batches of sites; does not modify the chain.  PM_ERR_ARG for a bad tree or site, before the first sweep, and for the
 * chains that keep no paths (the direct sampler). */
int pm_chain_get_maps(pm_chain* c, int32_t tree, const int64_t* sites, int64_t nsel, int64_t* off, double* len,
                      int32_t* st, int64_t cap, char* err, size_t errlen);
/* Partials of the current chain state at `site`, computed by a pruning pass that the call runs; tip rows are zero. */
int pm_chain_get_partials(pm_chain* c, int32_t tree, int64_t site, double* out /* [2T-1][n], tip rows zero */);
int64_t pm_chain_device_bytes(pm_chain* c);
/* Rate-updating samplers: per rate parameter, in the order of the trace columns (l01, l10, then for the hidden-rate
 * models kappa-> x k, kappa<- x k, gamma x k), how many Gamma proposals were drawn and how many were installed in Q
 * (the reference has no such counter; its accept / reject logic is src/phylomap.cpp:1205-1219, 1466-1500, ...).
 * Returns the number of parameters (0 for the fixed-Q samplers); at most `cap` entries are written. */
int32_t pm_chain_acceptance(pm_chain* c, int64_t* proposed, int64_t* accepted, int32_t cap);
void pm_chain_destroy(pm_chain* c);

/* Host-side random numbers used by the rate updates (R's Mersenne-Twister after set.seed(seed), unif_rand, exp_rand,
 * norm_rand, rgamma(a, scale=b)): n deviates of kind 0 unif, 1 exp, 2 norm, 3 gamma.  No device needed; lets the CPU tests
 * pin this restatement of R's nmath (Rf_rgamma at src/phylomap.cpp:1202, runif at :1210, ...) against known R outputs. */
void pm_rng_probe(uint32_t seed, int32_t kind, int32_t n, double a, double b, double* out);

/* Device memory of destroyed chains is cached per process for the next call of the same shape (cudaMalloc / cudaFree of
 * tens of GB would dominate a short call); this returns it to the driver.  PHYLOMAP_B200_CACHE=0 disables the cache. */
void pm_release_cached_memory(void);

/* Library / device probe: returns the number of CUDA devices with compute capability 10.x, or a negative error. */
int pm_device_count(void);
const char* pm_version(void);

#ifdef __cplusplus
}
#endif
#endif

// libphylomap_b200: host side of the B200 stochastic-mapping sampler and its C ABI (include/phylomap_b200.h).
//
// One pm_chain owns, per tree, the device-resident state of all local sites (layout in pm_kernels.cuh) and the
// small replicated model (Q, B, powers of B).  An iteration is four launches per tree (prune, node draws, branch
// paths, reduce); the fixed-Q samplers never synchronise inside pm_chain_run, the rate-updating samplers read
// one row of n + n^2 + 1 doubles back per iteration, update Q on the host (pm_rates.hpp) and upload the model.
//
// Replaces (reference src/phylomap.cpp): maketreelistMCMC :891, SPARSEmaketreelistMCMC :822,
// maketreelistMCMC_bigtree :942, maketreelistMCMCbf :1258, maketreelistMCMCks :1802, maketreelistMCMCmt :2267,
// maketreelistMCMCksmt :2722.
#include <cuda_runtime.h>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/phylomap_b200.h"
#include "pm_launch.cuh"
#include "pm_setup_kernels.cuh"
#include "pm_loglik.cuh"
#include "pm_expect.cuh"
#include "pm_maps.cuh"
#include "pm_exp.cuh"
#include "pm_nccl.hpp"
#include "pm_rates.hpp"
#include "pm_tree.hpp"

namespace {

struct Fail {
  int code;
  std::string msg;
};

[[noreturn]] void fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  throw Fail{code, buf};
}

#define CK(call)                                                                                     \
  do {                                                                                               \
    cudaError_t e_ = (call);                                                                         \
    if (e_ != cudaSuccess) fail(PM_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_));        \
  } while (0)

void set_err(char* err, size_t n, const std::string& m) {
  if (err && n) snprintf(err, n, "%s", m.c_str());
}

template <typename F>
int guarded(char* err, size_t errlen, F&& f) {
  try {
    f();
    if (err && errlen) err[0] = 0;
    return PM_OK;
  } catch (const Fail& x) {
    set_err(err, errlen, x.msg);
    return x.code;
  } catch (const std::string& s) {
    set_err(err, errlen, s);
    return PM_ERR_ARG;
  } catch (const std::exception& x) {
    set_err(err, errlen, x.what());
    return PM_ERR_ARG;
  }
}

// Device allocations go through a small per-process cache: cudaMalloc / cudaFree of tens of GB cost 0.1-0.4 s per call,
// which would dominate a short drop-in call (R users call the samplers repeatedly on the same tree).  Freed blocks are
// kept by (device, size) and handed back to the next chain that asks for exactly that size; pm_release_cached_memory()
// returns them to the driver, PHYLOMAP_B200_CACHE=0 disables the cache.
struct DevicePool {
  std::mutex mu;
  std::multimap<std::pair<int, size_t>, void*> free_blocks;
  bool enabled;
  DevicePool() { const char* v = getenv("PHYLOMAP_B200_CACHE"); enabled = !(v && v[0] == '0'); }
  void* take(int dev, size_t n) {
    if (enabled) {
      std::lock_guard<std::mutex> g(mu);
      auto it = free_blocks.find({dev, n});
      if (it != free_blocks.end()) { void* p = it->second; free_blocks.erase(it); return p; }
    }
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, n);
    if (e != cudaSuccess && enabled) {  // make room and retry once
      cudaGetLastError();
      release();
      e = cudaMalloc(&p, n);
    }
    if (e != cudaSuccess) fail(PM_ERR_CUDA, "cudaMalloc(%zu bytes) failed: %s", n, cudaGetErrorString(e));
    return p;
  }
  void give(int dev, size_t n, void* p) {
    if (!p) return;
    if (enabled) { std::lock_guard<std::mutex> g(mu); free_blocks.insert({{dev, n}, p}); }
    else cudaFree(p);
  }
  void release() {
    std::lock_guard<std::mutex> g(mu);
    for (auto& kv : free_blocks) cudaFree(kv.second);
    free_blocks.clear();
  }
};
DevicePool& pool() { static DevicePool p; return p; }

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  int dev = 0;
  DevBuf() {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { pool().give(dev, bytes, p); }
  void alloc(size_t n) {
    pool().give(dev, bytes, p);
    p = nullptr; bytes = n;
    cudaGetDevice(&dev);
    if (n) p = pool().take(dev, n);
  }
  template <typename T> T* as() const { return static_cast<T*>(p); }
};

template <typename T>
void upload(DevBuf& b, const std::vector<T>& v, cudaStream_t st) {
  b.alloc(std::max<size_t>(v.size(), 1) * sizeof(T));
  if (!v.empty()) CK(cudaMemcpyAsync(b.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, st));
}

struct Variant {
  int id;
  bool sparse, normalize, full_counts, redraw_tips, parity_tips, rates, multi, hidden, dic, two_state, exp, llonly;
};
// internal ids behind pm_loglik: a chain that only evaluates log p(y | Q) (no path state is allocated)
enum { V_LOGLIK = 100, V_LOGLIK_PARITY = 101 };
Variant variant_of(int v) {
  Variant r{};
  r.id = v;
  const bool bf = v == PM_V_BF || v == PM_V_DIC2S, ks = v == PM_V_KS || v == PM_V_DICKS;
  r.sparse = v == PM_V_SPARSE;
  r.normalize = v == PM_V_BIGTREE || bf || ks;
  r.full_counts = bf || ks || v == PM_V_MT || v == PM_V_KSMT;
  r.redraw_tips = ks || v == PM_V_MT || v == PM_V_KSMT;
  r.parity_tips = ks || v == PM_V_KSMT;
  r.rates = r.full_counts;
  r.multi = v == PM_V_MT || v == PM_V_KSMT;
  r.hidden = ks || v == PM_V_KSMT;
  r.dic = v == PM_V_DIC2S || v == PM_V_DICKS;
  r.two_state = bf || v == PM_V_MT;
  r.exp = v == PM_V_EXP;
  if (v == V_LOGLIK || v == V_LOGLIK_PARITY) { r.llonly = true; r.dic = true; r.normalize = true; r.parity_tips = v == V_LOGLIK_PARITY; }
  return r;
}

int ncols_of(int variant, int n) {
  const int k = n / 2 - 1;
  switch (variant) {
    case PM_V_PLAIN: case PM_V_SPARSE: case PM_V_BIGTREE: case PM_V_EXP: return n + n * (n - 1);
    case PM_V_BF: case PM_V_MT: return n + n * n + 3;
    case PM_V_DIC2S: return n + n * n + 4;
    case PM_V_KS: case PM_V_KSMT: return n + n * n + 2 + 3 * k + 1;
    case PM_V_DICKS: return n + n * n + 2 + 3 * k + 2;
    case V_LOGLIK: case V_LOGLIK_PARITY: return 1;
  }
  return -1;
}

// smallest c > lam with P(Poisson(lam) >= c) < eps, from the geometric bound on the tail beyond the mode:
// P(X >= c) <= pmf(c) / (1 - lam / (c + 1))
int poisson_cap(double lam, double eps) {
  if (!(lam > 0)) return 1;
  const double loglam = std::log(lam), logeps = std::log(eps);
  for (int c = (int)std::ceil(lam) + 1; c < 1000000; c++) {
    const double logpmf = -lam + c * loglam - std::lgamma(c + 1.0);
    if (logpmf - std::log1p(-lam / (c + 1.0)) < logeps) return c;
  }
  return 1000000;
}

// c such that P( sum_e X_e >= c ) < eps for independent X_e = (N_e + 1) 1[N_e >= 2], N_e ~ Poisson(lam_e):
// min over theta of (log(1/eps) + sum_e log E exp(theta X_e)) / theta
long long chernoff_records_cap(const std::vector<double>& lams, double eps, double copies = 1.0) {  // `copies` independent sites share the slice
  // (the small thetas serve slices shared by many sites: the bound tends to copies x mean + log(1 / eps) / theta)
  constexpr int NT = 11;
  const double thetas[NT] = {0.02, 0.04, 0.07, 0.12, 0.25, 0.5, 1.0, 1.5, 2.0, 3.0, 4.0};
  double acc[NT], eth[NT];
  bool ok[NT];
  // a slice of one site is bounded best by a large theta, a slice shared by many sites by a small one: half the grid each
  for (int t = 0; t < NT; t++) { acc[t] = 0; eth[t] = std::exp(thetas[t]); ok[t] = copies > 1.0 ? t < 7 : t >= 4; }
  static const std::vector<double> inv_j = [] { std::vector<double> v(400, 0.0); for (int j = 1; j < 400; j++) v[j] = 1.0 / j; return v; }();
  for (double lam : lams) {
    const double p0 = std::exp(-lam);
    for (int t = 0; t < NT; t++) {
      if (!ok[t]) continue;
      // E exp(theta X) = P(N < 2) + sum_{j >= 2} exp(theta (j + 1)) P(N = j); consecutive terms differ by the factor
      // exp(theta) lam / j (no exponential inside the loop: this runs for every branch at every chain creation)
      double mgf = p0 + p0 * lam;
      double term = eth[t] * eth[t] * p0 * lam;  // the j = 1 term of the series (not part of the sum)
      for (int j = 2; j < 400; j++) {
        term *= eth[t] * lam * inv_j[j];
        mgf += term;
        if (j > lam * eth[t] + 5 && term < 1e-30 * mgf) break;
      }
      if (!std::isfinite(mgf)) { ok[t] = false; continue; }
      acc[t] += std::log(mgf);
    }
  }
  double best = 1e300;
  for (int t = 0; t < NT; t++)
    if (ok[t]) best = std::min(best, (std::log(1.0 / eps) + copies * acc[t]) / thetas[t]);
  if (!(best < 1e15)) return 1LL << 40;
  return (long long)std::ceil(best);
}

// The run-time switches of INTEGRATION.md §5, read once: when a chain is created (and by the one-call entries, for the
// site tile).  PHYLOMAP_B200_CACHE belongs to the process-wide device pool and is read there.
struct Switches {
  bool small = true;             // PHYLOMAP_B200_SMALL=0: never the one-block-per-site kernel
  bool small_sites_set = false;  // PHYLOMAP_B200_SMALL_SITES=k: its site limit instead of the cost rule
  long long small_sites = 0;
  double small_work = 1.0;       // PHYLOMAP_B200_SMALL_WORK=f: scales its limit on the expected path cost
  bool rec_pool = true;          // PHYLOMAP_B200_REC_POOL=0: one record slice per site
  bool fused = true;             // PHYLOMAP_B200_FUSED=0: pruning and node draws as two kernels
  int graph = -1;                // PHYLOMAP_B200_GRAPH: 0 never, 1 always replay a captured sweep, otherwise by problem size
  bool trace = false;            // PHYLOMAP_B200_TRACE=1: host wall time of the phases of create(), on stderr
  bool debug_sync = false;       // PHYLOMAP_B200_DEBUG_SYNC=1: stop at the first sweep kernel that raises a device error flag
  long long site_tile = 0;       // PHYLOMAP_B200_SITE_TILE=k: fixed-Q one-call entries run k sites at a time (0: all)
};

Switches read_switches() {
  const auto env = [](const char* name) -> const char* { return getenv((std::string("PHYLOMAP_B200_") + name).c_str()); };
  const auto starts = [&](const char* name, char c) { const char* v = env(name); return v && v[0] == c; };
  Switches s;
  s.small = !starts("SMALL", '0');
  if (const char* v = env("SMALL_SITES")) { s.small_sites_set = true; s.small_sites = atoll(v); }
  if (const char* v = env("SMALL_WORK")) s.small_work = atof(v);
  s.rec_pool = !starts("REC_POOL", '0');
  s.fused = !starts("FUSED", '0');
  if (const char* v = env("GRAPH")) s.graph = atoi(v);
  s.trace = starts("TRACE", '1');
  s.debug_sync = starts("DEBUG_SYNC", '1');
  if (const char* v = env("SITE_TILE")) s.site_tile = atoll(v);
  return s;
}

// Host wall time of the phases of a chain's construction (PHYLOMAP_B200_TRACE=1), on stderr.
struct PhaseTrace {
  bool on;
  std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
  void mark(const char* what) {
    if (!on) return;
    const auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[phylomap_b200] create: %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t0).count());
    t0 = now;
  }
};

}  // namespace

// Range of %smid on a device (asked once per device with a one-thread kernel, see k_nsmid).
static int sm_id_range(int device, int reported_sms) {
  static std::mutex mu;
  static std::map<int, int> known;
  std::lock_guard<std::mutex> g(mu);
  auto it = known.find(device);
  if (it != known.end()) return it->second;
  int* d = nullptr;
  int v = 0;
  if (cudaMalloc(&d, sizeof(int)) != cudaSuccess) fail(PM_ERR_CUDA, "cudaMalloc failed");
  pm::k_nsmid<<<1, 1>>>(d);
  const cudaError_t e = cudaMemcpy(&v, d, sizeof(int), cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (e != cudaSuccess) fail(PM_ERR_CUDA, "reading %%nsmid failed: %s", cudaGetErrorString(e));
  v = std::max(v, reported_sms);
  known[device] = v;
  return v;
}

// NCCL communicators live as long as the process: a unique id can initialise a clique only once, and a session calls the
// samplers many times with the same id (ncclCommInitRank costs tenths of a second).  Keyed by the id's 128 bytes.
static pm::host::NcclApi::Comm clique(const void* id128, int world, int rank) {
  static std::mutex mu;
  static std::map<std::string, pm::host::NcclApi::Comm> comms;
  auto& api = pm::host::NcclApi::get();
  if (!api.ok()) fail(PM_ERR_CUDA, "NCCL could not be loaded: %s", api.why.c_str());
  const std::string key((const char*)id128, 128);
  std::lock_guard<std::mutex> g(mu);
  auto it = comms.find(key);
  if (it != comms.end()) return it->second;
  pm::host::NcclApi::UniqueId id;
  memcpy(&id, id128, sizeof id);
  pm::host::NcclApi::Comm c = nullptr;
  const int rc = api.CommInitRank(&c, world, id, rank);
  if (rc != 0) fail(PM_ERR_CUDA, "ncclCommInitRank failed: %s", api.error(rc).c_str());
  comms[key] = c;
  return c;
}

// ----------------------------------------------------------------------------------------------------------------
struct pm_chain {
  virtual ~pm_chain() {}
  virtual void run(int count, double* out, int64_t ld) = 0;
  virtual float time_prune(int tree, int reps) = 0;
  virtual void node_states(int tree, int32_t* out) = 0;
  virtual void piece_counts(int tree, int32_t* out) = 0;
  virtual int path(int tree, int64_t site, int e, double* len, int32_t* st, int cap) = 0;
  virtual void maps(int tree, const int64_t* sites, int64_t nsel, int64_t* off, double* len, int32_t* st, int64_t cap) = 0;
  virtual void partials(int tree, int64_t site, double* out) = 0;
  virtual double loglik() = 0;
  virtual void expected(bool write, double* stats, int64_t ld, double* loglik, double* branch_stats, double* node_marginals) = 0;
  virtual int64_t state_bytes() = 0;
  virtual void export_state(void* buf, int64_t bytes) = 0;
  virtual void import_state(const void* buf, int64_t bytes) = 0;
  double kernel_ms[4] = {0, 0, 0, 0};
  std::vector<long long> rate_proposed, rate_accepted;  // per rate parameter, trace-column order (pm_rates.hpp)
  double comm_ms = 0, host_update_ms = 0;  // with timing on: device time of the per-sweep all-reduces, host time of the rate updates
  int64_t launches = 0;
  int64_t dev_bytes = 0;
  bool timing = false;
};

namespace {

// ---- the plan of a tree's chain state: functions of the tree, the model and the options alone ----

// One block per site, state in shared memory (pm_small.cuh), when the sites are few and the tree fits: production
// arithmetic, 2 / 4 states (`eligible`; `smem`: the kernel's dynamic shared memory for this tree).  PHYLOMAP_B200_SMALL=0
// keeps the 32-sites-per-warp kernels (same rows: the tests compare), PHYLOMAP_B200_SMALL_SITES moves the site limit.
struct SmallChoice { bool ok, two; };  // two: more sites than SMs, two blocks per SM (128 registers) instead of one
template <typename Real>
SmallChoice choose_small_kernel(bool eligible, const std::vector<Real>& elen, double Omega, int T, long long S, int sms,
                                size_t smem, const Switches& sw) {
  long long small_sites = 16LL * sms;   // (hard cap; the cost rule below decides before it)
  if (sw.small_sites_set) small_sites = sw.small_sites;
  // ... and the paths of one site are short: a block walks its site's branches with 256 threads, one branch per thread
  // at a time, while the wide kernels spread the branch-sites of a long-path problem (the Squamate vignette: 877 000
  // jump points per site and sweep) over the whole device.  What costs is the general item routine: hard = the sum
  // over the branches of P(two or more jump points) x (2 + expected jump points), jump points ~ Poisson(Omega t).
  // Measured (scripts/small_calib.py, us per sweep, one character): this kernel ~ 20 + 0.05 hard + 0.03 T, the wide
  // ones ~ 65 + 0.13 T: it pays up to hard ~ 1500 + 0.7 T.  PHYLOMAP_B200_SMALL_WORK scales that limit.
  double hard = 0;
  for (size_t e = 0; e < elen.size(); e++) {
    const double lam = Omega * (double)elen[e];
    hard += (1.0 - std::exp(-lam) * (1.0 + lam)) * (2.0 + lam);
  }
  const double work_limit = sw.small_work * (1500.0 + 0.7 * T);
  SmallChoice c;
  c.two = S > sms;
  // More sites than SMs: two blocks per SM, waves of 2 x SMs sites; measured (profiles/r2_warp_per_site_attempt.log,
  // 100-800 tips, 296-2368 sites) a wave takes ~ 10 + 0.28 T + 0.05 hard us and the wide kernels ~ 160 + 0.09 T + 0.01 S.
  bool sites_ok = S <= small_sites;
  if (c.two && !sw.small_sites_set) {
    const double waves = std::ceil((double)S / (2.0 * sms));
    sites_ok = sites_ok && waves * (10.0 + 0.28 * T + 0.05 * hard) < 160.0 + 0.09 * T + 0.01 * (double)S;
  }
  c.ok = sw.small && eligible && sites_ok && smem <= (size_t)200 * 1024 && hard <= work_limit;
  return c;
}

// Launch geometry of the path kernels and the record capacity of every branch chunk, with slices shared by groups of
// 2^rec_shift consecutive sites.  (Production: the offset of a path's records inside its slice is a 16-bit field of the
// state word, so a chunk whose slice would be longer is split.)  Production slices are shared by groups of 32 consecutive
// sites (rec_shift = 5): the bound on the records of 32 independent sites together is far tighter, relative to its mean,
// than 32 bounds on one site each (3.8 -> 0.3 bytes per branch-site at the benchmark's size).  Where such a slice would
// not fit the 16-bit offset (long paths: the Squamate vignette) the plan is returned with fits = false, and the caller
// plans again with rec_shift = 0: every site keeps its own.
struct RecordPlan {
  int rec_shift = 0;
  long long gx = 0, ny = 0;  // path-kernel grid: site blocks x branch chunks
  int chunk = 0;             // consecutive branches per chunk
  std::vector<int> cap_off;  // [ny + 1] prefix sums of the chunks' record capacities (per slice)
  bool fits = true;
};
template <typename Real>
RecordPlan plan_records(int rec_shift, const std::vector<Real>& elen, const std::vector<long long>& moff, long long S,
                        double Omega, bool exact, bool no_paths, int path_capacity) {
  const int E = (int)elen.size();
  RecordPlan p;
  p.rec_shift = rec_shift;
  // a thread owns one site x one chunk of consecutive branches
  p.gx = (S + 127) / 128;
  long long ny = (148LL * 16 * 6 + p.gx - 1) / p.gx;
  ny = std::max(1LL, std::min<long long>(ny, (E + 15) / 16));
  ny = std::min<long long>(ny, 65535);
  ny = std::max<long long>(ny, (E + 2047) / 2048);  // the easy path kernel stages a chunk's topology in shared memory
  ny = std::max<long long>(ny, (E + ((1LL << 32) - 1) / S - 1) / std::max<long long>(1, ((1LL << 32) - 1) / S));  // ... and indexes the rows of a chunk with 32 bits: chunk x S < 2^32
  const double G = (double)(1 << rec_shift);
  for (;;) {
    p.chunk = (int)((E + ny - 1) / ny);
    ny = (E + p.chunk - 1) / p.chunk;
    long long cap_max = 0;
    // Real jumps sit on uniformization points, and in equilibrium the points of a chunk are Poisson(Omega x total
    // length), so the Poisson tail bounds them; a path with j real jumps stores j + 1 runs (<= 2j).  The first sweep
    // instead finds its points in the caller's maps (m_e - 1 per branch), so the initial segmentation is a second lower
    // bound.
    p.cap_off.assign(ny + 1, 0);
    for (long long c = 0; c < ny; c++) {
      const int b0 = (int)c * p.chunk, b1 = std::min(E, b0 + p.chunk);
      double len = 0;
      long long init_records = 0;
      for (int e = b0; e < b1; e++) {
        len += (double)elen[e];
        const long long m0 = moff[e + 1] - moff[e];
        if (exact || m0 >= 2) init_records += m0;
      }
      long long cap;
      if (no_paths) cap = 4;
      else if (path_capacity > 0) cap = (long long)path_capacity * (b1 - b0) * (long long)G;
      else if (exact) {
        const int jumps = poisson_cap(1.5 * Omega * len + 1.0, 1e-18);
        cap = std::max<long long>((long long)(b1 - b0) + jumps, init_records);
      } else {
        // production: only paths with >= 2 real jumps keep records (j + 1 of them); Chernoff bound on their sum
        // over the chunk with every branch's jump count dominated by Poisson(1.5 Omega t)
        std::vector<double> lams;
        long long init3 = 0;
        for (int e = b0; e < b1; e++) {
          lams.push_back(1.5 * Omega * (double)elen[e]);
          const long long m0 = moff[e + 1] - moff[e];
          if (m0 >= 3) init3 += m0;
        }
        // ... or, simpler and valid for any rate: every path stores at most (jumps + 1) records (+ a header), and the
        // jumps of the chunk together are dominated by one Poisson variable
        double lam_sum = 0, lam_max = 0;
        for (double l : lams) { lam_sum += l; lam_max = std::max(lam_max, l); }
        const long long simple = (long long)poisson_cap(G * lam_sum, 1e-18) + 2LL * (b1 - b0) * (long long)G;
        long long stat = simple;
        if (lam_max < 200.0) stat = std::min(stat, chernoff_records_cap(lams, 1e-18, G));  // (its series stops at 400 terms)
        cap = std::max<long long>(stat, init3 * (long long)G) + 4;
      }
      if (cap > (1 << 28)) { if (rec_shift) cap = 1 << 28; else fail(PM_ERR_CAPACITY, "path capacity of a branch chunk too large"); }
      cap = (cap + 3) & ~3;  // keep every slice 16-byte aligned
      cap_max = std::max(cap_max, cap);
      p.cap_off[c + 1] = p.cap_off[c] + (int)cap;
    }
    if (exact || no_paths || cap_max <= 65535) break;
    if (rec_shift) { p.fits = false; break; }  // shared slices too long for the offset field
    if (p.chunk <= 1 || ny >= 65535) fail(PM_ERR_CAPACITY, "a branch needs more than 65 535 path records per site");
    ny = std::min<long long>(std::min<long long>(2 * ny, E), 65535);
  }
  p.ny = ny;
  return p;
}

// The clade schedule of the production pruning and node-draw kernels (n = 2, 4), encoded as the byte offsets the kernels
// add to their per-lane bases.  rowPL: bytes of one node row of the partials buffer.
struct CladeCode {
  pm::host::CladeSchedule cs;   // (cs.top_off relative to the first top entry)
  std::vector<int> e16, top;    // bottom-up: the warps' entries, PM_CLADE_ENTRY_INTS ints each; the top levels
  std::vector<int> d16;         // top-down (k_nodes_clade): 16 ints per node
  std::vector<long long> tips;  // redrawn tips: entry v = tip v: the parent's node-state row, the jump-count row of its branch (bytes)
};
CladeCode encode_clade_schedule(const pm::host::Schedule& sch, long long S, long long TS, long long rowPL, bool redraw_tips) {
  const int T = sch.T;
  CladeCode c;
  pm::host::CladeSchedule& cs = c.cs;
  // clades of ~1/64 of the tree: ~8 per warp to balance, and only ~100 nodes left above them.  Small trees (where a
  // sweep is a matter of latency, not throughput): ~1/8 of the tree, so that almost every node is walked inside a
  // warp's prefetched sequence and only a few levels with block barriers are left above.  (A function of the tree
  // alone: the node draws are keyed by schedule position, and a site must not depend on how many others run.)
  const int clade_max = (T - 1 < 512) ? std::max(8, (T - 1) / 8) : std::max(8, std::min(512, (T - 1) / 64));
  pm::host::build_clade_schedule(sch, 8, clade_max, cs);
  const int n1 = cs.warp_off.back();
  c.e16.assign((size_t)PM_CLADE_ENTRY_INTS * (n1 + 17), 0);  // padded: the kernel forms addresses up to 16 entries ahead
  auto put64 = [](int* dst, long long v) { dst[0] = (int)(unsigned)(v & 0xffffffffLL); dst[1] = (int)(v >> 32); };
  for (int i = 0; i < n1; i++) {
    const int* en = &cs.entries[(size_t)8 * i];
    int* o = &c.e16[(size_t)PM_CLADE_ENTRY_INTS * i];
    const int pn = en[0], a = en[1], ea = en[2], b = en[3], eb = en[4];
    int fl = en[5] & 3;
    const int x = (en[5] & 4) ? a : (en[5] & 8) ? b : -1;
    if (a < T) fl |= 16;
    if (b < T) fl |= 32;
    put64(o + 0, (long long)(pn - T) * rowPL);
    put64(o + 2, x >= 0 ? (long long)(x - T) * rowPL : -1LL);
    put64(o + 4, (long long)ea * S * 4);
    put64(o + 6, (long long)eb * S * 4);
    put64(o + 8, a < T ? (long long)a * TS : -1LL);
    put64(o + 10, b < T ? (long long)b * TS : -1LL);
    o[12] = fl;
  }
  c.top.assign(cs.entries.begin() + (size_t)8 * n1, cs.entries.end());
  for (int& v : cs.top_off) v -= n1;
  const int n2 = cs.down_warp_off.back();
  c.d16.assign((size_t)16 * (n2 + 17), 0);
  for (int i = 0; i < n2; i++) {
    const int* en = &cs.down_seq[(size_t)4 * i];
    int* o = &c.d16[(size_t)16 * i];
    put64(o + 0, (long long)(en[0] - T) * rowPL);
    put64(o + 2, (long long)en[2] * S * 4);
    put64(o + 4, (long long)en[0] * S);
    put64(o + 6, en[3] ? -1LL : (long long)en[1] * S);
  }
  if (redraw_tips)
    for (int v = 0; v < T; v++) {
      const int e = sch.parent_edge[v];
      c.tips.push_back((long long)sch.e_parent[e] * S); c.tips.push_back((long long)e * S * 4);
    }
  return c;
}

// The one-block-per-site kernel's node draws and branch order.
struct SmallOrder {
  std::vector<int> down;    // 4 ints per drawn node: the generic schedule's (v, parent, edge) and the clade kernel's draw key
  std::vector<int> border;  // which thread takes which branch (-1: none)
};
template <typename Real>
SmallOrder small_draw_order(const pm::host::Schedule& sch, const pm::host::CladeSchedule& cs, const std::vector<Real>& elen) {
  const int T = sch.T, E = (int)elen.size();
  SmallOrder so;
  // the same draws node by node: every drawn node with the Philox block and word the clade kernel gives it
  // (k_small_chain decodes the key), grouped by depth like the generic schedule
  std::vector<uint32_t> key(2 * (size_t)T - 1, 0u);
  for (int i = 0; i < (int)cs.down_top.size() / 4; i++) key[cs.down_top[(size_t)4 * i]] = 0x80000000u | (uint32_t)i;
  for (int i = 0; i < cs.down_warp_off.back(); i++) key[cs.down_seq[(size_t)4 * i]] = (uint32_t)i;
  for (int v = 0; v < T; v++) key[v] = 0x40000000u | (uint32_t)v;
  const int nd = (int)sch.down_entries.size() / 3;
  so.down.assign((size_t)4 * std::max(nd, 1), 0);
  for (int i = 0; i < nd; i++) {
    const int* en = &sch.down_entries[(size_t)3 * i];
    so.down[(size_t)4 * i] = en[0]; so.down[(size_t)4 * i + 1] = en[1]; so.down[(size_t)4 * i + 2] = en[2]; so.down[(size_t)4 * i + 3] = (int)key[en[0]];
  }
  // Which thread takes which branch.  A warp runs the general item routine in lockstep: it takes as long as its
  // longest path, plus a share for every other shape among its items.  Up to 256 branches (one per thread): the
  // branches sorted by decreasing length are DEALT over the 8 warps, so that every warp gets one of the longest,
  // one of the next eight, ... (measured on configs[0]: all long branches in one warp 30 300 cycles for the path
  // phase, edge order 26 000).  Larger trees: decreasing length (warps of similar paths: throughput).
  std::vector<int> sorted(E);
  for (int e = 0; e < E; e++) sorted[e] = e;
  std::stable_sort(sorted.begin(), sorted.end(), [&](int x, int y) { return elen[x] > elen[y]; });
  if (E <= 256) {
    so.border.assign(256, -1);
    for (int k = 0; k < E; k++) so.border[(size_t)(k % 8) * 32 + k / 8] = sorted[k];   // warp k % 8, lane k / 8
  } else so.border = sorted;
  return so;
}

// Branch-major ballot array and the general path kernel's work items: branch e is cut into items of g_e ballot words
// (32 g_e sites), g_e chosen so that an item holds ~96 branch-sites with two or more jump points in equilibrium (their
// number on a branch of length t is Poisson(Omega t)).
struct WorkItems {
  std::vector<long long> off;  // [E + 1] first item of every branch
  std::vector<int> g;          // ballot words per item, per branch
};
template <typename Real>
WorkItems build_work_items(const std::vector<Real>& elen, double Omega, long long S) {
  const int E = (int)elen.size();
  const long long Wl = (S + 31) / 32;
  WorkItems w;
  w.off.assign(E + 1, 0);
  w.g.resize(E);
  for (int e = 0; e < E; e++) {
    const double lam = Omega * (double)elen[e];
    const double h = std::max(1e-6, 1.0 - std::exp(-lam) * (1.0 + lam));
    long long g = (long long)std::ceil(96.0 / (32.0 * h));
    g = std::max(1LL, std::min<long long>(std::min<long long>(g, 32), Wl));
    w.g[e] = (int)g;
    w.off[e + 1] = w.off[e] + (Wl + g - 1) / g;
  }
  return w;
}

template <typename Real>
struct TreeDev {
  pm::host::Schedule sch;
  long long S = 0, TS = 0;
  DevBuf cl_entries, cl_warp_off, cl_top_entries, cl_top_off, cd_top, cd_top_off, cd_entries, cd_warp_off, cd_tips;  // clade schedule
  DevBuf up_entries, up_off, down_entries, down_off, e_parent, e_child, e_len, maps_off, maps_len, cap_off;
  DevBuf tipcode, node_state, meta, PL, rec_len[2], rec_st[2], dw_partial, hard_ballot, wk_off, wk_g, wk_item, rec_cursor, shape;
  long long wk_total = 0, dw_rows = 0;
  int hard_blocks = 0;
  int pl_slots = 0;          // 32-site slots of the partials buffer (fused prune + node-draw kernel: SMs x resident blocks per SM); 0: separate kernels, partials of all sites
  int slots_per_sm = 0;
  DevBuf slot_busy;          // one flag per slot
  long long pl_sites = 0;    // sites per node row of the partials buffer: 32 pl_slots, or S
  int rec_shift = 0;         // production path records: 2^rec_shift consecutive sites share a slice
  // few sites on a tree whose per-site state fits shared memory (pm_small.cuh): a block per site runs the whole sweep, and
  // for the fixed-Q samplers all the sweeps of a call, in one launch
  bool small_ok = false;
  bool small_two = false;    // more sites than SMs: two blocks per SM (128 registers) instead of one
  int small_chunks = 0;      // record chunks (rows of rec_cursor)
  DevBuf small_down, small_part, small_cnt, small_root, small_border;
  DevBuf tip_stage;          // staging of the tip-state upload (create() only)
  int small_cap = 0;         // sweeps the output buffers hold
  int small_order_n = 0;     // entries of small_border
  long long rec_groups = 0;
  DevBuf e_len_d, TP, ll_partial;  // DIC samplers: branch lengths in FP64, exp(Q t_e) per branch, block partials of log p(y|Q)
  std::vector<int> cap_off_h;
  pm::ChainParams<Real> P;
  dim3 paths_grid;
  int chunk = 0;
  long long nblocks = 0;
};

template <typename Real>
struct ChainT : pm_chain {
  Variant V;
  int n = 0, ntrees = 0, N_total = 0, iters_done = 0, W = 0, WR = 0, ncols = 0;  // W statistics per row; WR = W + 1: row stride (error slot last)
  pm::host::NcclApi::Comm nccl = nullptr;
  int NS = 0;  // compile-time state count used for dispatch (2, 4 or 0)
  bool exact = false;
  double* Q = nullptr;  // caller's
  double* B = nullptr;  // caller's
  std::vector<double> pid, prior;
  double Omega = 0;
  pm_options opt;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  std::vector<std::unique_ptr<TreeDev<Real>>> trees;
  int jcap = 0;
  DevBuf model, cnt, root_out, err_flag, rows, tab_off, tab_u, q_dev;
  double* q_h = nullptr;  // pinned: Q row-major, for the DIC log-likelihood
  std::vector<double> own_B;                    // EXP: B = I + Q / Omega is internal (the entry takes no B)
  std::vector<double> eig_L, eig_R, eig_d;      // EXP: row-major eigenvectors, inverse, eigenvalues
  DevBuf eig_dev;
  Real* model_h = nullptr;   // pinned staging: model then ppow
  double* rows_h = nullptr;  // pinned: ntrees * W
  double* rows_h_dev = nullptr;  // the same buffer as the device sees it (mapped pinned memory)
  unsigned* err_h = nullptr;
  std::vector<double> scale_prev, rate_prev;
  pm::host::MersenneR mt{0};
  std::unique_ptr<pm::host::ReplaySource> replay;
  size_t smem_prune = 0, smem_nodes = 0, smem_paths = 0;
  int rows_cap = 0;
  int debug_kernel = 0;
  struct Timed { cudaEvent_t a, b; int k; };
  std::vector<Timed> timed;
  // CUDA-graph replay of one sweep (fixed-Q samplers on small problems: a sweep of a 100-tip tree is seven launches of a
  // few microseconds each, and the host cannot issue them as fast as the GPU retires them).  The sweep index and the
  // output row live in device memory (ChainParams::ctl), so one instantiated graph serves every sweep of the chain.
  DevBuf ctl, phase_ns;               // phase_ns: block-nanoseconds the fused kernel spent pruning / drawing nodes (timing on)
  uint32_t* ctl_h = nullptr;          // pinned
  cudaGraphExec_t sweep_graph = nullptr;
  void* graph_rows = nullptr;         // the rows buffer the graph writes to (re-captured if it moves)
  bool capturing = false;
  int launches_per_sweep = 0;
  Switches sw;

  ~ChainT() override {
    cudaSetDevice(opt.device);
    cudaDeviceSynchronize();
    for (auto& t : timed) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
    if (model_h) cudaFreeHost(model_h);
    if (rows_h) cudaFreeHost(rows_h);
    if (err_h) cudaFreeHost(err_h);
    if (q_h) cudaFreeHost(q_h);
    if (ctl_h) cudaFreeHost(ctl_h);
    if (sweep_graph) cudaGraphExecDestroy(sweep_graph);
    if (own_stream && stream) cudaStreamDestroy(stream);
  }

  pm::host::UniformSource& host_rng() { return replay ? static_cast<pm::host::UniformSource&>(*replay) : mt; }

  size_t model_elems() const { return (size_t)2 * n * n + 5 * n; }
  // the table of powers follows the model in ONE device buffer (one upload per sweep of a rate-updating sampler), 16-byte aligned
  size_t model_stride() const { return (model_elems() + 3) & ~(size_t)3; }

  // ---- model upload: B, thresholded B, pid, scales, table of powers ----
  void stage_model(bool first) {
    std::vector<double> Bd((size_t)n * n), Bs((size_t)n * n);
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) {
        const double v = B[i + (size_t)j * n];
        Bd[(size_t)i * n + j] = v;
        Bs[(size_t)i * n + j] = (V.sparse && !(v > 1e-7)) ? 0.0 : v;  // matTospmat keeps entries > 1e-7 (:811)
      }
    std::vector<double> scale_new(n);
    for (int s = 0; s < n; s++) scale_new[s] = 1.0 / (Omega + Q[s + (size_t)s * n]);
    std::vector<double> rate_new(n);
    for (int s = 0; s < n; s++) rate_new[s] = Omega + Q[s + (size_t)s * n];
    if (first) { scale_prev = scale_new; rate_prev = rate_new; }
    Real* m = model_h;
    for (size_t i = 0; i < (size_t)n * n; i++) { m[i] = (Real)Bd[i]; m[(size_t)n * n + i] = (Real)Bs[i]; }
    Real* v = m + 2 * (size_t)n * n;
    for (int s = 0; s < n; s++) {
      v[s] = (Real)pid[s]; v[n + s] = (Real)scale_prev[s]; v[2 * n + s] = (Real)scale_new[s];
      v[3 * n + s] = (Real)rate_prev[s]; v[4 * n + s] = (Real)rate_new[s];
    }
    scale_prev = scale_new; rate_prev = rate_new;
    // P_0 = I, P_j = Bs P_{j-1}: left-to-right dot products in double (column c of P_j is the reference's
    // backward vector B^j e_c bit for bit, src/phylomap.cpp:283-287)
    Real* pw = m + model_stride();
    std::vector<double> cur((size_t)n * n, 0.0), nxt((size_t)n * n);
    for (int i = 0; i < n; i++) cur[(size_t)i * n + i] = 1.0;
    for (int j = 0; j < jcap; j++) {
      for (size_t i = 0; i < (size_t)n * n; i++) pw[(size_t)j * n * n + i] = (Real)cur[i];
      if (j + 1 < jcap) {
        for (int r = 0; r < n; r++)
          for (int c = 0; c < n; c++) {
            double acc = 0;
            for (int l = 0; l < n; l++) acc = acc + Bs[(size_t)r * n + l] * cur[(size_t)l * n + c];
            nxt[(size_t)r * n + c] = acc;
          }
        cur.swap(nxt);
      }
    }
    CK(cudaMemcpyAsync(model.p, m, (model_stride() + (size_t)jcap * n * n) * sizeof(Real), cudaMemcpyHostToDevice, stream));
  }

  // ---- kernel dispatch ----
  // the production arithmetic for n = 2 / 4 has kernels of its own (pm::Sweep::production)
  bool production() const { return !exact && (NS == 2 || NS == 4); }
  // f(std::integral_constant<int, NS>) with the chain's compile-time state count: 2, 4, or 0 (run-time n)
  template <typename F>
  auto with_ns(F&& f) const {
    if (NS == 2) return f(std::integral_constant<int, 2>{});
    if (NS == 4) return f(std::integral_constant<int, 4>{});
    return f(std::integral_constant<int, 0>{});
  }
  // ... and f(ns, std::bool_constant<EXACT>): the deterministic kernels exist in FP64 only
  template <typename F>
  auto with_ns_exact(F&& f) const {
    if constexpr (std::is_same_v<Real, double>)
      if (exact) return with_ns([&](auto ns) { return f(ns, std::true_type{}); });
    return with_ns([&](auto ns) { return f(ns, std::false_type{}); });
  }

  template <int NSc, bool EX>
  void launch_sweep_t(TreeDev<Real>& t, uint32_t iter, double* row) {
    if (!EX && use_small(t)) { launch_small(t, iter, 1, row); launches_per_sweep = t.S == 1 ? 1 : 2; return; }
    const uint32_t* ctl_d = capturing ? ctl.as<uint32_t>() : nullptr;
    {
      pm::ChainParams<Real> P = t.P;
      P.ctl = ctl_d;
      const int gx = (int)((t.S + 31) / 32);
      if (t.pl_slots) {  // K1 + K2 in one launch; with timing on, the blocks report the time they spend in each pass
        begin_timed(4);
        pm::Sweep<Real, NSc, EX>::prune_nodes(P, gx, smem_nodes, stream, iter, 0, 3, t.slots_per_sm ? t.slot_busy.template as<int>() : nullptr,
                                              t.slots_per_sm, timing ? phase_ns.as<unsigned long long>() : nullptr);
        end_timed();
      } else {
        begin_timed(0);
        pm::Sweep<Real, NSc, EX>::prune(P, gx, smem_prune, stream);
        end_timed();
        begin_timed(1);
        pm::Sweep<Real, NSc, EX>::nodes(P, gx, smem_nodes, stream, iter);
        end_timed();
      }
    }
    begin_timed(2);
    if (!EX) CK(cudaMemsetAsync(t.rec_cursor.p, 0, t.rec_cursor.bytes, stream));  // (inside K3's timed region: it is part of the step)
    {
      pm::ChainParams<Real> P = t.P;
      P.ctl = ctl_d;
      // (a captured sweep serves every index: its kernels take `first` from the index they read, and the short-shape
      // kernel, which has nothing to do in a first sweep, is always part of it)
      pm::Sweep<Real, NSc, EX>::paths(P, t.paths_grid, smem_paths, stream, iter, (iter == 0 && !capturing) ? 1 : 0, t.chunk, t.hard_blocks);
    }
    end_timed();
    begin_timed(3);
    pm::k_reduce<<<1, 256, 0, stream>>>(t.dw_partial.template as<double>(), t.dw_rows, n, cnt.as<unsigned long long>(),
                                        root_out.as<int>(), row, 0, err_flag.as<unsigned>(), W, capturing ? ctl.as<uint32_t>() : nullptr, WR);
    end_timed();
    launches_per_sweep = (t.pl_slots ? 1 : 2) + (exact ? 2 : (iter == 0 && !capturing) ? 3 : 4);
    if (!capturing) launches += launches_per_sweep;
  }
  // Few sites on a small tree: sweeps [iter0, iter0 + nsweeps) of every site in one launch, a block per site, the state in
  // shared memory (pm_small.cuh); a second launch sums the sites and assembles the rows (WR doubles per sweep, from rows_d).
  bool use_small(const TreeDev<Real>& t) const { return t.small_ok && !timing && !sw.debug_sync && !capturing; }
  void launch_small(TreeDev<Real>& t, uint32_t iter0, int nsweeps, double* rows_d) {
    const long long S = t.S;
    pm::SmallOut o;
    o.down = reinterpret_cast<const int4*>(t.small_down.p); o.down_off = t.down_off.template as<int>();
    o.n_down_levels = (int)t.sch.down_off.size() - 1; o.n_chunks = t.small_chunks;
    o.br_order = t.small_border.template as<int>(); o.n_order = t.small_order_n;
    o.part = nullptr; o.cnt = nullptr; o.root = nullptr; o.rows = nullptr; o.row_stride = WR; o.err_slot = W;
    auto launch = [&](uint32_t it0, int nb) {
      with_ns([&](auto ns) { pm::Sweep<Real, decltype(ns)::value, false>::small_chain(t.P, (int)S, stream, it0, nb, o, t.small_two); });
    };
    if (S == 1) {  // the one block writes the rows itself: one launch, whatever the number of sweeps
      o.rows = rows_d;
      launch(iter0, nsweeps);
      launches += 1;
      return;
    }
    const int batch = (int)std::max<long long>(1, std::min<long long>(nsweeps, (64LL << 20) / (S * n * (long long)sizeof(double))));
    if (t.small_cap < batch) {
      t.small_part.alloc((size_t)batch * S * n * sizeof(double));
      t.small_cnt.alloc((size_t)batch * n * n * sizeof(unsigned long long));
      t.small_root.alloc((size_t)batch * sizeof(int));
      t.small_cap = batch;
      CK(cudaMemsetAsync(t.small_cnt.p, 0, t.small_cnt.bytes, stream));   // (k_small_reduce hands them back zeroed)
      CK(cudaMemsetAsync(t.small_root.p, 0, t.small_root.bytes, stream));
    }
    o.part = t.small_part.template as<double>(); o.cnt = t.small_cnt.template as<unsigned long long>(); o.root = t.small_root.template as<int>();
    for (int b0 = 0; b0 < nsweeps; b0 += batch) {
      const int nb = std::min(batch, nsweeps - b0);
      launch(iter0 + (uint32_t)b0, nb);
      pm::k_small_reduce<<<nb, 128, 0, stream>>>(o.part, o.cnt, o.root, S, n, rows_d + (size_t)b0 * WR, WR, err_flag.as<unsigned>(), W);
      launches += 2;
    }
  }
  // DIC samplers: log p(y | Q) of the current Q into row[n + n*n + 1] (after the sweep: PL is free again)
  void launch_loglik(TreeDev<Real>& t, double* row) {
    for (int i = 0; i < n; i++) for (int j = 0; j < n; j++) q_h[(size_t)i * n + j] = Q[i + (size_t)j * n];
    CK(cudaMemcpyAsync(q_dev.p, q_h, (size_t)n * n * sizeof(double), cudaMemcpyHostToDevice, stream));
    const int E = t.sch.E;
    pm::k_transprob<Real><<<(E + 127) / 128, 128, 0, stream>>>(q_dev.as<double>(), t.e_len_d.template as<double>(), E, n,
                                                              t.TP.template as<Real>());
    const int gx = (int)((t.S + 31) / 32);
    with_ns([&](auto ns) {
      pm::k_loglik<Real, decltype(ns)::value><<<gx, 256, 0, stream>>>(t.P, t.TP.template as<Real>(), t.ll_partial.template as<double>(), nullptr);
    });
    pm::k_reduce_ll<<<1, 256, 0, stream>>>(t.ll_partial.template as<double>(), gx, row + n + n * n + 1);
    launches += 3;
  }

  // the pruning pass alone: over all site tiles, or over the one tile that holds `only_site`
  template <int NSc, bool EX>
  void launch_prune_t(TreeDev<Real>& t, long long only_site) {
    const long long nb = (t.S + 31) / 32;
    if (t.pl_slots) {  // the pruning pass of the fused kernel: all site blocks, or the one that holds `only_site` (it lands in slot 0)
      if (only_site >= 0) pm::Sweep<Real, NSc, EX>::prune_nodes(t.P, 1, smem_nodes, stream, 0u, only_site / 32, 1, nullptr, 0, nullptr);
      else pm::Sweep<Real, NSc, EX>::prune_nodes(t.P, (int)nb, smem_nodes, stream, 0u, 0, 1, t.slots_per_sm ? t.slot_busy.template as<int>() : nullptr,
                                                 t.slots_per_sm, nullptr);
    } else pm::Sweep<Real, NSc, EX>::prune(t.P, (int)nb, smem_prune, stream);
    launches++;
  }

  void launch_sweep(TreeDev<Real>& t, uint32_t iter, double* row) {
    with_ns_exact([&](auto ns, auto ex) { launch_sweep_t<decltype(ns)::value, decltype(ex)::value>(t, iter, row); });
  }
  void launch_prune(TreeDev<Real>& t, long long only_site = -1) {
    with_ns_exact([&](auto ns, auto ex) { launch_prune_t<decltype(ns)::value, decltype(ex)::value>(t, only_site); });
  }

  void begin_timed(int k) {
    debug_kernel = k;
    if (!timing) return;
    Timed t; t.k = k;
    CK(cudaEventCreate(&t.a)); CK(cudaEventCreate(&t.b));
    CK(cudaEventRecord(t.a, stream));
    timed.push_back(t);
  }
  void end_timed() {
    if (timing) CK(cudaEventRecord(timed.back().b, stream));
    if (sw.debug_sync) {  // PHYLOMAP_B200_DEBUG_SYNC=1: stop at the first kernel that raises a device error flag
      try { check_device_errors(); }
      catch (Fail& f) { f.msg += " [raised by sweep kernel #" + std::to_string(debug_kernel) + ": 0 prune, 1 nodes, 2 paths, 3 reduce]"; throw; }
    }
  }
  void collect_timed() {
    double fused = 0;
    for (auto& t : timed) {
      float ms = 0;
      cudaEventElapsedTime(&ms, t.a, t.b);
      if (t.k == 4) fused += ms; else kernel_ms[t.k] += ms;
      cudaEventDestroy(t.a); cudaEventDestroy(t.b);
    }
    timed.clear();
    if (fused > 0) {  // the fused kernel's time goes to the two passes in proportion to the block-time spent in each
      unsigned long long ns[2] = {0, 0};
      cudaMemcpy(ns, phase_ns.p, sizeof ns, cudaMemcpyDeviceToHost);
      cudaMemset(phase_ns.p, 0, sizeof ns);
      const double tot = (double)ns[0] + (double)ns[1];
      const double share = tot > 0 ? (double)ns[0] / tot : 0.5;
      kernel_ms[0] += fused * share;
      kernel_ms[1] += fused * (1.0 - share);
    }
  }

  void check_device_errors() {
    CK(cudaMemcpyAsync(err_h, err_flag.p, sizeof(unsigned), cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    const unsigned f = *err_h;
    if (!f) return;
    if (f & PM_DE_BAD_STATE) fail(PM_ERR_ARG, "tip states must lie in 1..n");
    if (f & PM_DE_SAMPLE_NA) fail(PM_ERR_SAMPLE, "NAs not allowed in probability");
    if (f & PM_DE_SAMPLE_NEG) fail(PM_ERR_SAMPLE, "Negative probabilities not allowed");
    if (f & PM_DE_SAMPLE_ZERO)
      fail(PM_ERR_SAMPLE, opt.precision == PM_F32 ? "Not enough positive probabilities (FP32 partial likelihoods span ~1e-45: on large trees with "
                                                      "one-piece branches this can be an underflow; precision f64 has the reference's range)"
                                                    : "Not enough positive probabilities");
    if (f & PM_DE_REPLAY) fail(PM_ERR_REPLAY, "replay table exhausted");
    if (f & PM_DE_JUMP_LIMIT)
      fail(PM_ERR_CAPACITY, "a branch carries more than 63 state changes at one site: the deterministic mode holds at most 64 runs "
                            "per path (the production arithmetic has no such limit)");
    if (f & PM_DE_PATH_CAP) fail(PM_ERR_CAPACITY, "the run records of a branch chunk overflowed; raise pm_options.path_capacity");
    if (f & PM_DE_M_OVERFLOW) fail(PM_ERR_CAPACITY, "more than 65535 pieces on one branch");
    if (f & PM_DE_ZERO_LIK)
      fail(PM_ERR_SAMPLE, opt.precision == PM_F32 ? "the tip data of a site have zero likelihood under Q, or FP32 products underflowed "
                                                      "(precision f64 has the wider range): no posterior expectation exists"
                                                    : "the tip data of a site have zero likelihood under Q: no posterior expectation exists");
    fail(PM_ERR_CUDA, "inconsistent chain state (device flag %u)", f);
  }

  // ---- construction ----
  void create(int variant, const pm_tree* tr, int ntr, int n_, double* Q_, const double* pid_, double* B_, double Om,
              const double* prior_, int nprior, int Ntot, const pm_options* o) {
    V = variant_of(variant);
    n = n_; ntrees = ntr; N_total = Ntot; Q = Q_; B = B_; Omega = Om;
    opt = *o;
    sw = read_switches();
    PhaseTrace trace{sw.trace};
    std::vector<pm::host::Schedule> schedules = validate(variant, tr, pid_, prior_, nprior);
    trace.mark("validation + schedules");
    const int sms = open_device();
    trace.mark("device queries + stream");
    err_flag.alloc(sizeof(unsigned));
    CK(cudaMemsetAsync(err_flag.p, 0, err_flag.bytes, stream));
    // a second stream for the upload of the tip states (the largest transfer of create()): everything else -- schedule
    // uploads, the set-up kernels -- goes on `stream` meanwhile; the two are joined before create() returns
    cudaStream_t aux = nullptr;
    cudaEvent_t ev_a = nullptr, ev_b = nullptr;
    struct AuxGuard {
      cudaStream_t& s; cudaEvent_t& a; cudaEvent_t& b;
      ~AuxGuard() { if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); } if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
    } aux_guard{aux, ev_a, ev_b};
    CK(cudaStreamCreateWithFlags(&aux, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&ev_a, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ev_b, cudaEventDisableTiming));
    CK(cudaEventRecord(ev_a, stream));   // (the error flag is zeroed on `stream`)
    CK(cudaStreamWaitEvent(aux, ev_a, 0));
    double tmax = 0;
    for (int ti = 0; ti < ntr; ti++) trees.push_back(create_tree(tr[ti], ti, std::move(schedules[ti]), sms, aux, tmax, trace));

    alloc_model_and_host_buffers(tmax);
    if (opt.rng == PM_RNG_TABLE) upload_replay_table();
    mt.reseed((uint32_t)opt.seed);
    trace.mark("pinned buffers, replay table");
    // shared-memory sizes
    const int np_fast = production() ? std::min(PM_SMEM_POW, jcap) : 0;
    smem_prune = (size_t)n * n * sizeof(Real);
    smem_nodes = ((size_t)n * n + 3 * n + (size_t)np_fast * n * n) * sizeof(Real);
    smem_paths = (size_t)4 * n * sizeof(double) + ((size_t)n * n + ((n * n) & 1)) * sizeof(unsigned) +
                 ((size_t)2 * n * n + 5 * n + (size_t)np_fast * n * n) * sizeof(Real);

    for (int ti = 0; ti < ntr; ti++) {
      TreeDev<Real>& t = *trees[ti];
      fill_params(t, ti);
      // (the jump-count / shape words of every branch-site -- 15 GB of writes at the benchmark size -- do not depend on the
      // tip states, which are still on their way on the second stream)
      const pm::ChainParams<Real>& P = t.P;
      if (!V.exp && !V.llonly)
        pm::k_init_meta<Real><<<dim3((unsigned)((t.S + 255) / 256), (unsigned)std::min(P.E, 65535)), 256, 0, stream>>>(P.maps_off, P.maps_len, t.S, P.E, P.meta,
                                                                                                                         P.e_len, exact ? nullptr : P.shape);
      trace.mark("set-up kernels issued");
      CK(cudaGetLastError());
    }
    CK(cudaEventRecord(ev_b, aux));          // join: the tip states of every tree are in place
    CK(cudaStreamWaitEvent(stream, ev_b, 0));
    stage_model(true);
    if (V.exp) {
      std::vector<double> eg;
      eg.insert(eg.end(), eig_L.begin(), eig_L.end());
      eg.insert(eg.end(), eig_R.begin(), eig_R.end());
      eg.insert(eg.end(), eig_d.begin(), eig_d.end());
      upload(eig_dev, eg, stream);
      TreeDev<Real>& t = *trees[0];
      const int E = t.sch.E;
      const double* g = eig_dev.as<double>();
      pm::k_transprob_eig<Real><<<(E + 127) / 128, 128, 0, stream>>>(g, g + (size_t)n * n, g + (size_t)2 * n * n,
                                                                    t.e_len_d.template as<double>(), E, n, t.TP.template as<Real>());
      CK(cudaGetLastError());
    }
    check_device_errors();
    for (auto& t : trees) t->tip_stage.alloc(0);   // (everything is on the device now)
    trace.mark("tip states: H2D + transpose, init kernels, sync");
  }

  // The checks of the arguments and the trees that need no device (malformed input is reported as PM_ERR_ARG even where
  // no device exists); sets the chain's shape and returns the trees' schedules.
  std::vector<pm::host::Schedule> validate(int variant, const pm_tree* tr, const double* pid_, const double* prior_, int nprior) {
    const int ntr = ntrees;
    if (n < 2 || n > PM_NMAX) fail(PM_ERR_ARG, "number of states must be in 2..%d", PM_NMAX);
    if (!V.multi && ntr != 1) fail(PM_ERR_ARG, "this sampler takes exactly one tree");
    if (ntr < 1) fail(PM_ERR_ARG, "no trees");
    if (N_total < 0) fail(PM_ERR_ARG, "N must be non-negative");
    if (V.hidden && (n < 4 || (n & 1))) fail(PM_ERR_ARG, "hidden-rate samplers need an even number of states >= 4");
    if (V.two_state && n != 2) fail(PM_ERR_ARG, "this sampler is 2-state only");
    if (V.dic && n > PM_DIC_NMAX) fail(PM_ERR_ARG, "the DIC samplers support at most %d states", PM_DIC_NMAX);
    const int need_prior = V.two_state ? 4 : variant == PM_V_KSMT ? 8 : V.hidden ? 6 : 0;
    if (nprior < need_prior || (need_prior && !prior_)) fail(PM_ERR_ARG, "prior needs %d values", need_prior);
    if (need_prior) prior.assign(prior_, prior_ + nprior);
    pid.assign(pid_, pid_ + n);
    exact = opt.mode == PM_MODE_DETERMINISTIC;
    if (exact && opt.precision != PM_F64) fail(PM_ERR_ARG, "deterministic mode computes in FP64");
    if (exact && V.exp) fail(PM_ERR_ARG, "the direct sampler (maketreelistEXP) runs in production arithmetic only");
    if (opt.rng == PM_RNG_TABLE && (!opt.tab_off || !opt.tab_u)) fail(PM_ERR_ARG, "replay table missing");
    if (opt.rng == PM_RNG_TABLE && !exact) fail(PM_ERR_ARG, "the replay table feeds the deterministic mode only");
    if (opt.rng == PM_RNG_TABLE && (opt.site_offset != 0 || opt.allreduce || opt.nccl_world > 1)) fail(PM_ERR_ARG, "replay runs are single-process");
    if (opt.allreduce && !opt.cuda_stream)
      fail(PM_ERR_ARG, "an allreduce callback needs pm_options.cuda_stream: the collective must be ordered on the stream the chain launches on");
    if (opt.allreduce && opt.nccl_world > 1) fail(PM_ERR_ARG, "give either an allreduce callback or an NCCL clique, not both");
    if (opt.nccl_world > 1 && (!opt.nccl_id || opt.nccl_rank < 0 || opt.nccl_rank >= opt.nccl_world)) fail(PM_ERR_ARG, "bad NCCL clique (nccl_id / nccl_rank / nccl_world)");
    NS = (n == 2) ? 2 : (n == 4) ? 4 : 0;
    W = n + n * n + 1 + (V.dic ? 1 : 0);
    WR = W + 1;
    ncols = ncols_of(variant, n);

    if (!(Omega > 0)) fail(PM_ERR_ARG, "Omega must be positive");
    std::vector<pm::host::Schedule> schedules(ntr);
    for (int ti = 0; ti < ntr; ti++) {
      const pm_tree& x = tr[ti];
      if (x.n_tips != tr[0].n_tips || x.n_edges != tr[0].n_edges) fail(PM_ERR_ARG, "all trees must have the same number of tips");
      if (x.n_sites < 1 || x.n_sites != tr[0].n_sites) fail(PM_ERR_ARG, "n_sites must be >= 1 and equal across trees");
      if (x.n_sites >= (1LL << 31)) fail(PM_ERR_ARG, "at most 2^31 - 1 sites per process");
      if (!x.edge || !x.nen || !x.nodelist || !x.maps_off || !x.maps_len) fail(PM_ERR_ARG, "tree %d: missing field", ti);
      if (!x.states && !x.states_u8) fail(PM_ERR_ARG, "tree %d: states missing", ti);
      try {
        pm::host::build_schedule(x.n_tips, x.n_edges, x.edge, x.nen, x.nodelist, x.root, V.redraw_tips, schedules[ti]);
      } catch (const std::string& msg) { fail(PM_ERR_ARG, "tree %d: %s", ti, msg.c_str()); }
      if (x.maps_off[0] != 0) fail(PM_ERR_ARG, "tree %d: maps_off[0] must be 0", ti);
      for (int e = 0; e < x.n_edges; e++) {
        const long long a = x.maps_off[e], b = x.maps_off[e + 1];
        if (b <= a) fail(PM_ERR_ARG, "tree %d: branch %d has no segments", ti, e + 1);
        if (b - a > 65535) fail(PM_ERR_ARG, "tree %d: branch %d has more than 65535 segments", ti, e + 1);
        for (long long p = a; p < b; p++) {
          if (!(x.maps_len[p] >= 0)) fail(PM_ERR_ARG, "tree %d: negative or NA segment length", ti);
          if (x.maps_state && (x.maps_state[p] < 1 || x.maps_state[p] > n)) fail(PM_ERR_ARG, "tree %d: mapnames out of range", ti);
        }
      }
    }
    return schedules;
  }

  // Selects and checks the device, sets up the chain's stream; returns the number of SMs.
  int open_device() {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) fail(PM_ERR_CUDA, "no CUDA device (there is no CPU fallback)");
    if (opt.device < 0 || opt.device >= ndev) fail(PM_ERR_CUDA, "device %d not present", opt.device);
    CK(cudaSetDevice(opt.device));
    // (three attributes, not cudaGetDeviceProperties: that call reads every property of the device and takes 10-150 ms,
    // a quarter of a short call)
    int major = 0, minor = 0, sms = 0;
    CK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, opt.device));
    CK(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, opt.device));
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, opt.device));
    if (major != 10) fail(PM_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", opt.device, major, minor);
    if (opt.cuda_stream) stream = (cudaStream_t)opt.cuda_stream;
    else { CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking)); own_stream = true; }
    return sms;
  }

  // One tree's device state: tip upload on `aux` first, then the plan, the schedules and the buffers on `stream`.
  // tmax: the longest branch so far.
  std::unique_ptr<TreeDev<Real>> create_tree(const pm_tree& x, int ti, pm::host::Schedule&& sch, int sms, cudaStream_t aux,
                                             double& tmax, PhaseTrace& trace) {
    std::unique_ptr<TreeDev<Real>> tp(new TreeDev<Real>());
    TreeDev<Real>& t = *tp;
    t.sch = std::move(sch);
    t.S = x.n_sites;
    t.TS = (t.S + 15) / 16 * 16;  // tip-code rows are padded: every row starts 16-byte aligned whatever S is
    const int E = x.n_edges, T = x.n_tips;
    const long long S = t.S;
    const bool no_paths = V.exp || V.llonly;  // log-likelihood-only and direct-sampler chains keep no path state
    upload_tips(t, x, aux);
    std::vector<long long> moff(x.maps_off, x.maps_off + E + 1);
    std::vector<Real> elen(E);
    for (int e = 0; e < E; e++) {
      double tot = 0;
      for (long long p = moff[e]; p < moff[e + 1]; p++) tot = tot + x.maps_len[p];
      elen[e] = (Real)tot;
      tmax = std::max(tmax, tot);
    }
    std::vector<double> mlen(x.maps_len, x.maps_len + moff[E]);

    const size_t small_smem = with_ns([&](auto ns) { return pm::Sweep<Real, decltype(ns)::value, false>::small_smem(T); });
    const SmallChoice small = choose_small_kernel(production() && !no_paths && opt.rng != PM_RNG_TABLE, elen,
                                                  Omega, T, S, sms, small_smem, sw);
    t.small_ok = small.ok;
    t.small_two = small.two;
    const bool pooled_ok = !t.small_ok && !exact && !no_paths && sw.rec_pool;
    RecordPlan rp = plan_records(pooled_ok ? 5 : 0, elen, moff, S, Omega, exact, no_paths, opt.path_capacity);
    if (!rp.fits) rp = plan_records(0, elen, moff, S, Omega, exact, no_paths, opt.path_capacity);
    t.rec_shift = rp.rec_shift;
    t.rec_groups = (S + (1LL << t.rec_shift) - 1) >> t.rec_shift;
    t.chunk = rp.chunk;
    t.paths_grid = dim3((unsigned)rp.gx, (unsigned)rp.ny, 1);
    t.nblocks = rp.gx * rp.ny;
    t.small_chunks = (int)rp.ny;
    t.cap_off_h = std::move(rp.cap_off);
    trace.mark("record capacities");

    plan_partials_slots(t, sms);
    upload(t.up_entries, t.sch.up_entries, stream);
    upload(t.up_off, t.sch.up_off, stream);
    if (production()) {
      CladeCode cc = encode_clade_schedule(t.sch, S, t.TS, (long long)t.pl_sites * n * (long long)sizeof(Real), V.redraw_tips);
      upload(t.cl_entries, cc.e16, stream);
      upload(t.cl_warp_off, cc.cs.warp_off, stream);
      upload(t.cl_top_entries, cc.top, stream);
      upload(t.cl_top_off, cc.cs.top_off, stream);
      upload(t.cd_entries, cc.d16, stream);
      upload(t.cd_warp_off, cc.cs.down_warp_off, stream);
      upload(t.cd_top, cc.cs.down_top, stream);
      upload(t.cd_top_off, cc.cs.down_top_off, stream);
      upload(t.cd_tips, cc.tips, stream);
      t.P.n_cl_top_levels = (int)cc.cs.top_off.size() - 1;
      t.P.n_cd_top_levels = (int)cc.cs.down_top_off.size() - 1;
      t.P.n_cd_tips = (int)cc.tips.size() / 2;
      if (t.small_ok) {
        const SmallOrder so = small_draw_order(t.sch, cc.cs, elen);
        upload(t.small_down, so.down, stream);
        upload(t.small_border, so.border, stream);
        t.small_order_n = (int)so.border.size();
      }
    }
    upload(t.down_entries, t.sch.down_entries, stream);
    upload(t.down_off, t.sch.down_off, stream);
    upload(t.e_parent, t.sch.e_parent, stream);
    upload(t.e_child, t.sch.e_child, stream);
    upload(t.e_len, elen, stream);
    if (V.dic || V.exp) {
      std::vector<double> eld(E);
      for (int e = 0; e < E; e++) eld[e] = x.edge_length ? x.edge_length[e] : (double)elen[e];
      if (x.edge_length) for (int e = 0; e < E; e++) if (!(eld[e] >= 0)) fail(PM_ERR_ARG, "tree %d: negative or NA edge.length", ti);
      upload(t.e_len_d, eld, stream);
      t.TP.alloc((size_t)E * n * n * sizeof(Real));
      t.ll_partial.alloc((size_t)((S + 31) / 32) * sizeof(double));
    }
    trace.mark("clade schedules + uploads");
    alloc_path_state(t, moff, mlen, elen, sms);
    trace.mark("device buffers");
    return tp;
  }

  // The tip states start their way over PCIe FIRST: [S][T] rows staged in blocks and transposed to [T][S] on the device,
  // all asynchronous on the second stream, so that the host work of create() (record capacities, schedules) and the
  // set-up kernels run while they travel.  (The staging buffer is kept until the end of create(): the pool must not hand
  // it out again.)
  void upload_tips(TreeDev<Real>& t, const pm_tree& x, cudaStream_t aux) {
    const int T = x.n_tips;
    t.tipcode.alloc((size_t)T * t.TS);
    CK(cudaMemsetAsync(t.tipcode.p, 0, t.tipcode.bytes, aux));
    t.node_state.alloc((size_t)(2 * T - 1) * t.S);
    CK(cudaMemsetAsync(t.node_state.p, 0, t.node_state.bytes, aux));
    const size_t esz = x.states_u8 ? 1 : 4;
    long long rows_per = std::max<long long>(32, (256LL << 20) / ((long long)T * (long long)esz));
    rows_per = std::min<long long>(rows_per, std::min<long long>(t.S, 32LL * 65535));
    t.tip_stage.alloc((size_t)rows_per * T * esz);
    for (long long s0 = 0; s0 < t.S; s0 += rows_per) {
      const int ns = (int)std::min<long long>(rows_per, t.S - s0);
      const void* src = x.states_u8 ? (const void*)(x.states_u8 + s0 * T) : (const void*)(x.states + s0 * T);
      CK(cudaMemcpyAsync(t.tip_stage.p, src, (size_t)ns * T * esz, cudaMemcpyHostToDevice, aux));
      dim3 g((T + 31) / 32, (ns + 31) / 32), b(32, 8);
      if (x.states_u8)
        pm::k_init_tips<uint8_t><<<g, b, 0, aux>>>(t.tip_stage.template as<uint8_t>(), ns, s0, t.S, t.TS, T, n, V.parity_tips,
                                                     t.tipcode.template as<uint8_t>(), t.node_state.template as<uint8_t>(), err_flag.as<unsigned>());
      else
        pm::k_init_tips<int32_t><<<g, b, 0, aux>>>(t.tip_stage.template as<int32_t>(), ns, s0, t.S, t.TS, T, n, V.parity_tips,
                                                     t.tipcode.template as<uint8_t>(), t.node_state.template as<uint8_t>(), err_flag.as<unsigned>());
    }
    CK(cudaGetLastError());
  }

  // Partials are scratch between the pruning pass and the node draws of one sweep, and a block's partials are read by
  // nobody but the same block's node draws: the production kernels (n = 2, 4) run both passes in ONE kernel whose
  // blocks keep their partials in a slot of 32 sites, claimed for the life of the block (k_prune_nodes_clade): as many
  // slots per SM as blocks can be resident there (3 in FP32, 2 in FP64: the occupancy the runtime reports for the
  // smallest shared-memory configuration, an upper bound).  The DIC chains evaluate log p(y | Q) over all sites after
  // the sweep and keep the whole array, like the generic and the deterministic kernels.
  // PHYLOMAP_B200_FUSED=0: the two separate kernels and the full array (for comparison).
  void plan_partials_slots(TreeDev<Real>& t, int sms) {
    t.pl_slots = 0;
    t.pl_sites = t.S;
    if (!production() || V.dic || V.exp || V.llonly || !sw.fused) return;
    const size_t smem_lo = ((size_t)n * n + 3 * n) * sizeof(Real);
    const int per_sm = with_ns([&](auto ns) { return pm::Sweep<Real, decltype(ns)::value, false>::fused_blocks_per_sm(smem_lo); });
    if (per_sm < 1) fail(PM_ERR_CUDA, "cudaOccupancyMaxActiveBlocksPerMultiprocessor failed for the fused prune + node-draw kernel");
    t.slots_per_sm = per_sm;
    t.pl_slots = sm_id_range(opt.device, sms) * per_sm;  // slots are indexed by %smid
    t.pl_sites = 32LL * t.pl_slots;
    if (t.pl_sites >= ((t.S + 31) / 32) * 32) {  // fewer site blocks than slots: block i uses slot i
      t.pl_slots = (int)((t.S + 31) / 32); t.pl_sites = 32LL * t.pl_slots; t.slots_per_sm = 0;
    } else {
      t.slot_busy.alloc((size_t)t.pl_slots * sizeof(int));
      CK(cudaMemsetAsync(t.slot_busy.p, 0, t.slot_busy.bytes, stream));
    }
  }

  // The per-site state of the sweeps: piece counts, partials, path records, the general path kernel's work items and
  // the per-block partial sums.
  void alloc_path_state(TreeDev<Real>& t, const std::vector<long long>& moff, const std::vector<double>& mlen,
                        const std::vector<Real>& elen, int sms) {
    const int E = t.sch.E, T = t.sch.T;
    const long long S = t.S, R = t.cap_off_h.back();
    const bool no_paths = V.exp || V.llonly;
    upload(t.maps_off, moff, stream);
    upload(t.maps_len, mlen, stream);
    upload(t.cap_off, t.cap_off_h, stream);
    if (!no_paths) t.meta.alloc((size_t)E * S * sizeof(uint32_t));
    t.PL.alloc((size_t)(T - 1) * t.pl_sites * n * sizeof(Real));
    for (int b = 0; b < 2 && !no_paths; b++) {
      t.rec_len[b].alloc((size_t)R * t.rec_groups * sizeof(Real));
      t.rec_st[b].alloc((size_t)R * t.rec_groups);
    }
    if (!exact && !no_paths) {
      const long long Wl = (S + 31) / 32;
      t.hard_ballot.alloc((size_t)E * Wl * sizeof(uint32_t));
      const WorkItems w = build_work_items(elen, Omega, S);
      t.wk_total = w.off.back();
      upload(t.wk_off, w.off, stream);
      upload(t.wk_g, w.g, stream);
      t.wk_item.alloc((size_t)std::max<long long>(t.wk_total, 1) * sizeof(unsigned long long));
      pm::k_build_items<<<(unsigned)((t.wk_total + 255) / 256), 256, 0, stream>>>(t.wk_off.template as<long long>(), t.wk_g.template as<int>(), E, Wl,
                                                                                 t.wk_total, t.wk_item.template as<unsigned long long>());
      t.rec_cursor.alloc((size_t)t.small_chunks * t.rec_groups * sizeof(int));
      t.shape.alloc((size_t)E * S * sizeof(uint16_t));
      // persistent: 4 blocks of 4 warps per SM, fewer when there are not that many work items (a handful of sites)
      t.hard_blocks = (int)std::max<long long>(1, std::min<long long>(sms * 4LL, (t.wk_total + 3) / 4));
    }
    // partial dwell sums per block: [0, nblocks) easy / deterministic / direct-sampler kernel, then the general path kernel's
    t.dw_rows = t.nblocks + 3 * t.hard_blocks;  // general kernel: hard_blocks rows; short kernel: 2 hard_blocks (after them)
    t.dw_partial.alloc((size_t)t.dw_rows * n * sizeof(double));
    CK(cudaMemsetAsync(t.dw_partial.p, 0, t.dw_partial.bytes, stream));
    dev_bytes += t.tipcode.bytes + t.node_state.bytes + t.meta.bytes + t.PL.bytes + 2 * (t.rec_len[0].bytes + t.rec_st[0].bytes) +
                 t.dw_partial.bytes + t.hard_ballot.bytes + t.rec_cursor.bytes + t.shape.bytes + t.wk_item.bytes;
  }

  // The model buffer with the table of powers, the pinned host buffers and the chain's small device buffers.
  void alloc_model_and_host_buffers(double tmax) {
    jcap = opt.power_capacity > 0 ? opt.power_capacity : 64;
    if (V.exp) jcap = 302;  // newunifSample looks at up to 300 jumps (:120)
    else if (opt.power_capacity <= 0) {
      const double lam = Omega * tmax;
      const double want = lam + 10 * std::sqrt(lam) + 24;
      jcap = (int)std::min(16384.0, std::max(64.0, want));
    }
    if (jcap < 2) jcap = 2;
    model.alloc((model_stride() + (size_t)jcap * n * n) * sizeof(Real));
    CK(cudaMallocHost((void**)&model_h, (model_stride() + (size_t)jcap * n * n) * sizeof(Real)));
    memset(model_h, 0, (model_stride() + (size_t)jcap * n * n) * sizeof(Real));
    CK(cudaMallocHost((void**)&rows_h, (size_t)ntrees * WR * sizeof(double)));
    if (cudaHostGetDevicePointer((void**)&rows_h_dev, rows_h, 0) != cudaSuccess) { rows_h_dev = nullptr; (void)cudaGetLastError(); }
    if (opt.nccl_world > 1) nccl = clique(opt.nccl_id, opt.nccl_world, opt.nccl_rank);
    CK(cudaMallocHost((void**)&err_h, sizeof(unsigned)));
    CK(cudaMallocHost((void**)&ctl_h, 2 * sizeof(uint32_t)));
    ctl.alloc(2 * sizeof(uint32_t));
    phase_ns.alloc(2 * sizeof(unsigned long long));
    CK(cudaMemsetAsync(phase_ns.p, 0, phase_ns.bytes, stream));
    if (V.dic) { CK(cudaMallocHost((void**)&q_h, (size_t)n * n * sizeof(double))); q_dev.alloc((size_t)n * n * sizeof(double)); }
    cnt.alloc((size_t)n * n * sizeof(unsigned long long));
    root_out.alloc(sizeof(int));
    CK(cudaMemsetAsync(cnt.p, 0, cnt.bytes, stream));
    CK(cudaMemsetAsync(root_out.p, 0, root_out.bytes, stream));
  }

  // slots of the replay table per site and sweep: one per node, two per branch
  int replay_slots_per_iter() const { return (2 * trees[0]->sch.T - 1) + 2 * trees[0]->sch.E; }
  void upload_replay_table() {
    const long long nslots = (long long)ntrees * trees[0]->S * N_total * replay_slots_per_iter();
    std::vector<long long> off(nslots + 1);
    for (long long i = 0; i <= nslots; i++) off[i] = opt.tab_off[i];
    std::vector<double> u(opt.tab_u, opt.tab_u + off[nslots]);
    upload(tab_off, off, stream);
    upload(tab_u, u, stream);
    if (opt.host_tab) replay.reset(new pm::host::ReplaySource(opt.host_tab, opt.host_tab_n));
  }

  // The kernels' view of tree ti.
  void fill_params(TreeDev<Real>& t, int ti) {
    pm::ChainParams<Real>& P = t.P;
    const int T = t.sch.T, E = t.sch.E, spi = replay_slots_per_iter();
    P.n = n; P.T = T; P.E = E; P.S = t.S;
    P.cap_off = t.cap_off.template as<int>();
    P.hard_ballot = t.hard_ballot.template as<uint32_t>(); P.W = (int)((t.S + 31) / 32);
    P.wk_total = t.wk_total; P.wk_item = t.wk_item.template as<unsigned long long>();
    P.rec_cursor = t.rec_cursor.template as<int>(); P.chunk = t.chunk; P.easy_blocks = t.nblocks;
    P.shape = t.shape.template as<uint16_t>();
    P.model = model.as<Real>(); P.ppow = model.as<Real>() + model_stride(); P.jcap = jcap;
    P.up_entries = t.up_entries.template as<int>(); P.up_off = t.up_off.template as<int>();
    P.n_up_levels = (int)t.sch.up_off.size() - 1;
    P.cl_entries = t.cl_entries.template as<int>(); P.cl_warp_off = t.cl_warp_off.template as<int>();
    P.cl_top_entries = t.cl_top_entries.template as<int>(); P.cl_top_off = t.cl_top_off.template as<int>();
    P.cd_top = t.cd_top.template as<int>(); P.cd_top_off = t.cd_top_off.template as<int>();
    P.cd_entries = t.cd_entries.template as<int>(); P.cd_warp_off = t.cd_warp_off.template as<int>();
    P.cd_tips = t.cd_tips.template as<long long>();
    P.down_entries = t.down_entries.template as<int>(); P.down_off = t.down_off.template as<int>();
    P.n_down_levels = (int)t.sch.down_off.size() - 1;
    P.e_parent = t.e_parent.template as<int>(); P.e_child = t.e_child.template as<int>();
    P.e_len = t.e_len.template as<Real>();
    P.maps_off = t.maps_off.template as<long long>(); P.maps_len = t.maps_len.template as<double>();
    P.root = t.sch.root;
    P.tipcode = t.tipcode.template as<uint8_t>(); P.TS = t.TS; P.node_state = t.node_state.template as<uint8_t>();
    P.meta = t.meta.template as<uint32_t>(); P.PL = t.PL.template as<Real>();
    P.tile_base = 0; P.pl_S = t.pl_sites; P.rec_shift = t.rec_shift; P.rec_groups = t.rec_groups; P.ctl = nullptr;
    for (int b = 0; b < 2; b++) { P.rec_len[b] = t.rec_len[b].template as<Real>(); P.rec_st[b] = t.rec_st[b].template as<uint8_t>(); }
    // per-node rescaling (makePLrcpp_bigtree :525) only rescales the weights of each draw: the production
    // arithmetic always applies it (FP32 partials underflow after ~40 tips otherwise); the deterministic mode
    // follows the variant, underflow included.  No floor is applied: structural zeros stay exact.
    P.normalize = V.normalize || !exact; P.full_counts = V.full_counts; P.parity_tips = V.parity_tips;
    P.dw_partial = t.dw_partial.template as<double>(); P.cnt = cnt.as<unsigned long long>();
    P.root_out = root_out.as<int>(); P.err_flag = err_flag.as<unsigned>();
    const uint64_t key = opt.seed + (uint64_t)ti * 0x9E3779B97F4A7C15ull;
    P.rng.k0 = (uint32_t)key; P.rng.k1 = (uint32_t)(key >> 32);
    for (int r = 0; r < 10; r++) { P.rng.rk[2 * r] = P.rng.k0 + (uint32_t)r * 0x9E3779B9u; P.rng.rk[2 * r + 1] = P.rng.k1 + (uint32_t)r * 0xBB67AE85u; }
    P.rng.site0 = (uint32_t)opt.site_offset;
    P.rng.tab_off = opt.rng == PM_RNG_TABLE ? (const int64_t*)tab_off.p : nullptr;
    P.rng.tab_u = opt.rng == PM_RNG_TABLE ? tab_u.as<double>() : nullptr;
    P.rng.tab_site_stride = (int64_t)N_total * spi;
    P.rng.tab_base = (int64_t)ti * t.S * N_total * spi;
    P.rng.slots_per_iter = spi; P.rng.n_nodes = 2 * T - 1;
  }

  // sum `count` doubles at device address `buf` over the ranks, in stream order (no-op for a single process)
  void reduce_over_ranks(double* buf, int count) {
    if (nccl) {
      auto& api = pm::host::NcclApi::get();
      const int rc = api.AllReduce(buf, buf, (size_t)count, pm::host::NcclApi::kDouble, pm::host::NcclApi::kSum, nccl, stream);
      if (rc != 0) fail(PM_ERR_CUDA, "ncclAllReduce failed: %s", api.error(rc).c_str());
    } else if (opt.allreduce) {
      if (opt.allreduce(opt.allreduce_ctx, buf, count) != 0) fail(PM_ERR_CUDA, "allreduce callback failed");
    }
  }
  // the error slot of a reduced row: non-zero when any rank raised a device flag in that sweep
  void check_row_errors(const double* rows_host, int nrows) {
    bool any = false;
    for (int i = 0; i < nrows; i++) any = any || rows_host[(size_t)i * WR + W] != 0.0;
    if (!any) return;
    check_device_errors();  // throws with this rank's own reason if it has one
    fail(PM_ERR_CUDA, "another rank reported a device error in this sweep; all ranks stop together");
  }

  void ensure_rows(int count) {
    const int need = std::max(count, 1) * ntrees;
    if (need <= rows_cap) return;
    rows.alloc((size_t)need * WR * sizeof(double));
    rows_cap = need;
  }

  void write_fixed_row(const double* r, double* out, int64_t ld, int i) {
    for (int s = 0; s < n; s++) out[i + (int64_t)s * ld] = r[s];
    for (int a = 0; a < n; a++)
      for (int b = 0; b < n; b++) {
        if (a == b) continue;
        const int col = n + a * (n - 1) + b - (a < b ? 1 : 0);
        out[i + (int64_t)col * ld] = r[n + a * n + b];
      }
  }

  // ---- direct sampler (maketreelistEXP): independent histories, nothing carried between iterations ----
  void launch_exp_iteration(TreeDev<Real>& t, uint32_t iter, double* row) {
    const int gx = (int)((t.S + 31) / 32);
    Real* TP = t.TP.template as<Real>();
    double* llp = t.ll_partial.template as<double>();
    const size_t smem_b = (size_t)4 * n * sizeof(double) + ((size_t)n * n + ((n * n) & 1)) * sizeof(unsigned) + (size_t)n * n * sizeof(Real);
    const double* el = t.e_len_d.template as<double>();
    with_ns([&](auto ns) {
      constexpr int NSc = decltype(ns)::value;
      begin_timed(0);
      pm::k_loglik<Real, NSc><<<gx, 256, 0, stream>>>(t.P, TP, llp, nullptr);
      end_timed();
      begin_timed(1);
      pm::k_exp_nodes<Real, NSc><<<gx, 256, 0, stream>>>(t.P, TP, iter);
      end_timed();
      begin_timed(2);
      pm::k_exp_branches<Real, NSc><<<t.paths_grid, 128, smem_b, stream>>>(t.P, TP, el, (Real)Omega, iter, t.chunk);
      end_timed();
    });
    begin_timed(3);
    pm::k_reduce<<<1, 256, 0, stream>>>(t.dw_partial.template as<double>(), t.dw_rows, n, cnt.as<unsigned long long>(),
                                        root_out.as<int>(), row, 0, err_flag.as<unsigned>(), W);
    end_timed();
    launches += 4;
  }

  void run(int count, double* out, int64_t ld) override {
    if (count < 0 || iters_done + count > N_total) fail(PM_ERR_ARG, "cannot run %d more iterations (%d of %d done)", count, iters_done, N_total);
    if (count == 0) return;
    if (ld < count) fail(PM_ERR_ARG, "leading dimension smaller than the number of rows");
    CK(cudaSetDevice(opt.device));
    if (!V.rates) {
      ensure_rows(count);
      TreeDev<Real>& t = *trees[0];
      // small problems: the first sweep of the call goes out launch by launch (it also sets the kernels' attributes), the
      // others replay a captured sweep
      const bool small = (double)t.S * t.sch.E <= (double)(1 << 22);
      const bool one_launch = !V.exp && !exact && use_small(t);  // every sweep of the call inside one launch
      const bool use_graph = !one_launch && !V.exp && !timing && !sw.debug_sync && count > 1 && (sw.graph == 1 || (sw.graph != 0 && small));
      if (one_launch) launch_small(t, (uint32_t)iters_done, count, rows.as<double>());
      for (int i = 0; i < count && !one_launch; i++) {
        if (V.exp) launch_exp_iteration(t, (uint32_t)(iters_done + i), rows.as<double>() + (size_t)i * WR);
        else if (use_graph && i > 0) {
          if (i == 1) {
            if (sweep_graph && graph_rows != rows.p) { cudaGraphExecDestroy(sweep_graph); sweep_graph = nullptr; }
            if (!sweep_graph) {
              cudaGraph_t g = nullptr;
              CK(cudaStreamBeginCapture(stream, cudaStreamCaptureModeRelaxed));
              capturing = true;
              try { launch_sweep(t, 1u, rows.as<double>()); } catch (...) { capturing = false; cudaStreamEndCapture(stream, &g); if (g) cudaGraphDestroy(g); throw; }
              capturing = false;
              CK(cudaStreamEndCapture(stream, &g));
              const cudaError_t ge = cudaGraphInstantiate(&sweep_graph, g, 0);
              cudaGraphDestroy(g);
              if (ge != cudaSuccess) fail(PM_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ge));
              graph_rows = rows.p;
            }
            ctl_h[0] = (uint32_t)(iters_done + 1); ctl_h[1] = 1u;
            CK(cudaMemcpyAsync(ctl.p, ctl_h, 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
          }
          CK(cudaGraphLaunch(sweep_graph, stream));
          launches += launches_per_sweep;
        }
        else launch_sweep(t, (uint32_t)(iters_done + i), rows.as<double>() + (size_t)i * WR);
        if (opt.progress) { printf("%i \r", iters_done + i); }
      }
      CK(cudaGetLastError());
      reduce_over_ranks(rows.as<double>(), count * WR);
      std::vector<double> h((size_t)count * WR);
      CK(cudaMemcpyAsync(h.data(), rows.p, h.size() * sizeof(double), cudaMemcpyDeviceToHost, stream));
      CK(cudaStreamSynchronize(stream));
      check_row_errors(h.data(), count);
      collect_timed();
      for (int i = 0; i < count; i++) write_fixed_row(&h[(size_t)i * WR], out, ld, i);
      iters_done += count;
      return;
    }

    // rate-updating samplers: one host round trip per iteration
    ensure_rows(1);
    pm::host::RateModel rm{n, Q, B, Omega, prior.data()};
    const size_t nparam = V.hidden ? (size_t)2 + 3 * (n / 2 - 1) : 2;
    if (rate_proposed.size() != nparam) { rate_proposed.assign(nparam, 0); rate_accepted.assign(nparam, 0); }
    rm.proposed = rate_proposed.data(); rm.accepted = rate_accepted.data();
    pm::host::UniformSource& g = host_rng();
    std::vector<double> row(ncols);
    std::vector<std::vector<double>> jodt(ntrees, std::vector<double>(ncols, 0.0));
    for (int i = 0; i < count; i++) {
      const int it = iters_done;
      if (V.multi && it == 0) (void)g.next();  // the draw before the loop, :2332 / :2810
      // the one-block-per-site kernels of a single process write their rows straight into the pinned host buffer (mapped:
      // no copy to wait for after the launch); otherwise rows land in device memory, where the collective finds them
      bool host_rows = rows_h_dev != nullptr && !nccl && !opt.allreduce && !V.dic;
      for (int j = 0; j < ntrees; j++) host_rows = host_rows && use_small(*trees[j]);
      double* const row0 = host_rows ? rows_h_dev : rows.as<double>();
      for (int j = 0; j < ntrees; j++) launch_sweep(*trees[j], (uint32_t)it, row0 + (size_t)j * WR);
      if (V.dic) launch_loglik(*trees[0], rows.as<double>());
      CK(cudaGetLastError());
      // one small all-reduce per sweep (n + n^2 + 1 (+1) statistics + the error slot, per tree), then ONE synchronisation:
      // the device error flag travels in the row instead of a second copy
      cudaEvent_t ca = nullptr, cb = nullptr;
      if (timing) { CK(cudaEventCreate(&ca)); CK(cudaEventCreate(&cb)); CK(cudaEventRecord(ca, stream)); }
      reduce_over_ranks(rows.as<double>(), ntrees * WR);
      if (timing) CK(cudaEventRecord(cb, stream));
      if (!host_rows) CK(cudaMemcpyAsync(rows_h, rows.p, (size_t)ntrees * WR * sizeof(double), cudaMemcpyDeviceToHost, stream));
      CK(cudaStreamSynchronize(stream));
      if (timing) { float ms = 0; cudaEventElapsedTime(&ms, ca, cb); comm_ms += ms; cudaEventDestroy(ca); cudaEventDestroy(cb); }
      const auto host_t0 = std::chrono::steady_clock::now();
      check_row_errors(rows_h, ntrees);
      for (int j = 0; j < ntrees; j++) {
        std::fill(jodt[j].begin(), jodt[j].end(), 0.0);
        const double* r = rows_h + (size_t)j * WR;
        for (int c = 0; c < n + n * n; c++) jodt[j][c] = r[c];
        if (V.hidden) rm.record_hidden(jodt[j].data()); else rm.record_two_state(jodt[j].data());
        if (V.dic) { jodt[j][ncols - 2] = r[n + n * n]; jodt[j][ncols - 1] = r[n + n * n + 1]; }
        else jodt[j][ncols - 1] = r[n + n * n];  // root state of global site 0 (overwritten by the tree index for mt)
      }
      int pick = 0;
      if (V.multi) {  // sampleOnce with equal weights, :2347-2348
        const double u = g.next();
        double cum = 0;
        for (pick = 0; pick < ntrees; pick++) { cum += 1.0 / ntrees; if (u < cum) break; }
        if (pick >= ntrees) pick = ntrees - 1;
        jodt[pick][ncols - 1] = pick;
      }
      const double* st = jodt[pick].data();
      for (int c = 0; c < ncols; c++) out[i + (int64_t)c * ld] = st[c];
      if (V.hidden) rm.hidden_rates(st, g, V.multi); else rm.two_state(st, g, V.multi);
      if (g.exhausted()) fail(PM_ERR_REPLAY, "host replay table exhausted");
      iters_done++;
      stage_model(false);
      if (timing) host_update_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - host_t0).count();
      if (opt.progress) { printf("%i \r", it); }
    }
    CK(cudaStreamSynchronize(stream));
    collect_timed();
  }

  float time_prune(int tree, int reps) override {
    if (tree < 0 || tree >= ntrees || reps < 1) fail(PM_ERR_ARG, "bad arguments");
    CK(cudaSetDevice(opt.device));
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
    launch_prune(*trees[tree]);  // warm
    CK(cudaEventRecord(a, stream));
    for (int r = 0; r < reps; r++) launch_prune(*trees[tree]);
    CK(cudaEventRecord(b, stream));
    CK(cudaEventSynchronize(b));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, a, b));
    cudaEventDestroy(a); cudaEventDestroy(b);
    CK(cudaGetLastError());
    return ms / reps;
  }

  // ---- state read-back (parity tests) ----
  void node_states(int tree, int32_t* out) override {
    TreeDev<Real>& t = *trees.at(tree);
    const int NN = 2 * t.sch.T - 1;
    std::vector<uint8_t> h((size_t)NN * t.S);
    CK(cudaMemcpy(h.data(), t.node_state.p, h.size(), cudaMemcpyDeviceToHost));
    for (long long s = 0; s < t.S; s++) for (int v = 0; v < NN; v++) out[s * NN + v] = h[(size_t)v * t.S + s];
  }
  void piece_counts(int tree, int32_t* out) override {
    TreeDev<Real>& t = *trees.at(tree);
    const int E = t.sch.E;
    std::vector<uint32_t> h((size_t)E * t.S);
    CK(cudaMemcpy(h.data(), t.meta.p, h.size() * 4, cudaMemcpyDeviceToHost));
    for (long long s = 0; s < t.S; s++) for (int e = 0; e < E; e++) out[s * E + e] = (int)(h[(size_t)e * t.S + s] & 0xffffu);
  }
  int path(int tree, int64_t site, int e, double* len, int32_t* st, int cap) override {
    TreeDev<Real>& t = *trees.at(tree);
    if (site < 0 || site >= t.S || e < 0 || e >= t.sch.E) fail(PM_ERR_ARG, "bad site / branch");
    uint32_t m = 0;
    CK(cudaMemcpy(&m, t.meta.template as<uint32_t>() + (size_t)e * t.S + site, 4, cudaMemcpyDeviceToHost));
    if (iters_done == 0) fail(PM_ERR_ARG, "no sweep done yet");
    const int c = e / t.chunk, b0 = c * t.chunk;
    const int cap_c = t.cap_off_h[c + 1] - t.cap_off_h[c];
    const int buf = (iters_done - 1) & 1;
    auto records = [&](long long pos, int count) {
      const size_t base = (size_t)t.cap_off_h[c] * t.rec_groups + (size_t)(site >> t.rec_shift) * cap_c + pos;
      for (int k = 0; k < count && k < cap; k++) {
        Real L; uint8_t s;
        CK(cudaMemcpy(&L, t.rec_len[buf].template as<Real>() + base + k, sizeof(Real), cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(&s, t.rec_st[buf].template as<uint8_t>() + base + k, 1, cudaMemcpyDeviceToHost));
        len[k] = (double)L; st[k] = s;
      }
    };
    if (exact) {  // meta = m | nj << 16 | s0 << 24; every path keeps nj + 1 records
      const int nj = (m >> 16) & 0xff;
      long long pos = 0;
      for (int e2 = b0; e2 < e; e2++) {
        uint32_t m2 = 0;
        CK(cudaMemcpy(&m2, t.meta.template as<uint32_t>() + (size_t)e2 * t.S + site, 4, cudaMemcpyDeviceToHost));
        pos += ((m2 >> 16) & 0xff) + 1;
      }
      records(pos, nj + 1);
      return nj + 1;
    }
    // production: meta = m | q << 16 (q: 16-bit position of the jump point of a two-run path, or the offset of the path's
    // records in the site's slice); shape = nj (6 bits) | s0 << 6 | s1 << 11
    uint16_t shp = 0;
    CK(cudaMemcpy(&shp, t.shape.template as<uint16_t>() + (size_t)e * t.S + site, 2, cudaMemcpyDeviceToHost));
    int nj = shp & 0x3f;
    const int s0 = (shp >> 6) & 0x1f, s1 = (shp >> 11) & 0x1f;
    const uint32_t q = m >> 16;
    Real Le;
    CK(cudaMemcpy(&Le, t.e_len.template as<Real>() + e, sizeof(Real), cudaMemcpyDeviceToHost));
    if (nj == 0) {
      if (cap > 0) { len[0] = (double)Le; st[0] = s0; }
      return 1;
    }
    if (nj == 1) {
      const Real p1 = (Real)q * (Le * (Real)(1.0 / 65536.0));
      if (cap > 0) { len[0] = (double)p1; st[0] = s0; }
      if (cap > 1) { len[1] = (double)(Le - p1); st[1] = s1; }
      return 2;
    }
    long long pos = (long long)q;  // paths with two or more real jumps: the offset of their records in the site's slice
    if (nj == 63) {  // 64 runs or more: a header record holds the count
      Real cntv;
      CK(cudaMemcpy(&cntv, t.rec_len[buf].template as<Real>() + (size_t)t.cap_off_h[c] * t.rec_groups + (size_t)(site >> t.rec_shift) * cap_c + pos, sizeof(Real),
                    cudaMemcpyDeviceToHost));
      nj = (int)cntv - 1;
      pos += 1;
    }
    records(pos, nj + 1);
    return nj + 1;
  }
  // Stochastic maps of the selected sites (pm_maps.cuh), in batches of sites whose selection, counts and offsets take at
  // most half the scratch budget: count, scan, offsets to the caller; then the runs of as many consecutive sites of the
  // batch as the other half holds at a time (more for a single site that needs it).
  void maps(int tree, const int64_t* sites, int64_t nsel, int64_t* off, double* len, int32_t* st, int64_t cap) override {
    if (tree < 0 || tree >= ntrees) fail(PM_ERR_ARG, "bad tree");
    if (V.exp || V.llonly) fail(PM_ERR_ARG, "this chain keeps no path state");
    if (nsel < 0 || cap < 0 || !off || (nsel > 0 && !sites)) fail(PM_ERR_ARG, "bad arguments");
    TreeDev<Real>& t = *trees[tree];
    for (int64_t i = 0; i < nsel; i++)
      if (sites[i] < 0 || sites[i] >= t.S) fail(PM_ERR_ARG, "bad site / branch");
    if (iters_done == 0) fail(PM_ERR_ARG, "no sweep done yet");
    off[0] = 0;
    if (nsel == 0) return;
    CK(cudaSetDevice(opt.device));
    const long long E = t.sch.E;
    size_t free_b = 0, total_b = 0;
    CK(cudaMemGetInfo(&free_b, &total_b));
    const size_t budget = std::min(pm::kMapsScratchBytes, free_b / 2);
    const size_t per_site = (size_t)E * (sizeof(int) + sizeof(long long)) + sizeof(long long);
    const size_t run_bytes = sizeof(double) + sizeof(int32_t);
    const long long nb = std::min<long long>({(long long)nsel, (long long)(budget / 2 / per_site), 32LL * 65535});
    if (nb < 1) fail(PM_ERR_CUDA, "the maps of one site need %zu bytes of device scratch, %zu bytes are free", 2 * per_site, free_b);
    const long long runs_budget = (long long)((budget - (size_t)nb * per_site) / run_bytes);

    struct Scratch {  // stream-ordered device allocation
      void* p = nullptr;
      cudaStream_t s;
      explicit Scratch(cudaStream_t st) : s(st) {}
      ~Scratch() { if (p) cudaFreeAsync(p, s); }
      void alloc(size_t n) { if (p) cudaFreeAsync(p, s); p = nullptr; CK(cudaMallocAsync(&p, std::max<size_t>(n, 16), s)); }
    } d_sel(stream), d_cnt(stream), d_off(stream), d_tmp(stream), d_len(stream), d_st(stream);
    size_t tmp_bytes = 0;
    CK(cub::DeviceScan::ExclusiveScan(nullptr, tmp_bytes, (const int*)nullptr, (long long*)nullptr, ::cuda::std::plus<>{}, 0LL,
                                      nb * E + 1, stream));
    d_sel.alloc(nb * sizeof(long long));
    d_cnt.alloc((nb * E + 1) * sizeof(int));
    d_off.alloc((nb * E + 1) * sizeof(long long));
    d_tmp.alloc(tmp_bytes);

    pm::MapsSrc<Real> M;
    const int buf = (iters_done - 1) & 1;
    M.meta = t.meta.template as<uint32_t>(); M.shape = exact ? nullptr : t.shape.template as<uint16_t>();
    M.e_len = t.e_len.template as<Real>();
    M.rec_len = t.rec_len[buf].template as<Real>(); M.rec_st = t.rec_st[buf].template as<uint8_t>();
    M.cap_off = t.cap_off.template as<int>();
    M.S = t.S; M.rec_groups = t.rec_groups; M.E = (int)E; M.chunk = t.chunk; M.rec_shift = t.rec_shift; M.exact = exact ? 1 : 0;
    const dim3 blk(32, 8);
    const bool want_runs = len && st;
    long long runs_alloc = 0, base = 0;
    bool fits = true;
    for (long long s0 = 0; s0 < nsel; s0 += nb) {
      const long long nbb = std::min<long long>(nb, nsel - s0), ne = nbb * E;
      long long* const d_offp = static_cast<long long*>(d_off.p);
      CK(cudaMemcpyAsync(d_sel.p, sites + s0, nbb * sizeof(long long), cudaMemcpyHostToDevice, stream));
      CK(cudaMemsetAsync(static_cast<int*>(d_cnt.p) + ne, 0, sizeof(int), stream));
      pm::k_maps_count<Real><<<dim3((unsigned)((E + 31) / 32), (unsigned)((nbb + 31) / 32)), blk, 0, stream>>>(
          M, static_cast<const long long*>(d_sel.p), nbb, static_cast<int*>(d_cnt.p));
      CK(cudaGetLastError());
      CK(cub::DeviceScan::ExclusiveScan(d_tmp.p, tmp_bytes, static_cast<const int*>(d_cnt.p), d_offp, ::cuda::std::plus<>{}, base,
                                        ne + 1, stream));
      CK(cudaMemcpyAsync(off + s0 * E, d_offp, (ne + 1) * sizeof(long long), cudaMemcpyDeviceToHost, stream));
      CK(cudaStreamSynchronize(stream));
      const long long end = off[(s0 + nbb) * E];
      if (want_runs && end > cap) fits = false;
      for (long long j0 = 0; want_runs && fits && j0 < nbb;) {
        const long long r0 = off[(s0 + j0) * E];
        long long j1 = j0 + 1;
        while (j1 < nbb && off[(s0 + j1 + 1) * E] - r0 <= runs_budget) j1++;
        const long long nr = off[(s0 + j1) * E] - r0;
        if (nr > runs_alloc) {
          runs_alloc = std::max(nr, std::min(runs_budget, end - r0));
          d_len.alloc(runs_alloc * sizeof(double));
          d_st.alloc(runs_alloc * sizeof(int32_t));
        }
        pm::k_maps_write<Real><<<dim3((unsigned)((E + 31) / 32), (unsigned)((j1 - j0 + 31) / 32)), blk, 0, stream>>>(
            M, static_cast<const long long*>(d_sel.p), j0, j1, d_offp, r0, static_cast<double*>(d_len.p), static_cast<int32_t*>(d_st.p));
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(len + r0, d_len.p, nr * sizeof(double), cudaMemcpyDeviceToHost, stream));
        CK(cudaMemcpyAsync(st + r0, d_st.p, nr * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
        j0 = j1;
      }
      base = end;
    }
    CK(cudaStreamSynchronize(stream));
    if (want_runs && !fits) fail(PM_ERR_CAPACITY, "the maps hold %lld runs, the output arrays %lld", base, (long long)cap);
  }
  // ---- checkpoint / resume: everything a sweep reads that is not an input of pm_chain_create ----
  static constexpr uint32_t PM_STATE_FORMAT = 6;  // 6: model and table of powers in one buffer; 5: production record slices shared by groups of 32 sites; 1: round 1 (per-site masks); 2: branch-major ballots, global record cursors; 3: two-run paths count their virtual jumps together; 4: 16-bit positions inside meta, shape words
  struct StateHeader {
    char magic[8];
    int32_t variant, n, ntrees, precision, mode, T, E, iters_done, jcap, reserved;
    int64_t S, site_offset, total_bytes;
    uint64_t seed;
  };
  std::vector<DevBuf*> state_buffers() {
    std::vector<DevBuf*> v{&model};
    for (auto& t : trees) {
      v.push_back(&t->node_state); v.push_back(&t->meta); v.push_back(&t->shape);
      for (int b = 0; b < 2; b++) { v.push_back(&t->rec_len[b]); v.push_back(&t->rec_st[b]); }
    }
    return v;
  }
  size_t host_state_bytes() const { return sizeof(StateHeader) + 625 * sizeof(uint32_t) + ((size_t)2 * n * n + 2 * n) * sizeof(double); }
  int64_t state_bytes() override {
    size_t tot = host_state_bytes();
    for (DevBuf* b : state_buffers()) tot += (b->bytes + 15) & ~(size_t)15;
    return (int64_t)tot;
  }
  StateHeader make_header() {
    StateHeader h;
    memset(&h, 0, sizeof h);
    memcpy(h.magic, "PMB200S", 8);
    h.variant = V.id; h.n = n; h.ntrees = ntrees; h.precision = opt.precision; h.mode = opt.mode;
    h.T = trees[0]->sch.T; h.E = trees[0]->sch.E; h.iters_done = iters_done; h.jcap = jcap;
    h.S = trees[0]->S; h.site_offset = opt.site_offset; h.total_bytes = state_bytes(); h.seed = opt.seed;
    // format version and a hash of what fixes the interpretation of the buffers (the packing of `meta`, the record slices
    // of every chunk, the count-mode threshold, the local path buffer): a blob written under another layout is refused
    // instead of being read under this one (ADVICE r1)
    uint32_t hsh = 2166136261u;
    auto mix = [&](uint32_t v) { hsh = (hsh ^ v) * 16777619u; };
    mix(PM_STATE_FORMAT); mix(PM_META(1, 2)); mix((uint32_t)PM_SHAPE(1, 2, 3)); mix(PM_LAMBDA_INV); mix(PM_LOCAL_PATH_MAX); mix(PM_SMEM_POW);
    for (auto& t : trees) { mix((uint32_t)t->chunk); mix((uint32_t)t->rec_shift); for (int c : t->cap_off_h) mix((uint32_t)c); }
    h.reserved = (int32_t)((PM_STATE_FORMAT << 24) | (hsh & 0xffffffu));
    return h;
  }
  void export_state(void* buf, int64_t bytes) override {
    if (opt.rng == PM_RNG_TABLE) fail(PM_ERR_ARG, "replay-table runs cannot be checkpointed");
    if (!buf || bytes < state_bytes()) fail(PM_ERR_ARG, "state buffer too small (%lld bytes needed)", (long long)state_bytes());
    CK(cudaSetDevice(opt.device));
    CK(cudaStreamSynchronize(stream));
    unsigned char* p = (unsigned char*)buf;
    const StateHeader h = make_header();
    memcpy(p, &h, sizeof h); p += sizeof h;
    uint32_t w[625]; mt.save(w);
    memcpy(p, w, sizeof w); p += sizeof w;
    memcpy(p, Q, (size_t)n * n * sizeof(double)); p += (size_t)n * n * sizeof(double);
    memcpy(p, B, (size_t)n * n * sizeof(double)); p += (size_t)n * n * sizeof(double);
    memcpy(p, scale_prev.data(), n * sizeof(double)); p += n * sizeof(double);
    memcpy(p, rate_prev.data(), n * sizeof(double)); p += n * sizeof(double);
    for (DevBuf* b : state_buffers()) {
      if (b->bytes) CK(cudaMemcpyAsync(p, b->p, b->bytes, cudaMemcpyDeviceToHost, stream));
      p += (b->bytes + 15) & ~(size_t)15;
    }
    CK(cudaStreamSynchronize(stream));
  }
  void import_state(const void* buf, int64_t bytes) override {
    if (opt.rng == PM_RNG_TABLE) fail(PM_ERR_ARG, "replay-table runs cannot be checkpointed");
    if (!buf || bytes < (int64_t)sizeof(StateHeader)) fail(PM_ERR_ARG, "not a chain state");
    const unsigned char* p = (const unsigned char*)buf;
    StateHeader h; memcpy(&h, p, sizeof h); p += sizeof h;
    const StateHeader me = make_header();
    if (memcmp(h.magic, me.magic, 8) != 0) fail(PM_ERR_ARG, "not a chain state");
    if (h.variant != me.variant || h.n != me.n || h.ntrees != me.ntrees || h.precision != me.precision || h.mode != me.mode ||
        h.T != me.T || h.E != me.E || h.S != me.S || h.site_offset != me.site_offset || h.jcap != me.jcap || h.seed != me.seed ||
        h.total_bytes != me.total_bytes)
      fail(PM_ERR_ARG, "the state was exported by a chain of a different shape, sampler, precision, seed or site block");
    if (h.reserved != me.reserved)
      fail(PM_ERR_ARG, "the state was exported under another state format or buffer layout (format %d here, %d in the blob)",
           (int)PM_STATE_FORMAT, (int)((uint32_t)h.reserved >> 24));
    if (bytes < h.total_bytes) fail(PM_ERR_ARG, "truncated chain state");
    if (h.iters_done < 0 || h.iters_done > N_total) fail(PM_ERR_ARG, "the state has %d iterations done, this chain was created for %d", h.iters_done, N_total);
    CK(cudaSetDevice(opt.device));
    CK(cudaStreamSynchronize(stream));
    uint32_t w[625]; memcpy(w, p, sizeof w); p += sizeof w;
    if (w[624] > 624u) fail(PM_ERR_ARG, "corrupt chain state");
    mt.load(w);
    memcpy(Q, p, (size_t)n * n * sizeof(double)); p += (size_t)n * n * sizeof(double);
    memcpy(B, p, (size_t)n * n * sizeof(double)); p += (size_t)n * n * sizeof(double);
    memcpy(scale_prev.data(), p, n * sizeof(double)); p += n * sizeof(double);
    memcpy(rate_prev.data(), p, n * sizeof(double)); p += n * sizeof(double);
    for (DevBuf* b : state_buffers()) {
      if (b->bytes) CK(cudaMemcpyAsync(b->p, p, b->bytes, cudaMemcpyHostToDevice, stream));
      p += (b->bytes + 15) & ~(size_t)15;
    }
    CK(cudaStreamSynchronize(stream));
    iters_done = h.iters_done;
  }

  // log p(y | Q) of the chain's current Q, summed over the sites of all ranks (pm_loglik)
  double loglik() override {
    if (!V.dic) fail(PM_ERR_ARG, "this chain was not created with a log-likelihood column");
    CK(cudaSetDevice(opt.device));
    ensure_rows(1);
    double* row = rows.as<double>();
    launch_loglik(*trees[0], row);
    CK(cudaGetLastError());
    double* cell = row + n + n * n + 1;
    reduce_over_ranks(cell, 1);
    CK(cudaMemcpyAsync(rows_h, cell, sizeof(double), cudaMemcpyDeviceToHost, stream));
    check_device_errors();
    return rows_h[0];
  }
  // Exact posterior expectations of this log-likelihood chain's sites (pm_expected_sumstats): branch integrals, the inside
  // pass with its per-site log-likelihoods, the outside pass.  stats: column-major, leading dimension ld; write: the
  // per-branch statistics and node marginals of every site too.  With PHYLOMAP_B200_TRACE=1 the three kernels' CUDA-event
  // times go to stderr.
  void expected(bool write, double* stats, int64_t ld, double* ll, double* branch_stats, double* node_marginals) override {
    if (!V.llonly) fail(PM_ERR_ARG, "posterior expectations are computed by a log-likelihood chain");
    CK(cudaSetDevice(opt.device));
    TreeDev<Real>& t = *trees[0];
    const int E = t.sch.E, T = t.sch.T, NK = n * n;
    const long long S = t.S;
    for (int i = 0; i < n; i++) for (int j = 0; j < n; j++) q_h[(size_t)i * n + j] = Q[i + (size_t)j * n];
    CK(cudaMemcpyAsync(q_dev.p, q_h, (size_t)n * n * sizeof(double), cudaMemcpyHostToDevice, stream));
    DevBuf M, site_ll, st_d, br_d, nd_d;
    M.alloc((size_t)E * NK * NK * sizeof(Real));
    site_ll.alloc((size_t)S * sizeof(double));
    st_d.alloc((size_t)NK * S * sizeof(double));
    if (write) { br_d.alloc((size_t)S * E * NK * sizeof(double)); nd_d.alloc((size_t)S * (2 * T - 1) * n * sizeof(double)); }
    cudaEvent_t ev[4] = {};
    struct Events { cudaEvent_t* e; ~Events() { for (int i = 0; i < 4; i++) if (e[i]) cudaEventDestroy(e[i]); } } ev_guard{ev};
    if (sw.trace) for (int i = 0; i < 4; i++) CK(cudaEventCreate(&ev[i]));
    const auto mark = [&](int i) { if (sw.trace) CK(cudaEventRecord(ev[i], stream)); };
    const int gx = (int)((S + 31) / 32);
    const size_t smem = (size_t)8 * NK * 32 * sizeof(double);
    mark(0);
    pm::k_transprob<Real><<<(E + 127) / 128, 128, 0, stream>>>(q_dev.as<double>(), t.e_len_d.template as<double>(), E, n, t.TP.template as<Real>());
    pm::k_branch_integrals<Real><<<(unsigned)(((long long)E * NK + 127) / 128), 128, 0, stream>>>(q_dev.as<double>(), t.e_len_d.template as<double>(),
                                                                                              E, n, M.as<Real>());
    mark(1);
    with_ns([&](auto ns) {
      constexpr int NSc = decltype(ns)::value;
      pm::k_loglik<Real, NSc><<<gx, 256, 0, stream>>>(t.P, t.TP.template as<Real>(), t.ll_partial.template as<double>(), site_ll.as<double>());
      mark(2);
      const auto launch = [&](auto kern) {
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<gx, 256, smem, stream>>>(t.P, t.TP.template as<Real>(), M.as<Real>(), st_d.as<double>(), br_d.as<double>(), nd_d.as<double>());
      };
      if (write) launch(pm::k_expect<Real, NSc, true>);
      else launch(pm::k_expect<Real, NSc, false>);
    });
    mark(3);
    CK(cudaGetLastError());
    launches += 4;
    if (stats)
      CK(cudaMemcpy2DAsync(stats, (size_t)ld * sizeof(double), st_d.p, (size_t)S * sizeof(double), (size_t)S * sizeof(double), NK,
                           cudaMemcpyDeviceToHost, stream));
    if (ll) CK(cudaMemcpyAsync(ll, site_ll.p, (size_t)S * sizeof(double), cudaMemcpyDeviceToHost, stream));
    if (write && branch_stats) CK(cudaMemcpyAsync(branch_stats, br_d.p, br_d.bytes, cudaMemcpyDeviceToHost, stream));
    if (write && node_marginals) CK(cudaMemcpyAsync(node_marginals, nd_d.p, nd_d.bytes, cudaMemcpyDeviceToHost, stream));
    check_device_errors();
    if (sw.trace) {
      float ms[3] = {0, 0, 0};
      for (int i = 0; i < 3; i++) CK(cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]));
      fprintf(stderr, "[phylomap_b200] expect: %lld sites%s: P(t) + branch integrals %.4f ms, inside %.4f ms, outside %.4f ms\n", S,
              write ? " (selected)" : "", ms[0], ms[1], ms[2]);
    }
  }
  // partials of the current state: a pruning pass over the site's block (into slot 0 of the fused kernel's partials) or
  // over all sites, then the site's column
  void partials(int tree, int64_t site, double* out) override {
    TreeDev<Real>& t = *trees.at(tree);
    const int T = t.sch.T;
    if (site < 0 || site >= t.S) fail(PM_ERR_ARG, "bad site");
    CK(cudaSetDevice(opt.device));
    launch_prune(t, site);
    CK(cudaStreamSynchronize(stream));
    const long long col = t.pl_slots ? site % 32 : site;
    std::fill(out, out + (size_t)(2 * T - 1) * n, 0.0);
    std::vector<Real> v(n);
    for (int i = 0; i < T - 1; i++) {
      CK(cudaMemcpy(v.data(), t.PL.template as<Real>() + ((size_t)i * t.pl_sites + col) * n, n * sizeof(Real), cudaMemcpyDeviceToHost));
      for (int j = 0; j < n; j++) out[(size_t)(T + i) * n + j] = (double)v[j];
    }
  }
};

struct EigenIn { const double* lefts; const double* rights; const double* d; };

template <typename Real>
void prepare_exp(ChainT<Real>& c, int n, const double* Q, const EigenIn& eg, double*& B, double& Omega) {
  // Omega := -min diag(Q) (:3008); B = I + Q / Omega is internal; eigen inputs arrive column-major from R
  double mn = Q[0];
  for (int i = 1; i < n; i++) mn = std::min(mn, Q[i + (size_t)i * n]);
  Omega = -mn;
  c.own_B.assign((size_t)n * n, 0.0);
  for (int i = 0; i < n; i++) for (int j = 0; j < n; j++) c.own_B[i + (size_t)j * n] = (i == j ? 1.0 : 0.0) + Q[i + (size_t)j * n] / Omega;
  B = c.own_B.data();
  c.eig_L.resize((size_t)n * n); c.eig_R.resize((size_t)n * n); c.eig_d.resize(n);
  for (int i = 0; i < n; i++) {
    c.eig_d[i] = eg.d[i + (size_t)i * n];
    for (int j = 0; j < n; j++) { c.eig_L[(size_t)i * n + j] = eg.lefts[i + (size_t)j * n]; c.eig_R[(size_t)i * n + j] = eg.rights[i + (size_t)j * n]; }
  }
}

pm_chain* make_chain(int variant, const pm_tree* trees, int ntrees, int n, double* Q, const double* pid, double* B,
                     double Omega, const double* prior, int nprior, int N_total, const pm_options* opt,
                     const EigenIn* eg = nullptr, bool internal = false) {
  pm_options def;
  if (!opt) { pm_default_options(&def); opt = &def; }
  if (!trees || !Q || !pid || (!B && variant != PM_V_EXP)) fail(PM_ERR_ARG, "null argument");
  if (variant == PM_V_EXP && (!eg || !eg->lefts || !eg->rights || !eg->d)) fail(PM_ERR_ARG, "the direct sampler needs the eigendecomposition of Q");
  if (variant == PM_V_EXP && (n < 2 || n > PM_NMAX)) fail(PM_ERR_ARG, "number of states must be in 2..%d", PM_NMAX);
  if ((variant < PM_V_PLAIN || variant > PM_V_EXP) && !internal) fail(PM_ERR_ARG, "unknown variant");
  if (opt->precision == PM_F32) {
    std::unique_ptr<ChainT<float>> c(new ChainT<float>());
    if (variant == PM_V_EXP) prepare_exp(*c, n, Q, *eg, B, Omega);
    c->create(variant, trees, ntrees, n, Q, pid, B, Omega, prior, nprior, N_total, opt);
    return c.release();
  }
  std::unique_ptr<ChainT<double>> c(new ChainT<double>());
  if (variant == PM_V_EXP) prepare_exp(*c, n, Q, *eg, B, Omega);
  c->create(variant, trees, ntrees, n, Q, pid, B, Omega, prior, nprior, N_total, opt);
  return c.release();
}

// Fixed-Q samplers over a block of sites [s0, s0 + count) of `x`: a chain of its own (sites are independent given Q).
void run_site_block(int variant, const pm_tree* x, int n, double* Q, const double* pid, double* B, double Omega, int N,
                    const pm_options* opt, const EigenIn* eg, long long s0, long long count, double* out) {
  pm_tree t = *x;
  t.n_sites = count;
  if (x->states_u8) t.states_u8 = x->states_u8 + s0 * (long long)x->n_tips;
  if (x->states) t.states = x->states + s0 * (long long)x->n_tips;
  pm_options o = *opt;
  o.site_offset = opt->site_offset + s0;
  std::unique_ptr<pm_chain> c(make_chain(variant, &t, 1, n, Q, pid, B, Omega, nullptr, 0, N, &o, eg));
  c->run(N, out, N);
}

int one_call(int variant, const pm_tree* trees, int ntrees, int n, double* Q, const double* pid, double* B, double Omega,
             int N, const double* prior, int nprior, const pm_options* opt, double* out, char* err, size_t errlen,
             const EigenIn* eg = nullptr) {
  return guarded(err, errlen, [&] {
    if (!out && N > 0) fail(PM_ERR_ARG, "null output");
    pm_options def;
    if (!opt) { pm_default_options(&def); opt = &def; }
    const bool fixed_q = variant == PM_V_PLAIN || variant == PM_V_SPARSE || variant == PM_V_BIGTREE || variant == PM_V_EXP;
    const bool single_process = !opt->allreduce && opt->nccl_world <= 1;
    long long tile = read_switches().site_tile;  // sites per chain; 0 = all at once
    if (!fixed_q || !trees || ntrees != 1 || opt->rng == PM_RNG_TABLE || trees[0].n_sites < 2) tile = 0;
    const long long S = trees ? trees[0].n_sites : 0;
    // A call whose state does not fit in device memory is cut into site tiles, run one after the other (each an
    // independent chain of N sweeps: the fixed-Q samplers couple the sites through nothing but the final sum).  The tile
    // is halved until a chain can be allocated.  The rate-updating samplers need all sites resident in every sweep (Q
    // depends on their sum): they are left to fail with the allocator's message.  With several ranks the tile size must
    // be the same everywhere (one all-reduce per tile), so it is only taken from PHYLOMAP_B200_SITE_TILE there.
    for (;;) {
      const long long ts = (tile > 0 && tile < S) ? tile : S;
      try {
        if (ts >= S) {
          std::unique_ptr<pm_chain> c(make_chain(variant, trees, ntrees, n, Q, pid, B, Omega, prior, nprior, N, opt, eg));
          c->run(N, out, N);
        } else {
          const int nc = ncols_of(variant, n);
          std::vector<double> part((size_t)N * nc), acc((size_t)N * nc, 0.0);
          for (long long s0 = 0; s0 < S; s0 += ts) {
            run_site_block(variant, trees, n, Q, pid, B, Omega, N, opt, eg, s0, std::min(ts, S - s0), part.data());
            for (size_t i = 0; i < acc.size(); i++) acc[i] += part[i];
          }
          std::copy(acc.begin(), acc.end(), out);
        }
        return;
      } catch (const Fail& f) {
        const bool oom = f.code == PM_ERR_CUDA && f.msg.find("cudaMalloc") != std::string::npos;
        if (!oom || !fixed_q || !single_process || ts < 64 || ntrees != 1 || opt->rng == PM_RNG_TABLE) throw;
        cudaGetLastError();
        pool().release();
        tile = (ts + 1) / 2;
      }
    }
  });
}

// A chain that evaluates log p(y | Q) and keeps no path state (pm_loglik, pm_expected_sumstats), with the copy of Q it reads.
// The chain machinery wants a uniformization pair (Omega, B) although neither computation uses it.
struct LoglikChain {
  std::vector<double> q, b;
  std::unique_ptr<pm_chain> c;
  LoglikChain(const pm_tree* x, int n, const double* Q, const double* pid, int parity_tips, const pm_options* opt)
      : q(Q, Q + (size_t)n * n), b((size_t)n * n, 0.0) {
    double om = 0;
    for (int i = 0; i < n; i++) om = std::max(om, 2 * std::fabs(q[i + (size_t)i * n]));
    if (!(om > 0)) om = 1;
    for (int i = 0; i < n; i++) for (int j = 0; j < n; j++) b[i + (size_t)j * n] = (i == j ? 1.0 : 0.0) + q[i + (size_t)j * n] / om;
    c.reset(make_chain(parity_tips ? V_LOGLIK_PARITY : V_LOGLIK, x, 1, n, q.data(), pid, b.data(), om, nullptr, 0, 0, opt, nullptr, true));
  }
};

// pm_expected_sumstats over sites [s0, s0 + count) of x (write: per branch and per node too).
void expected_block(const pm_tree* x, int n, const double* Q, const double* pid, int parity_tips, const pm_options* opt, long long s0,
                    long long count, bool write, double* stats, long long ld, double* ll, double* branch_stats, double* node_marginals) {
  pm_tree t = *x;
  t.n_sites = count;
  if (x->states_u8) t.states_u8 = x->states_u8 + s0 * (long long)x->n_tips;
  if (x->states) t.states = x->states + s0 * (long long)x->n_tips;
  LoglikChain(&t, n, Q, pid, parity_tips, opt).c->expected(write, stats, ld, ll, branch_stats, node_marginals);
}

}  // namespace

// ----------------------------------------------------------------------------------------------------------------
extern "C" {

void pm_default_options(pm_options* o) {
  memset(o, 0, sizeof *o);
  o->precision = PM_F64;
  o->mode = PM_MODE_PRODUCTION;
  o->rng = PM_RNG_PHILOX;
  o->seed = 1;
}

int32_t pm_ncols(int32_t variant, int32_t n) { return ncols_of(variant, n); }

int pm_maketreelistMCMC(const pm_tree* x, int32_t n, double* Q, const double* pid, double* B, double Omega, int32_t N,
                        const pm_options* opt, double* out, char* err, size_t errlen) {
  return one_call(PM_V_PLAIN, x, 1, n, Q, pid, B, Omega, N, nullptr, 0, opt, out, err, errlen);
}
int pm_SPARSEmaketreelistMCMC(const pm_tree* x, int32_t n, double* Q, const double* pid, double* B, double Omega,
                              int32_t N, const pm_options* opt, double* out, char* err, size_t errlen) {
  return one_call(PM_V_SPARSE, x, 1, n, Q, pid, B, Omega, N, nullptr, 0, opt, out, err, errlen);
}
int pm_maketreelistMCMC_bigtree(const pm_tree* x, int32_t n, double* Q, const double* pid, double* B, double Omega,
                                int32_t N, const pm_options* opt, double* out, char* err, size_t errlen) {
  return one_call(PM_V_BIGTREE, x, 1, n, Q, pid, B, Omega, N, nullptr, 0, opt, out, err, errlen);
}
int pm_maketreelistMCMCbf(const pm_tree* x, int32_t n, double* Q, const double* pid, double* B, double Omega, int32_t N,
                          const double* prior, int32_t nprior, const pm_options* opt, double* out, char* err,
                          size_t errlen) {
  return one_call(PM_V_BF, x, 1, n, Q, pid, B, Omega, N, prior, nprior, opt, out, err, errlen);
}
int pm_maketreelistMCMCks(const pm_tree* x, int32_t n, double* Q, const double* pid, double* B, double Omega, int32_t N,
                          const double* prior, int32_t nprior, const pm_options* opt, double* out, char* err,
                          size_t errlen) {
  return one_call(PM_V_KS, x, 1, n, Q, pid, B, Omega, N, prior, nprior, opt, out, err, errlen);
}
int pm_maketreelistMCMCmt(const pm_tree* trees, int32_t ntrees, int32_t n, double* Q, const double* pid, double* B,
                          double Omega, int32_t N, const double* prior, int32_t nprior, const pm_options* opt,
                          double* out, char* err, size_t errlen) {
  return one_call(PM_V_MT, trees, ntrees, n, Q, pid, B, Omega, N, prior, nprior, opt, out, err, errlen);
}
int pm_maketreelistMCMCksmt(const pm_tree* trees, int32_t ntrees, int32_t n, double* Q, const double* pid, double* B,
                            double Omega, int32_t N, const double* prior, int32_t nprior, const pm_options* opt,
                            double* out, char* err, size_t errlen) {
  return one_call(PM_V_KSMT, trees, ntrees, n, Q, pid, B, Omega, N, prior, nprior, opt, out, err, errlen);
}

int pm_maketreelistEXP(const pm_tree* x, int32_t n, double* Q, const double* pid, int32_t N, const double* lefts,
                       const double* rights, const double* d, const pm_options* opt, double* out, char* err, size_t errlen) {
  EigenIn eg{lefts, rights, d};
  return one_call(PM_V_EXP, x, 1, n, Q, pid, nullptr, 0.0, N, nullptr, 0, opt, out, err, errlen, &eg);
}

int pm_maketreelistMCMC2sDICt(const pm_tree* x, int32_t n, double* Q, const double* pid, double* B, double Omega, int32_t N,
                              const double* prior, int32_t nprior, const pm_options* opt, double* out, char* err,
                              size_t errlen) {
  return one_call(PM_V_DIC2S, x, 1, n, Q, pid, B, Omega, N, prior, nprior, opt, out, err, errlen);
}
int pm_maketreelistMCMCksDICt(const pm_tree* x, int32_t n, double* Q, const double* pid, double* B, double Omega, int32_t N,
                              const double* prior, int32_t nprior, const pm_options* opt, double* out, char* err,
                              size_t errlen) {
  return one_call(PM_V_DICKS, x, 1, n, Q, pid, B, Omega, N, prior, nprior, opt, out, err, errlen);
}

int pm_loglik(const pm_tree* x, int32_t n, const double* Q, const double* pid, int32_t parity_tips, const pm_options* opt,
              double* out, char* err, size_t errlen) {
  return guarded(err, errlen, [&] {
    if (!x || !Q || !pid || !out) fail(PM_ERR_ARG, "null argument");
    if (n < 2 || n > PM_DIC_NMAX) fail(PM_ERR_ARG, "number of states must be in 2..%d", PM_DIC_NMAX);
    if (parity_tips && (n & 1)) fail(PM_ERR_ARG, "parity tip partials need an even number of states");
    *out = LoglikChain(x, n, Q, pid, parity_tips, opt).c->loglik();
  });
}

int pm_expected_sumstats(const pm_tree* x, int32_t n, const double* Q, const double* pid, int32_t parity_tips, const int64_t* sites,
                         int64_t nsel, const pm_options* opt, double* stats, double* loglik, double* branch_stats, double* node_marginals,
                         char* err, size_t errlen) {
  return guarded(err, errlen, [&] {
    if (!x || !Q || !pid) fail(PM_ERR_ARG, "null argument");
    if (n < 2 || n > PM_DIC_NMAX) fail(PM_ERR_ARG, "number of states must be in 2..%d", PM_DIC_NMAX);
    if (parity_tips && (n & 1)) fail(PM_ERR_ARG, "parity tip partials need an even number of states");
    if (x->n_sites < 1) fail(PM_ERR_ARG, "n_sites must be >= 1");
    if (!x->states && !x->states_u8) fail(PM_ERR_ARG, "states missing");
    if (nsel < 0 || (nsel > 0 && !sites)) fail(PM_ERR_ARG, "bad site selection");
    for (int64_t i = 0; i < nsel; i++)
      if (sites[i] < 0 || sites[i] >= x->n_sites) fail(PM_ERR_ARG, "site %lld out of range (%lld sites)", (long long)sites[i], (long long)x->n_sites);
    pm_options def;
    if (!opt) { pm_default_options(&def); opt = &def; }
    const long long S = x->n_sites, T = x->n_tips, E = x->n_edges, NK = (long long)n * n;
    const bool main_pass = stats || loglik, sel_pass = nsel > 0 && (branch_stats || node_marginals);
    if (!main_pass && !sel_pass) return;
    // Sites run in tiles whose per-site device state (partials, tip codes, node states, outputs) takes at most half of the
    // free memory beside the per-branch matrices.  A site's result does not depend on its tile.
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) fail(PM_ERR_CUDA, "no CUDA device (there is no CPU fallback)");
    CK(cudaSetDevice(opt->device));
    size_t free_b = 0, total_b = 0;
    CK(cudaMemGetInfo(&free_b, &total_b));
    const long long rsz = opt->precision == PM_F32 ? 4 : 8;
    const long long fixed = E * (NK * NK + NK) * rsz, avail = (long long)(free_b / 2) - fixed;
    const long long env_tile = read_switches().site_tile;
    const auto tile_of = [&](long long per_site, long long count) {
      long long ts = std::max<long long>(32, avail / per_site);
      if (env_tile > 0) ts = std::min(ts, env_tile);
      return std::min(ts, count);
    };
    const long long base = (T - 1) * n * rsz + (2 * T - 1) + T + (NK + 1) * 8;
    if (main_pass) {
      const long long ts = tile_of(base, S);
      for (long long s0 = 0; s0 < S; s0 += ts)
        expected_block(x, n, Q, pid, parity_tips, opt, s0, std::min(ts, S - s0), false, stats ? stats + s0 : nullptr, S,
                       loglik ? loglik + s0 : nullptr, nullptr, nullptr);
    }
    if (sel_pass) {
      // the selected sites as a problem of their own: their tip rows gathered in the order of `sites`
      const bool u8 = x->states_u8 != nullptr;
      std::vector<uint8_t> g8(u8 ? (size_t)nsel * T : 0);
      std::vector<int32_t> g32(u8 ? 0 : (size_t)nsel * T);
      for (int64_t i = 0; i < nsel; i++) {
        if (u8) std::copy(x->states_u8 + sites[i] * T, x->states_u8 + (sites[i] + 1) * T, g8.begin() + i * T);
        else std::copy(x->states + sites[i] * T, x->states + (sites[i] + 1) * T, g32.begin() + i * T);
      }
      pm_tree xs = *x;
      xs.n_sites = nsel;
      xs.states_u8 = u8 ? g8.data() : nullptr;
      xs.states = u8 ? nullptr : g32.data();
      const long long ts = tile_of(base + (E * NK + (2 * T - 1) * n) * 8, nsel);
      for (long long s0 = 0; s0 < nsel; s0 += ts) {
        const long long cnt = std::min(ts, nsel - s0);
        // (outputs the caller did not ask for still have a device buffer: the kernel writes both)
        expected_block(&xs, n, Q, pid, parity_tips, opt, s0, cnt, true, nullptr, cnt, nullptr,
                       branch_stats ? branch_stats + s0 * E * NK : nullptr, node_marginals ? node_marginals + s0 * (2 * T - 1) * n : nullptr);
      }
    }
  });
}

int pm_debug_clade_schedule(const int32_t* edge, int32_t n_edges, int32_t n_tips, const int32_t* nen, const int32_t* nodelist,
                            int32_t root, int32_t nwarps, int32_t clade_max, int64_t* stats, char* err, size_t errlen) {
  return guarded(err, errlen, [&] {
    if (!edge || !nen || !nodelist || !stats || nwarps < 1) fail(PM_ERR_ARG, "bad argument");
    pm::host::Schedule sch;
    try { pm::host::build_schedule(n_tips, n_edges, edge, nen, nodelist, root, false, sch); }
    catch (const std::string& msg) { fail(PM_ERR_ARG, "%s", msg.c_str()); }
    pm::host::CladeSchedule cs;
    pm::host::build_clade_schedule(sch, nwarps, clade_max, cs);
    const int T = n_tips, NN = 2 * T - 1;
    // bottom-up: every internal node exactly once; inside a warp's sequence both children of a node are tips, the node
    // just before (flag 1 / 2) or an earlier node of the SAME warp (flag 4 / 8); a top node's children are complete
    std::vector<int> owner(NN, -2), posn(NN, -1);  // -2 unseen, -1 top, else warp
    const int n1 = cs.warp_off[nwarps];
    long long lo = 1LL << 60, hi = 0, nprev = 0;
    for (int w = 0; w < nwarps; w++) {
      lo = std::min<long long>(lo, cs.warp_off[w + 1] - cs.warp_off[w]);
      hi = std::max<long long>(hi, cs.warp_off[w + 1] - cs.warp_off[w]);
      int prev = -1;
      for (int i = cs.warp_off[w]; i < cs.warp_off[w + 1]; i++) {
        const int* en = &cs.entries[(size_t)8 * i];
        const int v = en[0], fl = en[5];
        if (v < T || v >= NN || owner[v] != -2) fail(PM_ERR_ARG, "node %d scheduled twice or out of range", v);
        const int kids[2] = {en[1], en[3]};
        for (int c = 0; c < 2; c++) {
          const int k = kids[c], isprev = fl & (c ? 2 : 1), isload = fl & (c ? 8 : 4);
          if (k < T) { if (isprev || isload) fail(PM_ERR_ARG, "tip child of %d flagged", v); continue; }
          if (owner[k] != w) fail(PM_ERR_ARG, "child %d of %d is not an earlier node of the same warp", k, v);
          if (isprev ? (k != prev) : (!isload || posn[k] >= i - 1)) fail(PM_ERR_ARG, "flags of node %d", v);
          if (isprev) nprev++;
        }
        if ((fl & 4) && (fl & 8)) fail(PM_ERR_ARG, "node %d would load both children", v);
        owner[v] = w; posn[v] = i; prev = v;
      }
    }
    const int ntop = (int)cs.entries.size() / 8 - n1;
    for (size_t l = 0; l + 1 < cs.top_off.size(); l++)
      for (int i = cs.top_off[l]; i < cs.top_off[l + 1]; i++) {
        const int* en = &cs.entries[(size_t)8 * i];
        const int v = en[0];
        if (v < T || v >= NN || owner[v] != -2) fail(PM_ERR_ARG, "top node %d scheduled twice", v);
        const int kids[2] = {en[1], en[3]};
        for (int k : kids) if (k >= T && (owner[k] == -2 || (owner[k] == -1 && posn[k] >= cs.top_off[l]))) fail(PM_ERR_ARG, "top node %d before its child %d", v, k);
        owner[v] = -1; posn[v] = i;
      }
    for (int v = T; v < NN; v++) if (owner[v] == -2) fail(PM_ERR_ARG, "node %d never scheduled", v);
    // top-down: every internal node but the root exactly once, after its parent
    std::vector<int> seen(NN, 0);
    seen[sch.root] = 1;
    for (size_t l = 0; l + 1 < cs.down_top_off.size(); l++) {
      for (int i = cs.down_top_off[l]; i < cs.down_top_off[l + 1]; i++) {
        const int* en = &cs.down_top[(size_t)4 * i];
        if (seen[en[0]] || !seen[en[1]] || seen[en[1]] > (int)l + 1) fail(PM_ERR_ARG, "top-down order of node %d", en[0]);
      }
      for (int i = cs.down_top_off[l]; i < cs.down_top_off[l + 1]; i++) seen[cs.down_top[(size_t)4 * i]] = (int)l + 2;
    }
    for (int w = 0; w < nwarps; w++) {
      int prev = -1;
      for (int i = cs.down_warp_off[w]; i < cs.down_warp_off[w + 1]; i++) {
        const int* en = &cs.down_seq[(size_t)4 * i];
        if (seen[en[0]] || !seen[en[1]]) fail(PM_ERR_ARG, "pre-order of node %d", en[0]);
        if (en[3] && en[1] != prev) fail(PM_ERR_ARG, "parent-is-previous flag of node %d", en[0]);
        if (sch.e_child[en[2]] != en[0] || sch.e_parent[en[2]] != en[1]) fail(PM_ERR_ARG, "edge of node %d", en[0]);
        seen[en[0]] = 1 << 20; prev = en[0];
      }
    }
    for (int v = T; v < NN; v++) if (!seen[v]) fail(PM_ERR_ARG, "node %d never drawn", v);
    stats[0] = n1; stats[1] = ntop; stats[2] = (long long)cs.top_off.size() - 1; stats[3] = lo; stats[4] = hi; stats[5] = nprev;
    stats[6] = cs.down_warp_off[nwarps]; stats[7] = (long long)cs.down_top.size() / 4;
  });
}

int pm_tree_order(const int32_t* edge, int32_t n_edges, int32_t n_tips, int32_t* nen, int32_t* nodelist, int32_t* root,
                  char* err, size_t errlen) {
  return guarded(err, errlen, [&] {
    if (!edge || !nen || !nodelist || !root) fail(PM_ERR_ARG, "null argument");
    pm::host::tree_order(edge, n_edges, n_tips, nen, nodelist, root);
  });
}

int pm_chain_create(int32_t variant, const pm_tree* trees, int32_t ntrees, int32_t n, double* Q, const double* pid,
                    double* B, double Omega, const double* prior, int32_t nprior, int32_t N_total, const pm_options* opt,
                    pm_chain** out, char* err, size_t errlen) {
  return guarded(err, errlen, [&] {
    if (!out) fail(PM_ERR_ARG, "null output");
    *out = make_chain(variant, trees, ntrees, n, Q, pid, B, Omega, prior, nprior, N_total, opt);
  });
}
int pm_chain_run(pm_chain* c, int32_t count, double* out, int64_t ld, char* err, size_t errlen) {
  return guarded(err, errlen, [&] {
    if (!c || (!out && count > 0)) fail(PM_ERR_ARG, "null argument");
    c->run(count, out, ld);
  });
}
int64_t pm_chain_state_bytes(pm_chain* c) { return c ? c->state_bytes() : 0; }
int pm_chain_export_state(pm_chain* c, void* buf, int64_t bytes, char* err, size_t errlen) {
  return guarded(err, errlen, [&] {
    if (!c) fail(PM_ERR_ARG, "null argument");
    c->export_state(buf, bytes);
  });
}
int pm_chain_import_state(pm_chain* c, const void* buf, int64_t bytes, char* err, size_t errlen) {
  return guarded(err, errlen, [&] {
    if (!c) fail(PM_ERR_ARG, "null argument");
    c->import_state(buf, bytes);
  });
}
int pm_chain_time_prune(pm_chain* c, int32_t tree, int32_t reps, float* ms_per_pass, char* err, size_t errlen) {
  return guarded(err, errlen, [&] {
    if (!c || !ms_per_pass) fail(PM_ERR_ARG, "null argument");
    *ms_per_pass = c->time_prune(tree, reps);
  });
}
void pm_chain_kernel_times(pm_chain* c, double ms[4], int64_t* launches) {
  for (int i = 0; i < 4; i++) ms[i] = c->kernel_ms[i];
  if (launches) *launches = c->launches;
}
void pm_chain_enable_timing(pm_chain* c, int32_t on) { c->timing = on != 0; }
void pm_chain_overheads(pm_chain* c, double ms[2]) { ms[0] = c->comm_ms; ms[1] = c->host_update_ms; }
int pm_chain_get_node_states(pm_chain* c, int32_t tree, int32_t* out) {
  return guarded(nullptr, 0, [&] { c->node_states(tree, out); });
}
int pm_chain_get_piece_counts(pm_chain* c, int32_t tree, int32_t* out) {
  return guarded(nullptr, 0, [&] { c->piece_counts(tree, out); });
}
int pm_chain_get_path(pm_chain* c, int32_t tree, int64_t site, int32_t e, double* len, int32_t* st, int32_t cap) {
  int r = -1;
  const int rc = guarded(nullptr, 0, [&] { r = c->path(tree, site, e, len, st, cap); });
  return rc == PM_OK ? r : -rc;
}
int pm_chain_get_maps(pm_chain* c, int32_t tree, const int64_t* sites, int64_t nsel, int64_t* off, double* len, int32_t* st,
                      int64_t cap, char* err, size_t errlen) {
  return guarded(err, errlen, [&] {
    if (!c) fail(PM_ERR_ARG, "null argument");
    c->maps(tree, sites, nsel, off, len, st, cap);
  });
}
int pm_chain_get_partials(pm_chain* c, int32_t tree, int64_t site, double* out) {
  return guarded(nullptr, 0, [&] { c->partials(tree, site, out); });
}
int64_t pm_chain_device_bytes(pm_chain* c) { return c->dev_bytes; }
int pm_nccl_unique_id(void* out128, char* err, size_t errlen) {
  return guarded(err, errlen, [&] {
    if (!out128) fail(PM_ERR_ARG, "null argument");
    auto& api = pm::host::NcclApi::get();
    if (!api.ok()) fail(PM_ERR_CUDA, "NCCL could not be loaded: %s", api.why.c_str());
    pm::host::NcclApi::UniqueId id;
    const int rc = api.GetUniqueId(&id);
    if (rc != 0) fail(PM_ERR_CUDA, "ncclGetUniqueId failed: %s", api.error(rc).c_str());
    memcpy(out128, &id, sizeof id);
  });
}
int32_t pm_chain_acceptance(pm_chain* c, int64_t* proposed, int64_t* accepted, int32_t cap) {
  const int32_t np = (int32_t)c->rate_proposed.size();
  for (int32_t i = 0; i < np && i < cap; i++) { proposed[i] = c->rate_proposed[i]; accepted[i] = c->rate_accepted[i]; }
  return np;
}
void pm_chain_destroy(pm_chain* c) { delete c; }

void pm_rng_probe(uint32_t seed, int32_t kind, int32_t n, double a, double b, double* out) {
  pm::host::MersenneR g(seed);
  for (int i = 0; i < n; i++) {
    switch (kind) {
      case 0: out[i] = g.next(); break;
      case 1: out[i] = pm::host::r_exp_rand(g); break;
      case 2: out[i] = pm::host::r_norm_rand(g); break;
      default: out[i] = pm::host::r_rgamma(g, a, b); break;
    }
  }
}

void pm_release_cached_memory(void) { pool().release(); }

int pm_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return -PM_ERR_CUDA;
  int ok = 0;
  for (int d = 0; d < n; d++) {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, d) == cudaSuccess && p.major == 10) ok++;
  }
  return ok;
}
const char* pm_version(void) { return "phylomap_b200 0.1 (sm_100a)"; }

}  // extern "C"

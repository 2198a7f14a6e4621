// Drop-in replacement for the reference's src/phylomap.cpp: the ten functions its generated glue expects
// (src/RcppExports.cpp:10,33,56,79,105,131,158,184,210,236 declare them, src/phylomap.cpp:822,891,942,1258,1802,2267,
// 2722,3001,3183,3300 define them), implemented on libphylomap_b200's C ABI (include/phylomap_b200.h).  The package's
// src/RcppExports.cpp, R/RcppExports.R and every R wrapper stay as they are: same `.Call` symbols, same arguments, same
// returned matrices, Q and B rewritten in place by the rate-updating samplers like the reference (:1284).
//
// Build inside the R package (src/Makevars, see INTEGRATION.md):  replace src/phylomap.cpp by this file and add
//   PKG_CPPFLAGS += -I<repo>/include      PKG_LIBS += -L<repo>/phylomap_b200 -lphylomap_b200 -Wl,-rpath,<repo>/phylomap_b200
// It uses plain Rcpp only (no Armadillo).  In this repository it is compiled against the stand-in headers of
// oracle/standin/ together with oracle/shim_glue.cpp, the package's `.Call` glue as Rcpp generates it into
// src/RcppExports.cpp (oracle/Makefile, target `shim`), and driven through the `.Call` symbols by tests/test_shim.py.
//
// The site axis (new): x$states may be a matrix with one COLUMN per character (ntips x nsites); its column-major storage
// is already the [site][tip] order pm_tree.states wants, so it is passed through untouched.  A plain vector is the
// reference's one-character call.
//
// Run-time switches (environment): PHYLOMAP_B200_PRECISION = f64 (default) | f32, PHYLOMAP_B200_MODE = production
// (default) | deterministic, PHYLOMAP_B200_DEVICE = CUDA ordinal.  set.seed() keeps controlling the run: the 64-bit
// seed of the device generator and of the host-side rate draws comes from two unif_rand() calls under RNGScope.
#include <Rcpp.h>

#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "phylomap_b200.h"

using namespace Rcpp;

namespace {

// x$maps / x$mapnames / x$edge / x$states [/ x$edge.length] -> pm_tree (fields read by the reference at :896-910)
struct FlatTree {
  IntegerMatrix edge;
  IntegerVector states, nen, nodelist;
  NumericVector edge_length;
  std::vector<int64_t> off;
  std::vector<double> len;
  std::vector<int32_t> st;
  pm_tree t;

  FlatTree(const List& x, const IntegerVector& nen_, const IntegerVector& nodelist_, int root)
      : edge(as<IntegerMatrix>(x["edge"])), states(as<IntegerVector>(x["states"])), nen(nen_), nodelist(nodelist_) {
    List maps = x["maps"], names = x["mapnames"];
    if (maps.size() != names.size() || maps.size() != edge.nrow()) stop("maps, mapnames and edge disagree on the number of branches");
    off.push_back(0);
    for (int e = 0; e < maps.size(); e++) {
      NumericVector m = maps[e];
      IntegerVector s = names[e];
      if (m.size() != s.size()) stop("maps and mapnames disagree on a branch");
      for (int k = 0; k < m.size(); k++) { len.push_back(m[k]); st.push_back(s[k]); }
      off.push_back((int64_t)len.size());
    }
    SEXP sx = x["states"];
    std::memset(&t, 0, sizeof t);
    t.n_edges = edge.nrow();
    t.n_tips = Rf_isMatrix(sx) ? Rf_nrows(sx) : (int)states.size();
    t.n_sites = Rf_isMatrix(sx) ? Rf_ncols(sx) : 1;   // one column per character; column-major = [site][tip]
    t.edge = edge.begin(); t.nen = nen.begin(); t.nodelist = nodelist.begin(); t.root = root;
    t.maps_off = off.data(); t.maps_len = len.data(); t.maps_state = st.data();
    t.states = states.begin(); t.states_u8 = NULL;
    if (x.containsElementNamed("edge.length")) { edge_length = as<NumericVector>(x["edge.length"]); t.edge_length = edge_length.begin(); }
  }
};

// must run under an RNGScope: draws the seed from R's stream
pm_options options_from_env() {
  pm_options o;
  pm_default_options(&o);
  const char* p = std::getenv("PHYLOMAP_B200_PRECISION"); if (p && !std::strcmp(p, "f32")) o.precision = PM_F32;
  const char* m = std::getenv("PHYLOMAP_B200_MODE");      if (m && !std::strcmp(m, "deterministic")) o.mode = PM_MODE_DETERMINISTIC;
  const char* d = std::getenv("PHYLOMAP_B200_DEVICE");    if (d) o.device = std::atoi(d);
  const uint64_t hi = (uint64_t)(unif_rand() * 4294967296.0), lo = (uint64_t)(unif_rand() * 4294967296.0);
  o.seed = (hi << 32) | lo;
  return o;
}

void check(int rc, const char* err) { if (rc != PM_OK) stop(std::string(err)); }   // -> an R error, like BEGIN_RCPP / END_RCPP

typedef int (*fixed_fn)(const pm_tree*, int32_t, double*, const double*, double*, double, int32_t, const pm_options*, double*, char*, size_t);
typedef int (*prior_fn)(const pm_tree*, int32_t, double*, const double*, double*, double, int32_t, const double*, int32_t, const pm_options*,
                        double*, char*, size_t);
typedef int (*multi_fn)(const pm_tree*, int32_t, int32_t, double*, const double*, double*, double, int32_t, const double*, int32_t,
                        const pm_options*, double*, char*, size_t);

NumericMatrix run_fixed(fixed_fn fn, int variant, List& x, NumericMatrix& Q, NumericVector& pid, NumericMatrix& B, double Omega,
                        IntegerVector& nen, IntegerVector& nodelist, int root, int N) {
  RNGScope scope;
  FlatTree ft(x, nen, nodelist, root);
  pm_options o = options_from_env();
  const int n = Q.nrow();
  NumericMatrix out(N, pm_ncols(variant, n));   // column-major, like arma::mat dwelltimes (:926)
  char err[512] = "";
  check(fn(&ft.t, n, Q.begin(), pid.begin(), B.begin(), Omega, N, &o, out.begin(), err, sizeof err), err);
  return out;
}

NumericMatrix run_prior(prior_fn fn, int variant, List& x, NumericMatrix& Q, NumericVector& pid, NumericMatrix& B, double Omega,
                        IntegerVector& nen, IntegerVector& nodelist, int root, int N, NumericVector& prior) {
  RNGScope scope;
  FlatTree ft(x, nen, nodelist, root);
  pm_options o = options_from_env();
  const int n = Q.nrow();
  NumericMatrix out(N, pm_ncols(variant, n));
  char err[512] = "";
  // Q.begin() / B.begin() are the caller's matrices: the in-place rewrite of the reference is preserved
  check(fn(&ft.t, n, Q.begin(), pid.begin(), B.begin(), Omega, N, prior.begin(), (int)prior.size(), &o, out.begin(), err, sizeof err), err);
  return out;
}

// x: list of trees; nen / nodelist_m: one ROW per tree (R/sumstatMCMCmt.R:27-33); roots: one root per tree
NumericMatrix run_multi(multi_fn fn, int variant, List& x, NumericMatrix& Q, NumericVector& pid, NumericMatrix& B, double Omega,
                        IntegerMatrix& nen, IntegerMatrix& nodelist_m, IntegerVector roots, int N, NumericVector& prior) {
  RNGScope scope;
  const int nt = (int)x.size();
  if (nen.nrow() != nt || nodelist_m.nrow() != nt || roots.size() != nt) stop("nen, nodelist and roots need one row / entry per tree");
  std::vector<FlatTree*> fts;
  std::vector<pm_tree> trees;
  struct Cleanup { std::vector<FlatTree*>& v; ~Cleanup() { for (size_t i = 0; i < v.size(); i++) delete v[i]; } } cleanup = {fts};
  for (int i = 0; i < nt; i++) {
    IntegerVector ne_i(nen.ncol()), nl_i(nodelist_m.ncol());
    for (int j = 0; j < nen.ncol(); j++) ne_i[j] = nen(i, j);
    for (int j = 0; j < nodelist_m.ncol(); j++) nl_i[j] = nodelist_m(i, j);
    List xi = x[i];
    fts.push_back(new FlatTree(xi, ne_i, nl_i, roots[i]));
    trees.push_back(fts.back()->t);
  }
  pm_options o = options_from_env();
  const int n = Q.nrow();
  NumericMatrix out(N, pm_ncols(variant, n));
  char err[512] = "";
  check(fn(trees.data(), nt, n, Q.begin(), pid.begin(), B.begin(), Omega, N, prior.begin(), (int)prior.size(), &o, out.begin(), err,
           sizeof err), err);
  return out;
}

}  // namespace

// ---- the reference's exported functions (signatures as in src/RcppExports.cpp) ----------------------------------------

// [[Rcpp::export]]
NumericMatrix SPARSEmaketreelistMCMC(List& x, NumericMatrix& Q, NumericVector& pid, NumericMatrix& B, double Omega, IntegerVector& nen,
                                     IntegerVector& nodelist, int root, int N) {
  return run_fixed(pm_SPARSEmaketreelistMCMC, PM_V_SPARSE, x, Q, pid, B, Omega, nen, nodelist, root, N);
}

// [[Rcpp::export]]
NumericMatrix maketreelistMCMC(List& x, NumericMatrix& Q, NumericVector& pid, NumericMatrix& B, double Omega, IntegerVector& nen,
                               IntegerVector& nodelist, int root, int N) {
  return run_fixed(pm_maketreelistMCMC, PM_V_PLAIN, x, Q, pid, B, Omega, nen, nodelist, root, N);
}

// [[Rcpp::export]]
NumericMatrix maketreelistMCMC_bigtree(List& x, NumericMatrix& Q, NumericVector& pid, NumericMatrix& B, double Omega, IntegerVector& nen,
                                       IntegerVector& nodelist, int root, int N) {
  return run_fixed(pm_maketreelistMCMC_bigtree, PM_V_BIGTREE, x, Q, pid, B, Omega, nen, nodelist, root, N);
}

// [[Rcpp::export]]
NumericMatrix maketreelistMCMCbf(List& x, NumericMatrix& Q, NumericVector& pid, NumericMatrix& B, double Omega, IntegerVector& nen,
                                 IntegerVector& nodelist, int root, int N, NumericVector& prior) {
  return run_prior(pm_maketreelistMCMCbf, PM_V_BF, x, Q, pid, B, Omega, nen, nodelist, root, N, prior);
}

// [[Rcpp::export]]
NumericMatrix maketreelistMCMCks(List& x, NumericMatrix& Q, NumericVector& pid, NumericMatrix& B, double Omega, IntegerVector& nen,
                                 IntegerVector& nodelist, int root, int N, NumericVector& prior) {
  return run_prior(pm_maketreelistMCMCks, PM_V_KS, x, Q, pid, B, Omega, nen, nodelist, root, N, prior);
}

// [[Rcpp::export]]
NumericMatrix maketreelistMCMC2sDICt(List& x, NumericMatrix& Q, NumericVector& pid, NumericMatrix& B, double Omega, IntegerVector& nen,
                                     IntegerVector& nodelist, int root, int N, NumericVector& prior) {
  return run_prior(pm_maketreelistMCMC2sDICt, PM_V_DIC2S, x, Q, pid, B, Omega, nen, nodelist, root, N, prior);
}

// [[Rcpp::export]]
NumericMatrix maketreelistMCMCksDICt(List& x, NumericMatrix& Q, NumericVector& pid, NumericMatrix& B, double Omega, IntegerVector& nen,
                                     IntegerVector& nodelist, int root, int N, NumericVector& prior) {
  return run_prior(pm_maketreelistMCMCksDICt, PM_V_DICKS, x, Q, pid, B, Omega, nen, nodelist, root, N, prior);
}

// [[Rcpp::export]]
NumericMatrix maketreelistMCMCmt(List& x, NumericMatrix& Q, NumericVector& pid, NumericMatrix& B, double Omega, IntegerMatrix& nen_m,
                                 IntegerMatrix& nodelist_m, IntegerVector roots, int N, NumericVector& prior) {
  return run_multi(pm_maketreelistMCMCmt, PM_V_MT, x, Q, pid, B, Omega, nen_m, nodelist_m, roots, N, prior);
}

// [[Rcpp::export]]
NumericMatrix maketreelistMCMCksmt(List& x, NumericMatrix& Q, NumericVector& pid, NumericMatrix& B, double Omega, IntegerMatrix& nen_m,
                                   IntegerMatrix& nodelist_m, IntegerVector roots, int N, NumericVector& prior) {
  return run_multi(pm_maketreelistMCMCksmt, PM_V_KSMT, x, Q, pid, B, Omega, nen_m, nodelist_m, roots, N, prior);
}

// [[Rcpp::export]]
NumericMatrix maketreelistEXP(List& x, NumericMatrix& Q, NumericVector& pid, IntegerVector& nen, IntegerVector& nodelist, int root, int N,
                              NumericMatrix& lefts, NumericMatrix& rights, NumericMatrix& d) {
  RNGScope scope;
  FlatTree ft(x, nen, nodelist, root);
  pm_options o = options_from_env();
  const int n = Q.nrow();
  NumericMatrix out(N, pm_ncols(PM_V_EXP, n));
  char err[512] = "";
  check(pm_maketreelistEXP(&ft.t, n, Q.begin(), pid.begin(), N, lefts.begin(), rights.begin(), d.begin(), &o, out.begin(), err, sizeof err), err);
  return out;
}

// ---- two additions a maintainer can export next to them (not in the reference's NAMESPACE) ----------------------------

// O(E) replacement of pruningwiseedgeorder / makenodelist / myreorder (R/sumstatMCMC.R:1-18, O(E^2) R loops copied into every
// wrapper file): list(nen = , nodelist = , root = ).
// [[Rcpp::export]]
List phylomap_tree_order(IntegerMatrix& edge, int ntips) {
  const int E = edge.nrow();
  IntegerVector nen(E), nodelist(ntips - 2 > 0 ? ntips - 2 : 0);
  int root = 0;
  char err[512] = "";
  check(pm_tree_order(edge.begin(), E, ntips, nen.begin(), nodelist.begin(), &root, err, sizeof err), err);
  return List::create(Named("nen") = nen, Named("nodelist") = nodelist, Named("root") = root);
}

// log p(y | Q) summed over the characters: the expm-per-branch + node loop of make2stateDIC / make4stateDIC(big)
// (R/sourceme.R:141-177, 248-284, 445-516) as one call.  D <- -2 * phylomap_loglik(atree, Q, pid, nen, nodelist, root, FALSE)
// [[Rcpp::export]]
double phylomap_loglik(List& x, NumericMatrix& Q, NumericVector& pid, IntegerVector& nen, IntegerVector& nodelist, int root, bool parity_tips) {
  RNGScope scope;
  FlatTree ft(x, nen, nodelist, root);
  pm_options o = options_from_env();
  double ll = 0;
  char err[512] = "";
  check(pm_loglik(&ft.t, Q.nrow(), Q.begin(), pid.begin(), parity_tips ? 1 : 0, &o, &ll, err, sizeof err), err);
  return ll;
}

// TEST INFRASTRUCTURE ONLY.  The `.Call` glue of the package's ten exported functions, written the way
// Rcpp::compileAttributes() generates src/RcppExports.cpp, against the stand-in headers of oracle/standin/.  Linked with
// shim/phylomap_b200_shim.cpp it gives oracle/_ref/libphylomap_shim.so the same `phylomap_<fn>` symbols, argument order
// and argument conversions (a `T&` parameter shares the caller's object, so Q and B are rewritten in place) that an R
// session reaches, without the R package's sources (oracle/Makefile, target `shim`; tests/test_shim.py).  The declarations
// below must be the shim's definitions (a mismatch leaves the `.Call` symbol unresolved when the library loads), and those
// are pinned to the package's generated glue by tests/golden/shim/call_signatures.json (tests/test_shim.py).
#include <Rcpp.h>

using namespace Rcpp;

#define PM_IN(T, name) Rcpp::traits::input_parameter<T>::type name(name##SEXP)

#define PM_FIXED(fn)                                                                                                     \
  NumericMatrix fn(List& x, NumericMatrix& Q, NumericVector& pid, NumericMatrix& B, double Omega, IntegerVector& nen,   \
                   IntegerVector& nodelist, int root, int N);                                                            \
  RcppExport SEXP phylomap_##fn(SEXP xSEXP, SEXP QSEXP, SEXP pidSEXP, SEXP BSEXP, SEXP OmegaSEXP, SEXP nenSEXP,         \
                                SEXP nodelistSEXP, SEXP rootSEXP, SEXP NSEXP) {                                          \
    BEGIN_RCPP                                                                                                           \
    Rcpp::RNGScope rcpp_rngScope_gen;                                                                                    \
    PM_IN(List&, x); PM_IN(NumericMatrix&, Q); PM_IN(NumericVector&, pid); PM_IN(NumericMatrix&, B);                     \
    PM_IN(double, Omega); PM_IN(IntegerVector&, nen); PM_IN(IntegerVector&, nodelist); PM_IN(int, root);                 \
    PM_IN(int, N);                                                                                                       \
    return Rcpp::wrap(fn(x, Q, pid, B, Omega, nen, nodelist, root, N));                                                  \
    END_RCPP                                                                                                             \
  }

#define PM_PRIOR(fn)                                                                                                     \
  NumericMatrix fn(List& x, NumericMatrix& Q, NumericVector& pid, NumericMatrix& B, double Omega, IntegerVector& nen,   \
                   IntegerVector& nodelist, int root, int N, NumericVector& prior);                                      \
  RcppExport SEXP phylomap_##fn(SEXP xSEXP, SEXP QSEXP, SEXP pidSEXP, SEXP BSEXP, SEXP OmegaSEXP, SEXP nenSEXP,         \
                                SEXP nodelistSEXP, SEXP rootSEXP, SEXP NSEXP, SEXP priorSEXP) {                          \
    BEGIN_RCPP                                                                                                           \
    Rcpp::RNGScope rcpp_rngScope_gen;                                                                                    \
    PM_IN(List&, x); PM_IN(NumericMatrix&, Q); PM_IN(NumericVector&, pid); PM_IN(NumericMatrix&, B);                     \
    PM_IN(double, Omega); PM_IN(IntegerVector&, nen); PM_IN(IntegerVector&, nodelist); PM_IN(int, root);                 \
    PM_IN(int, N); PM_IN(NumericVector&, prior);                                                                         \
    return Rcpp::wrap(fn(x, Q, pid, B, Omega, nen, nodelist, root, N, prior));                                           \
    END_RCPP                                                                                                             \
  }

#define PM_MULTI(fn)                                                                                                     \
  NumericMatrix fn(List& x, NumericMatrix& Q, NumericVector& pid, NumericMatrix& B, double Omega, IntegerMatrix& nen_m, \
                   IntegerMatrix& nodelist_m, IntegerVector roots, int N, NumericVector& prior);                         \
  RcppExport SEXP phylomap_##fn(SEXP xSEXP, SEXP QSEXP, SEXP pidSEXP, SEXP BSEXP, SEXP OmegaSEXP, SEXP nen_mSEXP,       \
                                SEXP nodelist_mSEXP, SEXP rootsSEXP, SEXP NSEXP, SEXP priorSEXP) {                       \
    BEGIN_RCPP                                                                                                           \
    Rcpp::RNGScope rcpp_rngScope_gen;                                                                                    \
    PM_IN(List&, x); PM_IN(NumericMatrix&, Q); PM_IN(NumericVector&, pid); PM_IN(NumericMatrix&, B);                     \
    PM_IN(double, Omega); PM_IN(IntegerMatrix&, nen_m); PM_IN(IntegerMatrix&, nodelist_m); PM_IN(IntegerVector, roots);  \
    PM_IN(int, N); PM_IN(NumericVector&, prior);                                                                         \
    return Rcpp::wrap(fn(x, Q, pid, B, Omega, nen_m, nodelist_m, roots, N, prior));                                      \
    END_RCPP                                                                                                             \
  }

PM_FIXED(SPARSEmaketreelistMCMC)
PM_FIXED(maketreelistMCMC)
PM_FIXED(maketreelistMCMC_bigtree)
PM_PRIOR(maketreelistMCMCbf)
PM_PRIOR(maketreelistMCMCks)
PM_MULTI(maketreelistMCMCmt)
PM_MULTI(maketreelistMCMCksmt)
PM_PRIOR(maketreelistMCMC2sDICt)
PM_PRIOR(maketreelistMCMCksDICt)

NumericMatrix maketreelistEXP(List& x, NumericMatrix& Q, NumericVector& pid, IntegerVector& nen, IntegerVector& nodelist, int root, int N,
                              NumericMatrix& lefts, NumericMatrix& rights, NumericMatrix& d);
RcppExport SEXP phylomap_maketreelistEXP(SEXP xSEXP, SEXP QSEXP, SEXP pidSEXP, SEXP nenSEXP, SEXP nodelistSEXP, SEXP rootSEXP,
                                         SEXP NSEXP, SEXP leftsSEXP, SEXP rightsSEXP, SEXP dSEXP) {
  BEGIN_RCPP
  Rcpp::RNGScope rcpp_rngScope_gen;
  PM_IN(List&, x); PM_IN(NumericMatrix&, Q); PM_IN(NumericVector&, pid); PM_IN(IntegerVector&, nen);
  PM_IN(IntegerVector&, nodelist); PM_IN(int, root); PM_IN(int, N); PM_IN(NumericMatrix&, lefts);
  PM_IN(NumericMatrix&, rights); PM_IN(NumericMatrix&, d);
  return Rcpp::wrap(maketreelistEXP(x, Q, pid, nen, nodelist, root, N, lefts, rights, d));
  END_RCPP
}

"""The oracle pinned against THE REFERENCE ITSELF (CPU).

oracle/_ref/libphylomap_ref.so = the unmodified /root/reference/src/phylomap.cpp + RcppExports.cpp compiled against the
stand-in Rcpp / RcppArmadillo / Armadillo headers in oracle/standin/ (R is absent; oracle/Makefile target `ref`).
tests/golden/reference/*.json hold its outputs for all ten `.Call` entry points (made by
tests/golden/make_reference_golden.py).  The oracle restatement in R-sequential mode must reproduce them bit for bit;
where the library itself is present (this container; the GPU box gets the prebuilt file) it is re-run as well.
"""
import ctypes
import glob
import json
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import make_reference_golden as mrg  # noqa: E402

FIXTURES = sorted(glob.glob(os.path.join(HERE, "golden", "reference", "*.json")))
SYMBOLS = ["phylomap_SPARSEmaketreelistMCMC", "phylomap_maketreelistMCMC", "phylomap_maketreelistMCMC_bigtree",
           "phylomap_maketreelistEXP", "phylomap_maketreelistMCMCbf", "phylomap_maketreelistMCMCks",
           "phylomap_maketreelistMCMCmt", "phylomap_maketreelistMCMCksmt", "phylomap_maketreelistMCMC2sDICt",
           "phylomap_maketreelistMCMCksDICt"]  # src/RcppExports.cpp:11,34,57,80,106,132,159,185,211,237


def _load(path):
    with open(path) as f:
        d = json.load(f)
    return d["case"], np.array(d["rows"]), np.array(d["Q_after"]), np.array(d["B_after"])


def _loglik_col(case):
    return {"DIC2S", "DICKS"} & {case["variant"]}


def _same_rows(got, want, case):
    """Bit-exact, except the DIC log-likelihood column: arma::expmat is a Pade scheme the stand-in and the oracle each
    restate their own way (agreement to rounding, 1e-12 relative asked)."""
    if _loglik_col(case):
        assert np.array_equal(got[:, :-1], want[:, :-1])
        assert np.allclose(got[:, -1], want[:, -1], rtol=1e-12, atol=0)
    else:
        assert np.array_equal(got, want)


def test_fixture_set_covers_every_exported_function():
    assert len(FIXTURES) >= 16
    seen = {_load(p)[0]["variant"] for p in FIXTURES}
    assert seen == {"PLAIN", "SPARSE", "BIGTREE", "EXP", "BF", "KS", "MT", "KSMT", "DIC2S", "DICKS"}


@pytest.mark.parametrize("path", FIXTURES, ids=[os.path.basename(p)[:-5] for p in FIXTURES])
def test_oracle_in_r_order_reproduces_the_reference(oracle, path):
    case, rows, Q_after, B_after = _load(path)
    eig = [np.array(m) for m in case["eig"]] if "eig" in case else None
    o = oracle.OracleRun(getattr(oracle, case["variant"]), [t.oracle_dict() for t in mrg.trees_of(case)], np.array(case["Q"]),
                         np.array(case["pid"]), case["Omega"], case["N"], prior=case.get("prior"),
                         rng_mode=oracle.SEQUENTIAL, seed=case["seed"], eig=eig)
    got = o.run()
    _same_rows(got, rows, case)
    assert np.array_equal(o.Q, Q_after) and np.array_equal(o.B, B_after)  # in-place rewrite of Q and B (phylomap.cpp:1284)


@pytest.mark.parametrize("path", FIXTURES, ids=[os.path.basename(p)[:-5] for p in FIXTURES])
def test_reference_library_reproduces_its_fixtures(oracle, path):
    if oracle.ref_lib() is None:
        pytest.skip("oracle/_ref not built here (no /root/reference, no prebuilt library)")
    case, rows, Q_after, B_after = _load(path)
    got, Q, B = mrg.run_reference(oracle, case)
    assert np.array_equal(got, rows) and np.array_equal(Q, Q_after) and np.array_equal(B, B_after)


def test_reference_library_exports_the_call_symbols(oracle):
    if oracle.ref_lib() is None:
        pytest.skip("oracle/_ref not built here")
    L = ctypes.CDLL(oracle.ref_path())
    for s in SYMBOLS:
        assert hasattr(L, s), s


def test_reference_errors_surface(oracle):
    """A zero root prior makes RcppArmadillo::sample throw inside the reference (phylomap.cpp:627); BEGIN_RCPP / END_RCPP
    turn it into an R error -- here an OracleError carrying the same text, and the oracle restatement raises it too."""
    if oracle.ref_lib() is None:
        pytest.skip("oracle/_ref not built here")
    case = _load(os.path.join(HERE, "golden", "reference", "plain_2state.json"))[0]
    trees = [t.oracle_dict() for t in mrg.trees_of(case)]
    with pytest.raises(oracle.OracleError, match="Not enough positive probabilities"):
        oracle.ref_run(oracle.PLAIN, trees, np.array(case["Q"]), np.zeros(2), case["Omega"], 2, seed=1)
    with pytest.raises(oracle.OracleError, match="Not enough positive probabilities"):
        oracle.OracleRun(oracle.PLAIN, trees, np.array(case["Q"]), np.zeros(2), case["Omega"], 2,
                         rng_mode=oracle.SEQUENTIAL, seed=1).run()


def test_oracle_errors_like_the_reference(oracle):
    """The oracle half of test_reference_errors_surface, which needs no reference library: a zero root prior raises the
    text RcppArmadillo::sample throws inside the reference (phylomap.cpp:627)."""
    case = _load(os.path.join(HERE, "golden", "reference", "plain_2state.json"))[0]
    trees = [t.oracle_dict() for t in mrg.trees_of(case)]
    with pytest.raises(oracle.OracleError, match="Not enough positive probabilities"):
        oracle.OracleRun(oracle.PLAIN, trees, np.array(case["Q"]), np.zeros(2), case["Omega"], 2,
                         rng_mode=oracle.SEQUENTIAL, seed=1).run()


def test_reference_sees_the_pinned_r_generator(oracle):
    """The stand-in's unif_rand / exp_rand / norm_rand are R's, checked against published R outputs.  Without the
    reference's sources the stand-in is probed through the shim's library, which compiles the same headers."""
    L = oracle.ref_lib() or oracle.shim_lib()
    assert np.allclose(oracle.ref_rng_probe(1, "unif", 3, lib_=L), [0.2655087, 0.3721239, 0.5728534], atol=5e-8)
    assert np.allclose(oracle.ref_rng_probe(1, "exp", 3, lib_=L), [0.7551818, 1.1816428, 0.1457067], atol=5e-8)
    assert np.allclose(oracle.ref_rng_probe(1, "norm", 3, lib_=L), [-0.6264538, 0.1836433, -0.8356286], atol=5e-8)


def test_twenty_state_ties_are_the_one_known_divergence(oracle):
    """RcppArmadillo::sample sorts the weights with std::sort.  Up to 16 states that is an insertion sort (ties keep
    index order), which is what the oracle and the CUDA library implement; above 16 libstdc++ switches to introsort and
    EXACTLY equal weights may come out in another order.  Only a model with exact ties (Jukes-Cantor-like, 20 states:
    the tutorial's example) can tell the difference; an asymmetric 20-state model is bit-identical (fixture
    plain_20state).  This test documents the divergence instead of hiding it."""
    if oracle.ref_lib() is None:
        pytest.skip("oracle/_ref not built here")
    import cases
    Q = cases.jc(20, 0.02)
    z = cases.tree_n(Q, T=8, S=1, seed=36, mean_branch=2.0, segments=4)
    pid = np.full(20, 0.05)
    a = oracle.OracleRun(oracle.PLAIN, [z.oracle_dict()], Q, pid, 1.0, 5, rng_mode=oracle.SEQUENTIAL, seed=5).run()
    r, _, _ = oracle.ref_run(oracle.PLAIN, [z.oracle_dict()], Q, pid, 1.0, 5, seed=5)
    # same total dwell time (= tree length) either way; the histories differ once a tie is broken differently
    assert np.allclose(a[:, :20].sum(1), r[:, :20].sum(1), rtol=1e-12)

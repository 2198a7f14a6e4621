"""The drop-in shim (shim/phylomap_b200_shim.cpp) driven through the package's `.Call` symbols.

oracle/_ref/libphylomap_shim.so = the package's `.Call` glue (oracle/shim_glue.cpp, written as Rcpp generates
src/RcppExports.cpp) + the shim (which replaces src/phylomap.cpp) compiled against the stand-in Rcpp headers and linked
to libphylomap_b200.so.  The driver builds the R objects an R session would pass (tree list with maps / mapnames / edge /
states, Q, pid, B, nen, nodelist, root, N, prior; lists of trees and nen / nodelist MATRICES for mt / ksmt,
R/sumstatMCMCmt.R:27-33) and calls phylomap_<fn>.  The result must equal the library called directly with the seed the
shim derives from R's stream: that pins the flattening (CSR maps, column-major edge, the ntips x nsites states matrix, one
nen / nodelist row per tree) and the in-place rewrite of Q and B.  The glue is bound to the shim's signatures by the link;
tests/golden/shim/call_signatures.json binds those to the package's.
"""
import ctypes
import json
import os
import re

import numpy as np
import pytest

import cases
import phylomap_b200 as pb
from phylomap_b200 import capi

SYMBOLS = ["phylomap_SPARSEmaketreelistMCMC", "phylomap_maketreelistMCMC", "phylomap_maketreelistMCMC_bigtree",
           "phylomap_maketreelistEXP", "phylomap_maketreelistMCMCbf", "phylomap_maketreelistMCMCks",
           "phylomap_maketreelistMCMCmt", "phylomap_maketreelistMCMCksmt", "phylomap_maketreelistMCMC2sDICt",
           "phylomap_maketreelistMCMCksDICt"]


def test_shim_signatures_are_the_packages():
    """The shim defines the ten functions with the parameter types the package's generated glue passes."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "tests", "golden", "shim", "call_signatures.json")) as f:
        want = {k: v for k, v in json.load(f).items() if not k.startswith("_")}
    with open(os.path.join(root, "shim", "phylomap_b200_shim.cpp")) as f:
        src = f.read()
    assert len(want) == 10
    for fn, types in want.items():
        defs = re.findall(r"NumericMatrix %s\(([^)]*)\)\s*\{" % fn, src)
        assert len(defs) == 1, fn
        assert [" ".join(p.split()[:-1]) for p in defs[0].split(",")] == types, fn


def test_shim_exports_the_ten_call_symbols(oracle):
    oracle.shim_lib()
    L = ctypes.CDLL(oracle.shim_path())
    for s in SYMBOLS:
        assert hasattr(L, s), s


def test_shim_tree_order_is_pm_tree_order(oracle):
    """phylomap_tree_order (the O(E) replacement of R/sumstatMCMC.R:1-18) through the shim: host code, no device."""
    L = oracle.shim_lib()
    z = cases.tree2(T=40, S=1, seed=3)
    E = z.E
    edge = np.asfortranarray(z.edge, dtype=np.int32)
    nen, nodelist, root = np.zeros(E, np.int32), np.zeros(z.T - 2, np.int32), ctypes.c_int32(0)
    err = ctypes.create_string_buffer(256)
    rc = L.shim_tree_order(edge.ctypes.data, E, z.T, nen.ctypes.data, nodelist.ctypes.data, ctypes.byref(root), err, 256)
    assert rc == 0, err.value
    a, b, c = z.order()
    assert np.array_equal(nen, a) and np.array_equal(nodelist, b) and root.value == c


@pytest.fixture()
def det_env(monkeypatch):
    monkeypatch.setenv("PHYLOMAP_B200_MODE", "deterministic")
    monkeypatch.setenv("PHYLOMAP_B200_PRECISION", "f64")
    monkeypatch.setenv("PHYLOMAP_B200_DEVICE", "0")


def _trees_multi(base, k, seed):
    rng = np.random.default_rng(seed)
    return [base] + [pb.PhyloTree(base.edge, base.edge_length * rng.uniform(0.7, 1.3, size=base.E)).with_states(base.states)
                     for _ in range(k - 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["PLAIN", "SPARSE", "BIGTREE", "BF", "KS", "MT", "KSMT", "DIC2S", "DICKS"])
@pytest.mark.parametrize("S", [1, 5])
def test_shim_call_equals_direct_call(oracle, det_env, name, S):
    Q4, p4 = cases.q4(), np.full(4, 0.25)
    hidden = name in ("KS", "KSMT", "DICKS")
    two = name in ("BF", "MT", "DIC2S")
    if hidden:
        base, Q, pid, Om = cases.tree_hidden(Q4, T=14, S=S, seed=11, mean_branch=0.5), Q4, p4, 4.0
        prior = cases.PRIOR_KSMT if name == "KSMT" else cases.PRIOR_KS
    elif two:
        base, Q, pid, Om, prior = cases.tree2(T=16, S=S, seed=11), cases.Q2, cases.PID2, 0.5, cases.PRIOR_BF
    else:
        base, Q, pid, Om, prior = cases.tree_n(Q4, T=14, S=S, seed=7, mean_branch=0.6, segments=3), Q4, p4, 2.4, None
    trees = _trees_multi(base, 3, 5) if name in ("MT", "KSMT") else [base]
    N, seed = 7, 42
    rows, Qs, Bs = oracle.shim_run(getattr(oracle, name), [t.oracle_dict() for t in trees], Q, pid, Om, N, prior=prior, seed=seed)
    Qd = np.asfortranarray(np.array(Q, dtype=np.float64))
    ch = pb.Chain(getattr(capi, "PM_V_" + name), trees if len(trees) > 1 else trees[0], Qd, pid, Om, N, prior=prior,
                  seed=oracle.shim_seed(seed), mode="deterministic", precision="f64")
    want = ch.run()
    assert np.array_equal(rows, want)
    assert np.array_equal(Qs, Qd) and np.array_equal(Bs, ch.B)   # Q and B rewritten in place through the shim too
    if name == "PLAIN":
        assert rows.shape == (N, 16) and np.allclose(rows[:, :4].sum(1), S * base.edge_length.sum(), rtol=1e-9)


@pytest.mark.gpu
def test_shim_direct_sampler_and_errors(oracle, monkeypatch):
    monkeypatch.setenv("PHYLOMAP_B200_PRECISION", "f32")
    monkeypatch.delenv("PHYLOMAP_B200_MODE", raising=False)
    Q, pid = cases.jc(4, 0.1), np.full(4, 0.25)
    z = cases.tree_n(Q, T=20, S=3, seed=3, mean_branch=2.0)
    w, V = np.linalg.eig(Q)
    eig = (V.real, np.linalg.inv(V).real, np.diag(w.real))
    rows, _, _ = oracle.shim_run(oracle.EXP, [z.oracle_dict()], Q, pid, 0.3, 6, seed=9, eig=eig)
    want = pb.sumstatEXP(z, Q, pid, 6, seed=oracle.shim_seed(9), precision="f32")
    assert np.array_equal(rows, want)
    # an error of the library becomes Rcpp::stop -> an R error carrying the same text (a zero root prior, :627)
    with pytest.raises(oracle.OracleError, match="Not enough positive probabilities"):
        oracle.shim_run(oracle.PLAIN, [z.oracle_dict()], Q, np.zeros(4), 0.3, 2, seed=9)

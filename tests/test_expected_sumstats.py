"""Exact posterior expectations (pm_expected_sumstats): the float64 reference of tests/exact_ref.py against brute-force
enumeration and numerical quadrature, and the argument checks of the entry (no device needed)."""
import ctypes as C

import numpy as np
import pytest
from scipy.integrate import quad
from scipy.linalg import expm

import exact_ref
import phylomap_b200 as pb
from phylomap_b200 import capi, synth


@pytest.mark.parametrize("T,n,parity", [(3, 2, False), (4, 3, False), (5, 4, False), (6, 2, False), (6, 3, False),
                                        (4, 4, True), (5, 4, True)])
def test_reference_equals_brute_force(T, n, parity):
    rng = np.random.default_rng(100 * T + n + parity)
    tree = synth.yule_tree(T, seed=T + 7, mean_branch=0.7)
    Q = exact_ref.random_q(n, rng)
    pid = rng.dirichlet(np.ones(n))
    for _ in range(3):
        states = rng.integers(1, (2 if parity else n) + 1, size=T)
        got = exact_ref.exact(tree.edge, tree.edge_length, Q, pid, states, parity)
        want = exact_ref.brute_force(tree.edge, tree.edge_length, Q, pid, states, parity)
        for g, w in zip(got, want):
            np.testing.assert_allclose(g, w, rtol=1e-12, atol=1e-12)


def test_van_loan_blocks_equal_quadrature():
    rng = np.random.default_rng(5)
    n, t = 3, 0.8
    Q = exact_ref.random_q(n, rng, scale=1.5)
    M = exact_ref.branch_integrals(Q, t)
    P = lambda s: expm(Q * s)  # noqa: E731
    for k, (i, j) in enumerate(exact_ref.stat_pairs(n)):
        w = 1.0 if k < n else Q[i, j]
        for a in range(n):
            for b in range(n):
                v, _ = quad(lambda s: P(s)[a, i] * P(t - s)[j, b], 0.0, t, epsabs=1e-14, epsrel=1e-13)
                assert abs(M[k][a, b] - w * v) < 1e-10


@pytest.mark.parametrize("n", [2, 4, 8])
def test_dwell_integrals_sum_to_t_times_p(n):
    rng = np.random.default_rng(n)
    Q = exact_ref.random_q(n, rng)
    for t in (0.01, 0.9, 7.5):
        M = exact_ref.branch_integrals(Q, t)
        np.testing.assert_allclose(M[:n].sum(0), t * expm(Q * t), rtol=1e-12, atol=1e-14)


def _call(tree, n=2, Q=None, pid=None, parity=0, sites=None, nsel=None, null_tree=False):
    L = capi.lib()
    Q = np.asfortranarray(-np.eye(n) + (1 - np.eye(n)) / (n - 1)) if Q is None else Q
    pid = np.full(n, 1.0 / n) if pid is None else pid
    t, keep = tree.flat()
    sel = None if sites is None else np.ascontiguousarray(sites, dtype=np.int64)
    err = C.create_string_buffer(512)
    rc = L.pm_expected_sumstats(None if null_tree else C.byref(t), n, capi.ptr(Q), capi.ptr(pid), parity, capi.ptr(sel),
                                (0 if sel is None else len(sel)) if nsel is None else nsel, None, None, None, None, None, err, 512)
    return rc, err.value.decode()


def test_malformed_input_is_rejected_before_any_device_work():
    tree = synth.yule_tree(6, seed=2).with_states(np.array([[1, 2, 1, 2, 1, 1], [2, 2, 1, 1, 1, 2]], dtype=np.int32))
    Q2 = np.asfortranarray([[-1.0, 1.0], [1.0, -1.0]])
    L = capi.lib()
    err = C.create_string_buffer(512)
    assert L.pm_expected_sumstats(C.byref(tree.flat()[0]), 2, None, capi.ptr(np.full(2, 0.5)), 0, None, 0, None, None, None, None,
                                  None, err, 512) == capi.PM_ERR_ARG
    rc, msg = _call(tree, null_tree=True)
    assert rc == capi.PM_ERR_ARG and "null" in msg
    assert L.pm_expected_sumstats(C.byref(tree.flat()[0]), 2, capi.ptr(Q2), None, 0, None, 0, None, None, None, None, None,
                                  err, 512) == capi.PM_ERR_ARG
    for n in (1, 9):
        rc, msg = _call(tree, n=n, Q=np.zeros((max(n, 1), max(n, 1)), order="F"))
        assert rc == capi.PM_ERR_ARG and "number of states" in msg
    rc, msg = _call(tree, n=3, parity=1)
    assert rc == capi.PM_ERR_ARG and "even" in msg
    for bad in ([2], [-1], [0, 1, 5]):
        rc, msg = _call(tree, sites=bad)
        assert rc == capi.PM_ERR_ARG and "out of range" in msg
    rc, msg = _call(tree, sites=None, nsel=3)
    assert rc == capi.PM_ERR_ARG


def test_expected_sumstats_result_layout():
    """mapped_edge / transitions of the result object against a hand-made per-branch array (no device)."""
    n, E = 3, 4
    bs = np.arange(2 * E * n * n, dtype=np.float64).reshape(2, E, n * n)
    r = pb.ExpectedSumstats(n, None, None, np.array([0, 1]), bs, None)
    np.testing.assert_array_equal(r.mapped_edge(), bs[:, :, :n])
    tr = r.transitions()
    tot = bs.sum(1)
    for k, (i, j) in enumerate(exact_ref.stat_pairs(n)):
        if k >= n:
            np.testing.assert_array_equal(tr[:, i, j], tot[:, k])
    assert np.all(tr[:, np.arange(n), np.arange(n)] == 0)

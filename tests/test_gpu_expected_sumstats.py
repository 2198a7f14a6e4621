"""Exact posterior expectations on the device (pb.expected_sumstats / pm_expected_sumstats): against the float64
reference of tests/exact_ref.py, their internal identities, bit-exact tiling, and the samplers' convergence to them."""
import ctypes as C

import numpy as np
import pytest

import cases
import exact_ref
import phylomap_b200 as pb
from phylomap_b200 import capi, synth

pytestmark = pytest.mark.gpu

# FP32: the partials, P(t_e) and M_e are stored in FP32 (unit roundoff u = 6e-8).  Each node's partial picks up O(n)
# roundings per level and a contraction n^2 more; over the <= 60 levels of these trees that is at most a few thousand u,
# i.e. below 2e-4 relative to the size of the output.
F32_TOL = 2e-4


def _tree(Q, T, S, seed, parity=False):
    if parity:
        return cases.tree_hidden(Q, T=T, S=S, seed=seed)
    return cases.tree_n(Q, T=T, S=S, seed=seed)


def _states(z):
    st = np.asarray(z.states)
    return st[None, :] if st.ndim == 1 else st


def _check(got, want, tol):
    got, want = np.asarray(got), np.asarray(want)
    np.testing.assert_allclose(got, want, rtol=tol, atol=tol * max(1.0, float(np.abs(want).max())))


def _reference(z, Q, pid, parity, sites, blen=None):
    blen = z.edge_length if blen is None else blen
    model = exact_ref.branch_model(blen, Q)
    st = _states(z)
    out = [exact_ref.exact(z.edge, blen, Q, pid, st[s], parity, model) for s in range(len(st))]
    stats = np.array([o[0] for o in out])
    ll = np.array([o[3] for o in out])
    return stats, ll, np.array([out[s][1] for s in sites]), np.array([out[s][2] for s in sites])


CASES = [  # (n, tips, sites, parity)
    (2, 4, 1, False), (3, 20, 37, False), (4, 100, 33, False), (6, 30, 5, False), (8, 12, 3, False),
    (4, 50, 40, True), (4, 300, 2, False), (6, 16, 7, True)]


@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("n,T,S,parity", CASES)
def test_against_reference(n, T, S, parity, precision):
    rng = np.random.default_rng(10 * n + T)
    if parity:
        Q = cases.q4() if n == 4 else cases.q6()
    else:
        Q = exact_ref.random_q(n, rng)
    pid = rng.dirichlet(np.ones(n))
    z = _tree(Q, T, S, seed=T, parity=parity)
    sites = [0, S - 1, S // 2, 0]
    r = pb.expected_sumstats(z, Q, pid, parity_tips=parity, sites=sites, precision=precision)
    stats, ll, bs, nm = _reference(z, Q, pid, parity, sites)
    tol = 1e-10 if precision == "f64" else F32_TOL
    _check(r.stats, stats, tol)
    _check(r.loglik, ll, tol)
    _check(r.branch_stats, bs, tol)
    _check(r.node_marginals, nm, tol)
    assert r.stats.shape == (S, n * n) and r.branch_stats.shape == (4, z.E, n * n) and r.node_marginals.shape == (4, 2 * T - 1, n)


def test_branch_lengths_from_edge_length_or_maps():
    """edge_length when given, else the sums of the maps (pm_loglik's rule): maps whose sums differ from edge_length."""
    Q = cases.jc(3, 0.4)
    pid = np.full(3, 1 / 3)
    z = cases.tree_n(Q, T=15, S=6, seed=3)
    maps = [np.array([0.6 * t, 0.9 * t]) for t in z.edge_length]
    z = pb.PhyloTree(z.edge, z.edge_length, z.states, maps, [np.array([1, 1], dtype=np.int32)] * z.E)
    r = pb.expected_sumstats(z, Q, pid, sites=[1])
    stats, ll, bs, _ = _reference(z, Q, pid, False, [1])
    _check(r.stats, stats, 1e-10)
    # the same tree with edge_length NULL: the maps sums (1.5 t) are the branch lengths
    L = capi.lib()
    t, keep = z.flat()
    t.edge_length = None
    S, NK = 6, 9
    out = np.zeros((S, NK), order="F")
    ll_out = np.zeros(S)
    err = C.create_string_buffer(512)
    opt = capi.default_options()
    Qf = np.asfortranarray(Q)
    capi.check(L.pm_expected_sumstats(C.byref(t), 3, capi.ptr(Qf), capi.ptr(pid), 0, None, 0, C.byref(opt), capi.ptr(out),
                                      capi.ptr(ll_out), None, None, err, 512), err)
    stats2, ll2, _, _ = _reference(z, Q, pid, False, [], blen=1.5 * z.edge_length)
    _check(out, stats2, 1e-10)
    _check(ll_out, ll2, 1e-10)


@pytest.mark.parametrize("parity", [False, True])
def test_consistency(parity):
    Q = cases.q4() if parity else exact_ref.random_q(4, np.random.default_rng(7))
    pid = np.full(4, 0.25)
    S = 70
    z = _tree(Q, 60, S, seed=9, parity=parity)
    sel = [3, 69, 3]
    r = pb.expected_sumstats(z, Q, pid, parity_tips=parity, sites=sel)
    assert abs(r.loglik.sum() - pb.loglik(z, Q, pid, parity_tips=parity)) <= 1e-12 * abs(r.loglik.sum())
    np.testing.assert_allclose(r.stats[:, :4].sum(1), z.edge_length.sum(), rtol=1e-12)
    np.testing.assert_allclose(r.node_marginals.sum(2), 1.0, rtol=1e-12)
    np.testing.assert_allclose(r.branch_stats.sum(1), r.stats[sel], rtol=1e-12, atol=1e-12 * np.abs(r.stats).max())
    np.testing.assert_array_equal(r.branch_stats[0], r.branch_stats[2])
    f32 = pb.expected_sumstats(z, Q, pid, parity_tips=parity, precision="f32")
    np.testing.assert_allclose(f32.stats[:, :4].sum(1), z.edge_length.sum(), rtol=1e-5)


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_tiles_and_repeats_give_the_same_bits(precision, monkeypatch):
    Q = exact_ref.random_q(4, np.random.default_rng(3))
    pid = np.full(4, 0.25)
    z = cases.tree_n(Q, T=80, S=301, seed=5)
    sel = list(range(0, 301, 7))
    a = pb.expected_sumstats(z, Q, pid, sites=sel, precision=precision)
    b = pb.expected_sumstats(z, Q, pid, sites=sel, precision=precision)
    monkeypatch.setenv("PHYLOMAP_B200_SITE_TILE", "37")
    c = pb.expected_sumstats(z, Q, pid, sites=sel, precision=precision)
    for r in (b, c):
        for f in ("stats", "loglik", "branch_stats", "node_marginals"):
            assert np.array_equal(getattr(a, f), getattr(r, f)), f


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_zero_likelihood_is_reported(precision):
    Q = np.zeros((2, 2))  # no changes possible: tips in different states have probability 0
    z = cases.tree2(T=10, S=3)
    st = np.array([[1] * 10, [1, 2] * 5, [2] * 10], dtype=np.int32)
    z = z.with_states(st)
    with pytest.raises(capi.PhylomapError) as ei:
        pb.expected_sumstats(z, Q, cases.PID2, sites=[0], precision=precision)
    assert ei.value.code == capi.PM_ERR_SAMPLE and "zero likelihood" in ei.value.msg


def _batch_se(x, nb):
    """Mean and batch-means standard error of a [K, ...] series."""
    K = (len(x) // nb) * nb
    b = x[:K].reshape(nb, K // nb, *x.shape[1:]).mean(1)
    return x[:K].mean(0), b.std(0, ddof=1) / np.sqrt(nb)


# The sampler rows sum over sites: with 4 000 sites x 2 000 sweeps the batch-means error of a column mean is ~0.1 % of
# it, well under the 1 % bars of the sampler-against-sampler tests.
@pytest.mark.parametrize("sampler,precision", [("sumstatMCMC", "f64"), ("sumstatMCMC", "f32"), ("sumstatMCMC_bigtree", "f64"),
                                               ("sumstatMCMC_bigtree", "f32"), ("sumstatEXP", "f64")])
def test_samplers_converge_to_the_exact_expectations(sampler, precision):
    Q = np.array([[-0.5, 0.3, 0.2], [0.4, -0.6, 0.2], [0.1, 0.5, -0.6]])
    pid = np.array([0.5, 0.3, 0.2])
    S, N, burn = 4000, 2000, 100
    z = cases.tree_n(Q, T=24, S=S, seed=11, segments=2)
    exact = pb.expected_sumstats(z, Q, pid).stats.sum(0)
    if sampler == "sumstatEXP":
        rows = pb.sumstatEXP(z, Q, pid, N, seed=3, precision=precision)
    else:
        rows = getattr(pb, sampler)(z, Q.copy(), pid, 1.5, N, seed=3, precision=precision)
    mean, se = _batch_se(rows[burn:], 40)
    z_scores = (mean - exact) / se
    assert np.all(np.abs(z_scores) < 4), (sampler, precision, mean, exact, z_scores)
    assert np.all(se < 2e-3 * np.abs(exact))


def test_sampled_maps_and_node_states_converge_to_the_exact_values():
    """A chain's exported maps (mapped_edge / transitions) and node states, averaged over sweeps, against the exact
    per-branch expectations and node marginals of three sites.  Per-element z-scores over ~300 comparisons: the bound
    is the Bonferroni level of a 1e-3 family-wise false alarm (4.9 standard errors), not a widened tolerance."""
    Q = np.array([[-0.8, 0.8], [0.5, -0.5]])
    pid = np.array([0.4, 0.6])
    z = cases.tree_n(Q, T=12, S=64, seed=2, mean_branch=0.8, segments=2)
    sel = [0, 17, 63]
    ex = pb.expected_sumstats(z, Q, pid, sites=sel)
    ch = pb.Chain(capi.PM_V_PLAIN, z, Q.copy(), pid, 2.0, 4200, seed=8)
    ch.run(200)
    me, tr, ns = [], [], []
    for _ in range(4000):
        ch.run(1)
        m = ch.maps(sel)
        me.append(m.mapped_edge())
        tr.append(m.transitions())
        nst = ch.node_states()[sel]
        ns.append(np.eye(2)[nst])
    bound = 4.9
    for got, want in ((np.array(me), ex.mapped_edge()), (np.array(tr), ex.transitions()), (np.array(ns), ex.node_marginals)):
        mean, se = _batch_se(got, 100)
        d = mean - want
        live = se > 0
        assert np.all(np.abs(d[~live]) < 1e-9)
        assert np.all(np.abs(d[live] / se[live]) < bound), np.abs(d[live] / se[live]).max()


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_benchmark_size(precision):
    """One call at the benchmark's per-GPU size: 10 000 tips x 125 000 sites, 4 states."""
    Q = synth.make2sQ(0.1, 0.1, 0.2, 0.2, 10.0)
    tree = synth.yule_tree(10000, seed=4, mean_branch=0.1 / float(np.max(-np.diag(Q))))
    st = synth.simulate_tip_states(tree, Q, np.full(4, 0.25), 125000, seed=101, device="cuda", batch_sites=32768)
    z = tree.with_states(st.to("cpu").to(dtype=__import__("torch").uint8).numpy(), segments=2)
    r = pb.expected_sumstats(z, Q, np.full(4, 0.25), sites=[0, 124999], precision=precision)
    tol = 1e-10 if precision == "f64" else 1e-4
    np.testing.assert_allclose(r.stats[:, :4].sum(1), tree.edge_length.sum(), rtol=tol)
    assert np.all(np.isfinite(r.stats)) and np.all(np.isfinite(r.loglik))

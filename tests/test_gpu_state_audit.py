"""Audit of the production chain state against exact FP64 recomputations in plain numpy.

The production kernels (FP32 / FP64, fused prune + node draw, pooled record slices, 16-bit jump positions, header records,
the one-block-per-site kernel, graph replay) are compared elsewhere with each other bit for bit and with the oracle only
in distribution.  Neither would notice a bug that all production kernel sets share.  Here the state a chain leaves behind
is read back (node states, piece counts, stored paths, partials) and the row it returned is rebuilt from it:

- dwell time per state = the FP64 sum of the stored run lengths by state;
- off-diagonal counts = the transitions between consecutive stored runs (the diagonal, virtual-jump counts of the
  rate samplers cannot be rebuilt from the stored state and are left out);
- every path joins its parent's and its child's node state, its runs differ from their neighbours and add up to the
  branch length, and there are no more runs than pieces;
- tips equal the data (or its parity for the hidden-rate samplers).

Partials are compared with an exact pruning with B^(m-1), log-likelihoods with a pruning with scipy's expm, and every
node draw must have positive probability under the piece counts the sweep pruned with.  The helpers are first checked
against the CPU oracle (no GPU needed).
"""
import time

import numpy as np
import pytest

import cases
import phylomap_b200 as pb
from phylomap_b200 import capi, synth

FULL_COUNTS = {capi.PM_V_BF, capi.PM_V_KS, capi.PM_V_MT, capi.PM_V_KSMT, capi.PM_V_DIC2S, capi.PM_V_DICKS}
PARITY = {capi.PM_V_KS, capi.PM_V_KSMT, capi.PM_V_DICKS}
MULTI = {capi.PM_V_MT, capi.PM_V_KSMT}
SPARSE_DROP = 1e-7          # matTospmat keeps the entries of B above this
FP32_GAPS = {}              # largest relative FP32 gap against the FP64 references, by quantity (printed at the end)


def _note_gap(what, gap):
    FP32_GAPS[what] = max(FP32_GAPS.get(what, 0.0), float(gap))


@pytest.fixture(scope="module", autouse=True)
def _report_fp32_gaps():
    t0 = time.perf_counter()
    yield
    for k, v in sorted(FP32_GAPS.items()):
        print("\nlargest FP32 gap, %s: %.3g" % (k, v))
    print("\nstate audit module: %.1f s" % (time.perf_counter() - t0))


def _data(tree):
    return np.atleast_2d(np.asarray(tree.states)).astype(np.int64)


# ---- FP64 reference helpers -------------------------------------------------------------------------------------
def rebuild_row(chain, tree, tree_index=0, full=False, parity=False, len_rtol=1e-12, cap=4096):
    """Dwell time per state (FP64 sums of the stored runs) and the n x n matrix of transitions between consecutive stored
    runs of every site and branch of `chain` (a pb.Chain or an oracle run); raises AssertionError if the stored state is
    not a valid history: paths that do not join their node states, equal neighbouring runs, lengths that do not add up to
    the branch, more runs than pieces, tips that are not the data."""
    n = chain.n
    ns = chain.node_states(tree_index)
    m = chain.piece_counts(tree_index)
    S, T, E = ns.shape[0], tree.T, tree.E
    data = _data(tree)
    assert data.shape == (S, T)
    if parity:
        assert np.array_equal(ns[:, :T] % 2, data - 1), "tip states do not match the parity of the data"
    else:
        assert np.array_equal(ns[:, :T], data - 1), "tip states differ from the data"
    assert ns.min() >= 0 and ns.max() < n
    par, chi = tree.edge[:, 0] - 1, tree.edge[:, 1] - 1
    lens, sts, trans, bad = [], [], [], []
    for s in range(S):
        for e in range(E):
            ln, st = chain.path(s, e, tree_index, cap=cap)
            k = len(st)
            L = tree.edge_length[e]
            if not (0 < k < cap and st[0] == ns[s, par[e]] and st[-1] == ns[s, chi[e]] and np.all(st[1:] != st[:-1])
                    and k <= m[s, e] and np.all(ln >= 0) and abs(ln.sum() - L) <= len_rtol * L):
                bad.append("site %d branch %d: m %d, runs %s, lengths %s (branch %.17g), node states %d -> %d"
                           % (s, e, m[s, e], st[:8], ln[:8], L, ns[s, par[e]], ns[s, chi[e]]))
                continue
            lens.append(ln)
            sts.append(st)
            trans.append(st[:-1] * n + st[1:])
    assert not bad, "%d invalid stored paths, e.g.\n  %s" % (len(bad), "\n  ".join(bad[:5]))
    R = np.bincount(np.concatenate(sts), weights=np.concatenate(lens), minlength=n)
    N = np.bincount(np.concatenate(trans), minlength=n * n).reshape(n, n)
    return R, N


def row_counts(row, n, full):
    """The off-diagonal transition counts of a row, as an n x n matrix with a zero diagonal."""
    off = ~np.eye(n, dtype=bool)
    C = np.zeros((n, n))
    C[off] = row[n:n + n * n].reshape(n, n)[off] if full else row[n:n + n * (n - 1)]
    return C


def audit_row(row, R, N, n, full, dwell_rtol):
    """Counts must match exactly, dwell times to dwell_rtol; returns the largest relative dwell gap."""
    off = ~np.eye(n, dtype=bool)
    got = row_counts(row, n, full)
    assert np.array_equal(got[off], N[off]), "transition counts differ:\nrow\n%s\nrebuilt\n%s" % (got, N * off)
    gap = np.max(np.abs(row[:n] - R) / np.maximum(R, 1e-300))
    assert gap <= dwell_rtol, "dwell times %s, rebuilt %s (relative gap %.3g)" % (row[:n], R, gap)
    return gap


def _power_table(B, ks, support):
    out = {}
    if support:
        P0 = B > 0
        for k in ks:
            R, P, kk = np.eye(len(B), dtype=bool), P0, int(k)
            while kk:
                if kk & 1:
                    R = (R.astype(np.int64) @ P.astype(np.int64)) > 0
                P = (P.astype(np.int64) @ P.astype(np.int64)) > 0
                kk >>= 1
            out[k] = R.astype(np.float64)
        return out
    return {k: np.linalg.matrix_power(B, int(k)) for k in ks}


def _tip_partials(data_row, n, parity):
    T = len(data_row)
    PL = np.zeros((T, n))
    if parity:   # observed 1 -> the even 0-based hidden states, 2 -> the odd ones
        for i in range(T):
            PL[i, (0 if data_row[i] % 2 == 1 else 1)::2] = 1
    else:
        PL[np.arange(T), data_row - 1] = 1
    return PL


def exact_partials(tree, site, m, B, parity=False, sparse=False, normalize=True, support=False):
    """FP64 pruning of one site with B^(m_e - 1) on every branch (m: [S, E] piece counts), every node normalised to sum 1
    as the production arithmetic does (the oracle normalises only BIGTREE and the rate samplers).  SPARSE prunes with the
    entries of B <= 1e-7 dropped.  support=True: the exact 0/1 support instead (boolean matrix powers, no underflow).
    Returns [2T - 1, n]."""
    B = np.asarray(B, dtype=np.float64)
    n, T = B.shape[0], tree.T
    if sparse:
        B = np.where(B > SPARSE_DROP, B, 0.0)
    nen = tree.order()[0]
    chi, par = tree.edge[:, 1] - 1, tree.edge[:, 0] - 1
    ms = np.asarray(m)[site]
    pows = _power_table(B, np.unique(ms - 1), support)
    PL = np.zeros((2 * T - 1, n))
    PL[:T] = _tip_partials(_data(tree)[site], n, parity)
    for i in range(T - 1):
        ea, eb = nen[2 * i] - 1, nen[2 * i + 1] - 1
        v = (pows[ms[eb] - 1] @ PL[chi[eb]]) * (pows[ms[ea] - 1] @ PL[chi[ea]])
        if support:
            v = (v > 0).astype(np.float64)
        elif normalize:
            v = v / v.sum()
        PL[par[ea]] = v
    return PL


def exact_loglik(tree, Q, pid, parity=False, max_doubles=1 << 23):
    """log p(y | Q) summed over the sites of `tree`: pruning with scipy's expm(Q t_e), every node rescaled (the algorithm
    of test_gpu_parity._loglik_scipy), vectorised over blocks of sites so that large trees fit in memory."""
    from scipy.linalg import expm
    Q = np.asarray(Q, dtype=np.float64)
    n, T = Q.shape[0], tree.T
    nen, _, root = tree.order()
    chi, par = tree.edge[:, 1] - 1, tree.edge[:, 0] - 1
    PT = np.stack([expm(Q * t).T for t in tree.edge_length])      # row vectors times P^T
    data = _data(tree)
    blk = max(1, max_doubles // ((2 * T - 1) * n))
    tot = 0.0
    for s0 in range(0, data.shape[0], blk):
        d = data[s0:s0 + blk]
        b = d.shape[0]
        PL = np.zeros((2 * T - 1, b, n))
        if parity:
            odd = (d % 2 == 1).T[:, :, None]
            PL[:T, :, 0::2] = odd
            PL[:T, :, 1::2] = ~odd
        else:
            PL[np.arange(T)[:, None], np.arange(b)[None, :], (d - 1).T] = 1
        acc = np.zeros(b)
        for i in range(T - 1):
            ea, eb = nen[2 * i] - 1, nen[2 * i + 1] - 1
            v = (PL[chi[ea]] @ PT[ea]) * (PL[chi[eb]] @ PT[eb])
            sv = v.sum(1)
            acc += np.log(sv)
            PL[par[ea]] = v / sv[:, None]
        tot += float(np.sum(np.log(PL[root - 1] @ np.asarray(pid, dtype=np.float64)) + acc))
    return tot


def _root_state_col(variant, ncols):
    return ncols - 2 if variant in (capi.PM_V_DIC2S, capi.PM_V_DICKS) else ncols - 1


# ---- the helpers against the CPU oracle -------------------------------------------------------------------------
# oracle variant ids differ from the C ABI's after KSMT
def _oracle_variant(oracle, v):
    return {capi.PM_V_PLAIN: oracle.PLAIN, capi.PM_V_SPARSE: oracle.SPARSE, capi.PM_V_BIGTREE: oracle.BIGTREE,
            capi.PM_V_BF: oracle.BF, capi.PM_V_KS: oracle.KS, capi.PM_V_MT: oracle.MT, capi.PM_V_KSMT: oracle.KSMT,
            capi.PM_V_DIC2S: oracle.DIC2S, capi.PM_V_DICKS: oracle.DICKS}[v]


SPARSE_THRESHOLD_Q = np.array([[-0.1, 0.1, 0.0], [1e-9, -0.1 - 1e-9, 0.1], [0.05, 0.05, -0.1]])   # test_sparse_threshold_active


def _oracle_case(name):
    """(variant, trees, Q, pid, Omega, prior) of the small oracle cases."""
    q4, p4 = cases.q4(), np.full(4, 0.25)
    if name == "plain":
        return capi.PM_V_PLAIN, [cases.tree2(T=12, S=3, seed=3)], cases.Q2, cases.PID2, 0.2, None
    if name == "sparse":
        return (capi.PM_V_SPARSE, [cases.tree_n(cases.jc(3), T=16, S=5, seed=2, mean_branch=3.0, segments=4)],
                SPARSE_THRESHOLD_Q, np.full(3, 1 / 3), 0.4, None)
    if name == "bigtree":
        return (capi.PM_V_BIGTREE, [cases.tree_n(q4, T=10, S=2, seed=5, mean_branch=0.8, segments=3)], q4, p4, 2.4, None)
    if name in ("bf", "dic2s"):
        v = capi.PM_V_BF if name == "bf" else capi.PM_V_DIC2S
        return v, [cases.tree2(T=12, S=3, seed=9)], cases.Q2, cases.PID2, 0.5, cases.PRIOR_BF
    if name in ("ks", "dicks"):
        v = capi.PM_V_KS if name == "ks" else capi.PM_V_DICKS
        return v, [cases.tree_hidden(q4, T=10, S=2, seed=4, mean_branch=0.5)], q4, p4, 4.0, cases.PRIOR_KS
    if name == "mt":
        base = cases.tree2(T=10, S=3, seed=11)
        trees = [base, pb.PhyloTree(base.edge, base.edge_length * 1.3).with_states(base.states)]
        return capi.PM_V_MT, trees, cases.Q2, cases.PID2, 0.5, cases.PRIOR_BF
    if name == "ksmt":
        base = cases.tree_hidden(q4, T=10, S=2, seed=4, mean_branch=0.5)
        trees = [base, pb.PhyloTree(base.edge, base.edge_length * 1.2).with_states(base.states, segments=3)]
        return capi.PM_V_KSMT, trees, q4, p4, 4.0, cases.PRIOR_KSMT
    raise KeyError(name)


def _oracle_run(oracle, name, N, seed=7):
    v, trees, Q, pid, Om, prior = _oracle_case(name)
    orc = oracle.OracleRun(_oracle_variant(oracle, v), [t.oracle_dict() for t in trees], np.array(Q, dtype=np.float64),
                           pid, Om, N, prior=prior, rng_mode=oracle.KEYED, seed=seed)
    return v, trees, orc, orc.run()


@pytest.mark.parametrize("name", ["plain", "sparse", "bigtree", "bf", "dic2s", "ks", "dicks", "mt", "ksmt"])
def test_rebuild_row_reproduces_the_oracle(oracle, name):
    """The last oracle row is an exact function of the oracle's state: dwell times to 1e-12, off-diagonal counts exactly.
    For the multi-tree samplers the row is the tree named in its last column; both trees are exercised."""
    picks = set()
    for N in ((3, 4, 5, 6) if name in ("mt", "ksmt") else (5,)):
        v, trees, orc, rows = _oracle_run(oracle, name, N)
        row = rows[-1]
        t = int(row[-1]) if v in MULTI else 0
        picks.add(t)
        R, Nm = rebuild_row(orc, trees[t], t, full=v in FULL_COUNTS, parity=v in PARITY)
        audit_row(row, R, Nm, orc.n, v in FULL_COUNTS, 1e-12)
        if v in MULTI:   # and not the other tree's
            R2, N2 = rebuild_row(orc, trees[1 - t], 1 - t, full=True, parity=v in PARITY)
            assert not (np.allclose(R2, row[:orc.n], rtol=1e-12) and np.array_equal(N2, row_counts(row, orc.n, True) + np.diag(np.diag(N2))))
    if name in ("mt", "ksmt"):
        assert picks == {0, 1}


@pytest.mark.parametrize("name", ["bf", "dic2s", "ks", "dicks"])
def test_root_state_column_is_the_root_of_site_zero(oracle, name):
    v, trees, orc, rows = _oracle_run(oracle, name, 5)
    root = trees[0].order()[2]
    assert rows[-1, _root_state_col(v, orc.ncols)] == orc.node_states()[0, root - 1]


@pytest.mark.parametrize("name", ["plain", "sparse", "bigtree", "ks"])
def test_exact_partials_reproduce_the_oracle(oracle, name):
    """The oracle's stored partials are those of the last sweep's pruning, which used the piece counts the sweep before it
    left: after one sweep the initial maps, after two the counts read back after the first (KEYED streams do not depend
    on the chain length, so a one-sweep run shows them)."""
    v, trees, orc1, _ = _oracle_run(oracle, name, 1)
    _, _, orc2, _ = _oracle_run(oracle, name, 2)
    z = trees[0]
    S = z.n_sites()
    m0 = np.tile([len(mp) for mp in z.maps], (S, 1))
    norm = v in (capi.PM_V_BIGTREE,) or v in FULL_COUNTS
    B0 = np.eye(orc1.n) + np.asarray(_oracle_case(name)[2]) / _oracle_case(name)[4]
    for orc, m, B in ((orc1, m0, B0), (orc2, orc1.piece_counts(), np.array(orc1.B))):
        for s in range(S):
            want = exact_partials(z, s, m, B, parity=v in PARITY, sparse=v == capi.PM_V_SPARSE, normalize=norm)
            np.testing.assert_allclose(orc.partials(s)[z.T:], want[z.T:], rtol=1e-10, atol=0)
    assert not np.array_equal(orc1.piece_counts(), m0)   # the second comparison is not the first one again


def test_exact_loglik_reproduces_the_oracle_dic_columns(oracle):
    for name in ("dic2s", "dicks"):
        v, trees, orc, rows = _oracle_run(oracle, name, 4)
        for row in rows:
            if v == capi.PM_V_DIC2S:
                Q = np.array([[-row[6], row[6]], [row[7], -row[7]]])
            else:
                Q = synth.make2sQ(*row[20:25])
            np.testing.assert_allclose(row[-1], exact_loglik(trees[0], Q, orc.pid, parity=v == capi.PM_V_DICKS), rtol=1e-12)
    z = cases.tree2(T=30, S=7, seed=3)   # and the blocking over sites does not change the sum
    np.testing.assert_allclose(exact_loglik(z, cases.Q2, cases.PID2, max_doubles=1), exact_loglik(z, cases.Q2, cases.PID2), rtol=1e-13)


# ---- GPU: rows and stored paths ---------------------------------------------------------------------------------
def _bench_tree():
    import bench
    return bench.workload_tree()


def _gpu_case(name):
    """dict(v, trees, Q, pid, Om, prior, env, opts) of one audited production case."""
    q4, p4 = cases.q4(), np.full(4, 0.25)
    c = dict(prior=None, env={}, opts={}, pid=None)
    if name.startswith("plain2"):
        c.update(v=capi.PM_V_PLAIN, trees=[cases.tree2(T=100, S=1, seed=1, mean_branch=5.0)], Q=cases.Q2, pid=cases.PID2,
                 Om=0.2, env={"PHYLOMAP_B200_SMALL": name[-1]})
    elif name.startswith("bigtree4"):
        S = int(name.split("_")[1][1:])          # long branches: paths with several real jumps keep records
        c.update(v=capi.PM_V_BIGTREE, trees=[cases.tree_n(q4, T=300, S=S, seed=5, mean_branch=1.5, segments=3)], Q=q4,
                 pid=p4, Om=2.4)
        if "_f" in name:                          # _f<FUSED>p<REC_POOL>
            f, p = name.split("_f")[1].split("p")
            c["env"] = {"PHYLOMAP_B200_SMALL": "0", "PHYLOMAP_B200_FUSED": f, "PHYLOMAP_B200_REC_POOL": p}
    elif name == "sparse3_threshold":           # run-time n (the *_gen kernels), an entry of B below the SPARSE cut
        c.update(v=capi.PM_V_SPARSE, trees=[cases.tree_n(cases.jc(3), T=40, S=20, seed=2, mean_branch=3.0, segments=4)],
                 Q=SPARSE_THRESHOLD_Q, pid=np.full(3, 1 / 3), Om=0.4)
    elif name == "sparse5":
        Q = cases.jc(5, 0.1)
        c.update(v=capi.PM_V_SPARSE, trees=[cases.tree_n(Q, T=40, S=20, seed=3, mean_branch=2.0, segments=2)], Q=Q,
                 pid=np.full(5, 0.2), Om=1.0)
    elif name == "gap":                           # Omega t ~ 30: virtual jumps from exponential gaps on most branches
        c.update(v=capi.PM_V_PLAIN, trees=[cases.tree2(T=40, S=20, seed=6, mean_branch=75.0)], Q=cases.Q2, pid=cases.PID2,
                 Om=0.4)
    elif name == "saturated":                     # hundreds of runs per path: header records
        c.update(v=capi.PM_V_PLAIN, trees=[cases.tree2(T=6, S=40, seed=3, mean_branch=150.0)],
                 Q=np.array([[-1.0, 1.0], [1.0, -1.0]]), pid=cases.PID2, Om=2.0)
    elif name.startswith("ragged"):
        S = int(name[6:])
        tree = synth.yule_tree(333, seed=8, mean_branch=0.2)
        st = synth.simulate_tip_states(tree, q4, p4, S, seed=S).numpy()
        c.update(v=capi.PM_V_BIGTREE, trees=[tree.with_states(st, segments=2)], Q=q4, pid=p4, Om=2.4)
    elif name == "graph":
        c.update(v=capi.PM_V_BIGTREE, trees=[cases.tree_n(q4, T=60, S=45, seed=5, mean_branch=1.5, segments=3)], Q=q4,
                 pid=p4, Om=2.4, env={"PHYLOMAP_B200_SMALL": "0", "PHYLOMAP_B200_GRAPH": "1"})
    elif name == "powcap2":                       # a table of two powers: B^k by repeated products beyond it
        c.update(v=capi.PM_V_BIGTREE, trees=[cases.tree_n(q4, T=60, S=30, seed=7, mean_branch=2.0, segments=3)], Q=q4,
                 pid=p4, Om=2.4, opts={"power_capacity": 2})
    elif name == "bench":                         # the benchmark's tree
        tree, Q, pid = _bench_tree()
        st = synth.simulate_tip_states(tree, Q, pid, 4, seed=7).numpy()
        c.update(v=capi.PM_V_BIGTREE, trees=[tree.with_states(st, segments=2)], Q=Q, pid=pid, Om=2.4)
    elif name in ("bf", "dic2s"):
        c.update(v=capi.PM_V_BF if name == "bf" else capi.PM_V_DIC2S, trees=[cases.tree2(T=40, S=20, seed=8, mean_branch=4.0)],
                 Q=cases.Q2, pid=cases.PID2, Om=1.0, prior=cases.PRIOR_BF)
    elif name in ("ks4", "dicks"):
        c.update(v=capi.PM_V_KS if name == "ks4" else capi.PM_V_DICKS,
                 trees=[cases.tree_hidden(q4, T=60, S=20, seed=4, mean_branch=0.5)], Q=q4, pid=p4, Om=4.0, prior=cases.PRIOR_KS)
    elif name == "ks6":
        Q = cases.q6()
        c.update(v=capi.PM_V_KS, trees=[cases.tree_hidden(Q, T=40, S=10, seed=6, mean_branch=0.5)], Q=Q, pid=np.full(6, 1 / 6),
                 Om=8.0, prior=cases.PRIOR_KS)
    elif name == "mt":
        base = cases.tree2(T=30, S=10, seed=11, mean_branch=3.0)
        trees = [base, pb.PhyloTree(base.edge, base.edge_length * 1.3).with_states(base.states)]
        c.update(v=capi.PM_V_MT, trees=trees, Q=cases.Q2, pid=cases.PID2, Om=0.5, prior=cases.PRIOR_BF)
    elif name == "ksmt":
        base = cases.tree_hidden(q4, T=40, S=10, seed=4, mean_branch=0.5)
        trees = [base, pb.PhyloTree(base.edge, base.edge_length * 1.2).with_states(base.states, segments=3)]
        c.update(v=capi.PM_V_KSMT, trees=trees, Q=q4, pid=p4, Om=4.0, prior=cases.PRIOR_KSMT)
    else:
        raise KeyError(name)
    return c


def _chain(c, N, precision, monkeypatch, seed=11):
    for k, val in c["env"].items():
        monkeypatch.setenv(k, val)
    x = c["trees"] if c["v"] in MULTI else c["trees"][0]
    return pb.Chain(c["v"], x, np.asfortranarray(np.array(c["Q"], dtype=np.float64)), c["pid"], c["Om"], N, prior=c["prior"],
                    precision=precision, seed=seed, **c["opts"])


def _audit_last_row(ch, c, row, precision, name):
    v, n = c["v"], ch.n
    t = int(row[-1]) if v in MULTI else 0
    tree = c["trees"][t]
    R, N = rebuild_row(ch, tree, t, full=v in FULL_COUNTS, parity=v in PARITY,
                       len_rtol=1e-12 if precision == "f64" else 2e-5)
    gap = audit_row(row, R, N, n, v in FULL_COUNTS, 1e-12 if precision == "f64" else 1e-5)
    if precision == "f32":
        _note_gap("dwell times (%s)" % name.split("_")[0], gap)
    if v in (capi.PM_V_BF, capi.PM_V_KS, capi.PM_V_DIC2S, capi.PM_V_DICKS):
        assert row[_root_state_col(v, ch.ncols)] == ch.node_states()[0, tree.order()[2] - 1]
    return N


AUDIT_CASES = (["plain2_small1", "plain2_small0"] +
               ["bigtree4_S37_f%dp%d" % (f, p) for f in (0, 1) for p in (0, 1)] + ["bigtree4_S203"] +
               ["sparse3_threshold", "sparse5", "gap", "saturated", "ragged33", "ragged129", "graph", "powcap2",
                "bf", "dic2s", "ks4", "ks6", "dicks", "mt", "ksmt"])


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("name", AUDIT_CASES)
def test_row_is_the_sum_over_stored_paths(name, precision, monkeypatch):
    """run(k), then the last row must be rebuilt exactly from the stored state (dwell times: 1e-12 in FP64, 1e-5 in FP32)."""
    c = _gpu_case(name)
    K = 5
    ch = _chain(c, K, precision, monkeypatch)
    rows = ch.run(K)
    N = _audit_last_row(ch, c, rows[-1], precision, name)
    assert N.sum() > 0


@pytest.mark.gpu
def test_benchmark_tree_row_is_the_sum_over_stored_paths(monkeypatch):
    c = _gpu_case("bench")
    ch = _chain(c, 3, "f32", monkeypatch)
    _audit_last_row(ch, c, ch.run(3)[-1], "f32", "bench")


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("name", ["plain2_small1", "bigtree4_S37_f1p1", "bigtree4_S37_f0p0", "gap", "saturated",
                                  "sparse5", "graph", "ks4", "ksmt"])
def test_row_audit_after_every_call(name, precision, monkeypatch):
    """run(1) four times, audited after each call: the stored records alternate between two buffers from sweep to sweep
    and each sweep regenerates the previous sweep's virtual jumps from the stored counts."""
    c = _gpu_case(name)
    ch = _chain(c, 4, precision, monkeypatch)
    for _ in range(4):
        _audit_last_row(ch, c, ch.run(1)[-1], precision, name)


# ---- GPU: node draws and partials -------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("name", ["bigtree4_S37", "sparse3_threshold", "ks4", "ks6", "dicks", "ksmt"])
def test_node_draws_have_positive_probability(name, precision, monkeypatch):
    """Models with structural zeros (hidden-rate generators, a SPARSE-dropped entry, parity tips): after run(k - 1) the
    next sweep prunes with the piece counts m read back then; every node it draws must have a positive exact partial
    (the root: positive pid x partial) and every branch B^(m - 1)[parent state, child state] > 0."""
    c = _gpu_case(name)
    v = c["v"]
    ch = _chain(c, 4, precision, monkeypatch)
    ch.run(3)
    sparse = v == capi.PM_V_SPARSE
    trees = c["trees"] if v in MULTI else c["trees"][:1]
    m_prev = [ch.piece_counts(t) for t in range(len(trees))]
    B = np.array(ch.B)                     # the rate update that ended sweep k - 1 set the B of sweep k
    ch.run(1)
    for t, tree in enumerate(trees):
        m = m_prev[t]
        ns = ch.node_states(t)
        T, root = tree.T, tree.order()[2]
        Bs = np.where(B > SPARSE_DROP, B, 0.0) if sparse else B
        par, chi = tree.edge[:, 0] - 1, tree.edge[:, 1] - 1
        for s in range(tree.n_sites()):
            sup = exact_partials(tree, s, m, B, parity=v in PARITY, sparse=sparse, support=True)
            assert np.all(sup[np.arange(T, 2 * T - 1), ns[s, T:]] > 0), "site %d: a node drawn into a state of probability 0" % s
            assert c["pid"][ns[s, root - 1]] > 0
            pw = _power_table(Bs, np.unique(m[s] - 1), True)
            ok = [pw[m[s, e] - 1][ns[s, par[e]], ns[s, chi[e]]] > 0 for e in range(tree.E)]
            assert all(ok), "site %d: branches %s join states B^(m-1) cannot" % (s, np.flatnonzero(~np.array(ok))[:5])


def _audit_partials(ch, tree, sites, m, B, precision, parity=False, sparse=False, tree_index=0, what=""):
    T = tree.T
    for s in sites:
        exact = exact_partials(tree, s, m, B, parity=parity, sparse=sparse)[T:]
        got = ch.partials(s, tree_index)[T:]
        assert np.all(got[exact == 0] == 0), "site %d: structural zeros must stay exact zeros" % s
        big = exact > 1e-6
        np.testing.assert_allclose(got[big], exact[big], rtol=2e-3 if precision == "f32" else 1e-9, err_msg="site %d" % s)
        assert np.all(got[exact < 1e-30] < 1e-20)
        if precision == "f32":
            _note_gap("partials above 1e-6 (%s)" % what, np.max(np.abs(got[big] - exact[big]) / exact[big]))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("name", ["plain2_small0", "bigtree4_S37_f0p1", "bigtree4_S37_f1p1", "sparse3_threshold", "sparse5",
                                  "powcap2", "ksmt"])
def test_partials_match_exact_pruning(name, precision, monkeypatch):
    """time_prune on the state of run(k), then partials(s) against exact_partials with the piece counts read back."""
    c = _gpu_case(name)
    v = c["v"]
    ch = _chain(c, 3, precision, monkeypatch)
    ch.run(3)
    t = 1 if v == capi.PM_V_KSMT else 0
    tree = c["trees"][t]
    m = ch.piece_counts(t)
    ch.time_prune(reps=1, tree=t)
    if name == "powcap2":
        assert m.max() - 1 > 2      # powers beyond the table in use
    S = tree.n_sites()
    sites = sorted(set([0, S // 2, S - 1]))
    _audit_partials(ch, tree, sites, m, np.array(ch.B), precision, parity=v in PARITY, sparse=v == capi.PM_V_SPARSE,
                    tree_index=t, what=name.split("_")[0])


PARTIALS_LAYOUTS = ([(name, p) for name in ["plain2_small1", "bigtree4_S40000_f1p1", "bigtree4_S37_f1p1", "bigtree4_S37_f0p1",
                                             "dic2s"] for p in ("f32", "f64")] + [("bigtree4_S37_deterministic", "f64")])


@pytest.mark.gpu
@pytest.mark.parametrize("name,precision", PARTIALS_LAYOUTS)
def test_partials_prune_the_current_state(name, precision, monkeypatch):
    """partials(s) right after run(k), with no time_prune before it, against exact_partials with the piece counts read back:
    the call prunes the current state itself, whichever kernels the chain runs.  The layouts: the one-block-per-site chain
    (which writes no partials array of its own), the fused kernel with more site blocks than slots, with fewer, the separate
    kernels, a DIC chain (whose log-likelihood pass reuses the partials array) and the deterministic mode."""
    if name == "bigtree4_S40000_f1p1":          # more site blocks than any B200 has slots (at most 8 x 148 x 32 sites)
        c = _gpu_case("bigtree4_S37_f1p1")
        c["trees"] = [cases.tree_n(cases.q4(), T=40, S=40000, seed=5, mean_branch=1.5, segments=3)]
    elif name == "bigtree4_S37_deterministic":
        c = _gpu_case("bigtree4_S37")
        c["opts"] = {"mode": "deterministic"}
    else:
        c = _gpu_case(name)
    ch = _chain(c, 3, precision, monkeypatch)
    ch.run(3)
    tree = c["trees"][0]
    S = tree.n_sites()
    _audit_partials(ch, tree, sorted(set([0, S // 2, S - 1])), ch.piece_counts(), np.array(ch.B), precision,
                    what=name.split("_")[0])


def _underflow_sites(tree, m, B, limit=1e-30):
    """Sites of `tree` where some node's unnormalised product of the two (normalised) child contributions sums to less
    than `limit` in FP64: where FP32 pruning redoes the node in double."""
    n, T = B.shape[0], tree.T
    nen = tree.order()[0]
    chi, par = tree.edge[:, 1] - 1, tree.edge[:, 0] - 1
    ks = np.unique(m - 1)
    pw = np.zeros((ks.max() + 1, n, n))
    for k in ks:
        pw[k] = np.linalg.matrix_power(B, int(k))
    data = _data(tree)
    S = data.shape[0]
    low = np.full(S, np.inf)
    blk = 2048
    for s0 in range(0, S, blk):
        d = data[s0:s0 + blk]
        b = d.shape[0]
        PL = np.zeros((2 * T - 1, b, n))
        PL[np.arange(T)[:, None], np.arange(b)[None, :], (d - 1).T] = 1
        for i in range(T - 1):
            ea, eb = nen[2 * i] - 1, nen[2 * i + 1] - 1
            va = np.einsum("sij,sj->si", pw[m[s0:s0 + b, ea] - 1], PL[chi[ea]])
            vb = np.einsum("sij,sj->si", pw[m[s0:s0 + b, eb] - 1], PL[chi[eb]])
            v = va * vb
            sv = v.sum(1)
            low[s0:s0 + b] = np.minimum(low[s0:s0 + b], sv)
            PL[par[ea]] = v / sv[:, None]
    return np.flatnonzero(low < limit)


@pytest.mark.gpu
def test_partials_fp32_underflow_redo():
    """Two clades of eight tips, each all but certain of a different state, meet at the root: with B = I + Q / Omega mixing
    states by 1e-4 on the two-piece tip branches and not at all on the one-piece internal branches, each clade's partial
    of the other state is 1e-32, and the FP32 product at the root (2e-32) underflows the 1e-30 bar although both factors
    are representable.  The kernel redoes such nodes in double.  (The Squamate tree with the vignette's Q and Omega has no
    such site among 20 000 simulated ones.)  The sites are found on the host first, then their partials audited."""
    Q = np.array([[-1e-4, 1e-4], [1e-4, -1e-4]])
    tree = synth.balanced_tree(4, branch=1.0)
    S = 24
    st = np.ones((S, tree.T), dtype=np.int32)
    st[: S // 2, tree.T // 2:] = 2
    st[S // 2:, : tree.T // 2] = 2
    maps = [np.full(2 if c <= tree.T else 1, L / (2 if c <= tree.T else 1)) for c, L in zip(tree.edge[:, 1], tree.edge_length)]
    z = pb.PhyloTree(tree.edge, tree.edge_length, st, maps, [np.ones(len(mp), dtype=np.int32) for mp in maps])
    ch = pb.Chain(capi.PM_V_BIGTREE, z, np.asfortranarray(Q), cases.PID2, 1.0, 1, precision="f32", seed=3)
    m = ch.piece_counts()          # the initial maps: the first sweep prunes with these
    B = np.array(ch.B)
    sites = _underflow_sites(z, m, B)
    assert len(sites) == S, "the sites do not exercise the FP32 redo (found %d)" % len(sites)
    ch.time_prune(reps=1)
    _audit_partials(ch, z, range(S), m, B, "f32", what="underflow redo")
    root = z.order()[2]
    np.testing.assert_allclose(ch.partials(0)[root - 1], [0.5, 0.5], rtol=1e-6)


# ---- GPU: log-likelihood ----------------------------------------------------------------------------------------
def _loglik_case(name):
    if name == "squamate_n2":
        Q = np.array([[-0.001, 0.001], [0.006, -0.006]])
        z = synth.simulate_2_state_tree(101, cases.squamate_tree(), Q, cases.PID2, n_sites=2000, device="cuda")
        return z, Q, cases.PID2, False
    if name == "bench_parity":
        tree, Q, pid = _bench_tree()
        st = synth.simulate_tip_states(tree, Q, pid, 1024, seed=7, device="cuda").cpu().numpy()
        return tree.with_states(((st.astype(np.int64) - 1) % 2 + 1).astype(np.int32)), Q, pid, True
    if name == "n8_parity":
        Q = synth.make2sQ(0.1, 0.15, [0.2, 0.1, 0.3], [0.2, 0.3, 0.1], [5.0, 0.5, 1.0])
        z = cases.tree_hidden(Q, T=200, S=64, seed=9, mean_branch=0.7)
        return z, Q, np.full(8, 1 / 8), True
    if name == "long_branches":               # ||Q t|| ~ 50: many squarings in the matrix exponential
        Q = np.array([[-1.0, 1.0], [1.0, -1.0]])
        z = cases.tree2(T=60, S=64, seed=4, mean_branch=25.0)
        return z, Q, cases.PID2, False
    if name == "long_branches_n5":
        Q = cases.jc(5, 0.5)
        z = cases.tree_n(Q, T=60, S=64, seed=4, mean_branch=12.5)
        return z, Q, np.full(5, 0.2), False
    raise KeyError(name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["squamate_n2", "bench_parity", "n8_parity", "long_branches", "long_branches_n5"])
def test_loglik_at_scale(name):
    z, Q, pid, parity = _loglik_case(name)
    want = exact_loglik(z, Q, pid, parity=parity)
    np.testing.assert_allclose(pb.loglik(z, Q, pid, parity_tips=parity, precision="f64"), want, rtol=1e-10)
    got32 = pb.loglik(z, Q, pid, parity_tips=parity, precision="f32")
    _note_gap("log-likelihood", abs(got32 - want) / abs(want))
    np.testing.assert_allclose(got32, want, rtol=1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_dicks_loglik_column_at_4096_sites(precision):
    Q, pid = cases.q4(), np.full(4, 0.25)
    tree = synth.yule_tree(200, seed=6, mean_branch=0.4)
    z = synth.simulate_4_state_tree(9, tree, Q, pid, n_sites=4096, device="cuda", segments=2)
    rows = pb.sumstatMCMCksDICt(z, np.asfortranarray(Q.copy()), pid, 4.0, 4, cases.PRIOR_KS, precision=precision, seed=5)
    row = rows[-1]
    want = exact_loglik(z, synth.make2sQ(*row[20:25]), pid, parity=True)
    if precision == "f64":
        np.testing.assert_allclose(row[-1], want, rtol=1e-10)
    else:
        _note_gap("log-likelihood", abs(row[-1] - want) / abs(want))
        np.testing.assert_allclose(row[-1], want, rtol=1e-4)


@pytest.mark.gpu
def test_loglik_rejects_more_than_eight_states():
    Q = cases.jc(10, 0.1)
    z = cases.tree_n(Q, T=12, S=2, seed=1)
    with pytest.raises(capi.PhylomapError) as ei:
        pb.loglik(z, Q, np.full(10, 0.1))
    assert ei.value.code == capi.PM_ERR_ARG

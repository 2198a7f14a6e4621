"""Stochastic maps exported from a resident chain (Chain.maps / pm_chain_get_maps) against the per-path read-back
pm_chain_get_path, bit for bit, on every chain layout of the state audit (tests/test_gpu_state_audit.py): the
one-block-per-site kernel, pooled and per-site record slices, header records, ragged site counts, graph replay, run-time
n, the rate samplers and both trees of mt / ksmt; and against the rows the sweeps returned."""
import ctypes as C

import numpy as np
import pytest

import cases
import phylomap_b200 as pb
from phylomap_b200 import capi
from test_gpu_state_audit import AUDIT_CASES, FULL_COUNTS, MULTI, _chain, _gpu_case, rebuild_row, row_counts


def _reference(ch, tree_index, S, E):
    """Every (site, branch) through path(): {(site, e): (lengths, states)}."""
    return {(s, e): ch.path(s, e, tree_index, cap=4096) for s in range(S) for e in range(E)}


def _state(ch):
    """export_state() into a zeroed buffer: the blob pads every device buffer to 16 bytes, and the padding is not written."""
    L = capi.lib()
    buf = np.zeros(int(L.pm_chain_state_bytes(ch.h)), dtype=np.uint8)
    err = C.create_string_buffer(512)
    capi.check(L.pm_chain_export_state(ch.h, capi.ptr(buf), buf.size, err, 512), err)
    return buf


def _same_bits(a, b):
    return a.shape == b.shape and np.array_equal(np.asarray(a, dtype=np.float64).view(np.int64), np.asarray(b, dtype=np.float64).view(np.int64))


def _check_against(ref, m, pairs=None):
    E = m.E
    bad = []
    for i, e in (pairs if pairs is not None else ((i, e) for i in range(len(m)) for e in range(E))):
        ln, st = m.path(i, e)
        rl, rs = ref[(int(m.sites[i]), e)]
        if not (_same_bits(ln, rl) and np.array_equal(st, rs)):
            bad.append("selection %d (site %d) branch %d: %s %s, path() %s %s" % (i, m.sites[i], e, ln[:6], st[:6], rl[:6], rs[:6]))
    assert not bad, "%d runs differ from path(), e.g.\n  %s" % (len(bad), "\n  ".join(bad[:5]))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("name", AUDIT_CASES)
def test_maps_equal_path_for_every_site_and_branch(name, precision, monkeypatch):
    """run(5), then the export of all sites and of a shuffled selection with repeats equals path() bit for bit; the maps
    sum to the last row (dwell times: 1e-12 in FP64, 1e-5 in FP32; off-diagonal counts exactly), and the call leaves the
    exported chain state byte for byte as it was."""
    c = _gpu_case(name)
    v = c["v"]
    ch = _chain(c, 5, precision, monkeypatch)
    row = ch.run(5)[-1]
    before = _state(ch)
    rng = np.random.default_rng(3)
    trees = c["trees"] if v in MULTI else c["trees"][:1]
    for t, tree in enumerate(trees):
        S, E = tree.n_sites(), tree.E
        ref = _reference(ch, t, S, E)
        m = ch.maps(tree=t)
        assert m.tree is ch.trees[t] and len(m) == S
        np.testing.assert_array_equal(m.sites, np.arange(S))
        _check_against(ref, m)
        sel = np.concatenate([rng.permutation(S), rng.integers(0, S, size=7)])
        _check_against(ref, ch.maps(sel, tree=t))
        if t == (int(row[-1]) if v in MULTI else 0):     # the tree this row describes
            n = ch.n
            off = ~np.eye(n, dtype=bool)
            N = m.transitions().sum(0)
            assert np.array_equal(N[off], row_counts(row, n, v in FULL_COUNTS)[off])
            assert N.sum() > 0
            R = m.mapped_edge().sum((0, 1))
            np.testing.assert_allclose(row[:n], R, rtol=1e-12 if precision == "f64" else 1e-5)
    assert np.array_equal(_state(ch), before), "maps() changed the chain state"


@pytest.mark.gpu
def test_maps_equal_path_in_deterministic_mode(monkeypatch):
    """Deterministic mode keeps every path as records, the paths of a chunk one after the other."""
    c = _gpu_case("bigtree4_S37")
    c["opts"] = {"mode": "deterministic"}
    ch = _chain(c, 5, "f64", monkeypatch)
    row = ch.run(5)[-1]
    tree = c["trees"][0]
    S, E = tree.n_sites(), tree.E
    ref = _reference(ch, 0, S, E)
    m = ch.maps()
    _check_against(ref, m)
    _check_against(ref, ch.maps(np.random.default_rng(5).integers(0, S, size=50)))
    n = ch.n
    off = ~np.eye(n, dtype=bool)
    assert np.array_equal(m.transitions().sum(0)[off], row_counts(row, n, False)[off])
    np.testing.assert_allclose(row[:n], m.mapped_edge().sum((0, 1)), rtol=1e-12)


def _same_maps(a, b):
    return np.array_equal(a.off, b.off) and _same_bits(a.length, b.length) and np.array_equal(a.state, b.state)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["bigtree4_S37_f1p1", "ks4"])
def test_sample_maps_rows_equal_one_run(name, monkeypatch):
    c = _gpu_case(name)
    a = _chain(c, 10, "f32", monkeypatch)
    rows, maps = a.sample_maps(10, 2, sites=[3, 1, 3])
    assert len(maps) == 5 and all(len(m) == 3 for m in maps)
    c = _gpu_case(name)
    b = _chain(c, 10, "f32", monkeypatch)
    want = b.run(10)
    assert np.array_equal(rows, want)
    assert _same_maps(maps[-1], b.maps([3, 1, 3]))
    assert not _same_maps(maps[0], maps[-1])


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_maps_after_import_state_equal_the_uninterrupted_chain(precision, monkeypatch):
    c = _gpu_case("bigtree4_S37_f1p1")
    a = _chain(c, 6, precision, monkeypatch)
    a.run(3)
    blob = a.export_state()
    a.run(2)
    b = _chain(c, 6, precision, monkeypatch)
    b.import_state(blob)
    b.run(2)
    assert _same_maps(b.maps(), a.maps())


@pytest.mark.gpu
def test_selection_larger_than_one_batch_on_the_benchmark_tree(monkeypatch):
    """The benchmark tree (19 998 branches) with more selected sites than one batch holds: sampled (site, branch) pairs,
    among them both sides of every batch boundary, against path()."""
    import bench
    from phylomap_b200 import synth
    tree, Q, pid = bench.workload_tree()
    S = 1200
    st = synth.simulate_tip_states(tree, Q, pid, S, seed=7).numpy()
    z = tree.with_states(st, segments=2)
    ch = pb.Chain(capi.PM_V_BIGTREE, z, np.asfortranarray(Q.copy()), pid, 2.4, 3, precision="f32", seed=5)
    ch.run(3)
    E = tree.E
    per_batch = (512 << 20) // 2 // (E * 12 + 8)        # sites per batch (pm_maps.cuh kMapsScratchBytes, pm_host.cu maps())
    rng = np.random.default_rng(11)
    sel = np.concatenate([np.arange(S), rng.integers(0, S, size=2 * per_batch + 100 - S)])
    assert len(sel) > 2 * per_batch
    m = ch.maps(sel)
    pairs = set(zip(rng.integers(0, len(sel), size=2000).tolist(), rng.integers(0, E, size=2000).tolist()))
    for b in range(per_batch, len(sel), per_batch):
        for i in (b - 1, b):
            pairs.update((i, e) for e in (0, 1, E // 2, E - 2, E - 1))
    ref = {}
    for i, e in pairs:
        s = int(sel[i])
        if (s, e) not in ref:
            ref[(s, e)] = ch.path(s, e, cap=4096)
    _check_against(ref, m, sorted(pairs))
    assert np.all(np.diff(m.off) >= 1)


def _raw_maps(ch, sel, cap, with_runs=True, tree=0):
    E = ch.trees[0].E
    sel = np.ascontiguousarray(sel, dtype=np.int64)
    off = np.full(len(sel) * E + 1, -1, dtype=np.int64)
    ln = np.zeros(max(cap, 1))
    st = np.zeros(max(cap, 1), dtype=np.int32)
    err = C.create_string_buffer(512)
    rc = capi.lib().pm_chain_get_maps(ch.h, tree, capi.ptr(sel), len(sel), capi.ptr(off), capi.ptr(ln) if with_runs else None,
                                      capi.ptr(st) if with_runs else None, cap, err, 512)
    return rc, err.value.decode(), off


@pytest.mark.gpu
def test_maps_errors(monkeypatch):
    c = _gpu_case("bigtree4_S37_f1p1")
    ch = _chain(c, 3, "f32", monkeypatch)
    rc, msg, _ = _raw_maps(ch, [0], 0, with_runs=False)
    assert rc == capi.PM_ERR_ARG and "no sweep done yet" in msg
    ch.run(2)
    for sel in ([37], [-1], [0, 5, 40]):
        rc, msg, _ = _raw_maps(ch, sel, 0, with_runs=False)
        assert rc == capi.PM_ERR_ARG and "bad site" in msg
    rc, msg, _ = _raw_maps(ch, [0], 0, with_runs=False, tree=1)
    assert rc == capi.PM_ERR_ARG and "bad tree" in msg
    m = ch.maps([4, 2])
    total = int(m.off[-1])
    rc, msg, off = _raw_maps(ch, [4, 2], total - 1)
    assert rc == capi.PM_ERR_CAPACITY
    assert np.array_equal(off, m.off)
    rc, msg, off = _raw_maps(ch, [4, 2], total)
    assert rc == capi.PM_OK and np.array_equal(off, m.off)
    # the direct sampler keeps no paths, and it cannot be created as a resident chain at all
    z = cases.tree2(T=8)
    with pytest.raises(capi.PhylomapError) as ei:
        pb.Chain(capi.PM_V_EXP, z, np.asfortranarray(cases.Q2), cases.PID2, 0.1, 2)
    assert ei.value.code == capi.PM_ERR_ARG


@pytest.mark.gpu
def test_exported_map_seeds_a_new_chain(monkeypatch):
    """A single-site export, as to_tree(0), is the initial maps of a new chain, which runs and leaves a valid history."""
    c = _gpu_case("bigtree4_S37")
    ch = _chain(c, 3, "f64", monkeypatch)
    ch.run(3)
    m = ch.maps([5])
    z = m.to_tree(0)
    assert [len(x) for x in z.maps] == list(np.diff(m.off))
    assert pb.PhyloTree.from_mapping(z.to_mapping()).n_sites() == 1
    ch2 = pb.Chain(capi.PM_V_BIGTREE, z, np.asfortranarray(np.array(c["Q"], dtype=np.float64)), c["pid"], c["Om"], 3,
                   precision="f64", seed=4)
    np.testing.assert_array_equal(ch2.piece_counts()[0], [len(x) for x in z.maps])
    row = ch2.run(3)[-1]
    R, N = rebuild_row(ch2, z)
    np.testing.assert_allclose(row[:ch2.n], R, rtol=1e-12)

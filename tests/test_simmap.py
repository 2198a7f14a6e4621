"""CPU checks of the stochastic-map export's host side: summaries of hand-built maps, the phytools simmap / multiSimmap
objects through the RDS writer and reader, the phylomap layout of `to_tree`, and the entry's refusal to run without a B200."""
import ctypes as C

import numpy as np
import pytest

import cases
import phylomap_b200 as pb
from phylomap_b200 import capi, rds
from phylomap_b200.simmap import StochasticMaps, multi_simmap


def _tree():
    # ((1,2)4,3)5 written as an ape edge matrix: tips 1..3, root 4, internal node 5
    edge = np.array([[4, 5], [5, 1], [5, 2], [4, 3]], dtype=np.int32)
    return pb.PhyloTree(edge, [1.0, 2.0, 3.0, 4.0], np.array([[1, 2, 2], [2, 2, 1]], dtype=np.int32))


def _maps():
    """Two sites on _tree(), 3 states.  Site 0: branch 0 = (0.25, s0), (0.75, s2); branch 1 = (2, s0); branch 2 = (1, s0),
    (1.5, s1), (0.5, s0); branch 3 = (4, s1).  Site 1: every branch one run of state 1 except branch 3 = (1, s1), (3, s2)."""
    t = _tree()
    runs = [[[(0.25, 0), (0.75, 2)], [(2.0, 0)], [(1.0, 0), (1.5, 1), (0.5, 0)], [(4.0, 1)]],
            [[(1.0, 1)], [(2.0, 1)], [(3.0, 1)], [(1.0, 1), (3.0, 2)]]]
    off, ln, st = [0], [], []
    for site in runs:
        for br in site:
            for L, s in br:
                ln.append(L)
                st.append(s)
            off.append(len(ln))
    return StochasticMaps([0, 1], off, ln, st, 3, t)


def test_mapped_edge_and_transitions_of_hand_built_maps():
    m = _maps()
    me = m.mapped_edge()
    assert me.shape == (2, 4, 3)
    np.testing.assert_array_equal(me[0], [[0.25, 0, 0.75], [2, 0, 0], [1.5, 1.5, 0], [0, 4, 0]])
    np.testing.assert_array_equal(me[1], [[0, 1, 0], [0, 2, 0], [0, 3, 0], [0, 1, 3]])
    np.testing.assert_array_equal(me.sum(2), np.tile(m.tree.edge_length, (2, 1)))
    tr = m.transitions()
    want0 = np.zeros((3, 3), dtype=np.int64)
    want0[0, 2] = want0[0, 1] = want0[1, 0] = 1
    want1 = np.zeros((3, 3), dtype=np.int64)
    want1[1, 2] = 1
    np.testing.assert_array_equal(tr, [want0, want1])
    ln, st = m.path(0, 2)
    np.testing.assert_array_equal(ln, [1.0, 1.5, 0.5])
    np.testing.assert_array_equal(st, [0, 1, 0])


def test_inconsistent_csr_arrays_are_refused():
    m = _maps()
    with pytest.raises(ValueError):
        StochasticMaps([0], m.off, m.length, m.state, 3, m.tree)


def test_simmap_and_multisimmap_survive_an_rds_round_trip(tmp_path):
    m = _maps()
    Q = np.array([[-1.0, 0.5, 0.5], [0.2, -0.4, 0.2], [0.1, 0.1, -0.2]])
    one = m.to_simmap(0, Q=Q, labels=["a", "b", "c"])
    path = str(tmp_path / "one.rds")
    rds.write_rds(path, one)
    got = rds.read_rds(path)
    assert got.attributes["class"] == ["simmap", "phylo"]
    v = got.value
    assert list(v) == ["edge", "edge.length", "Nnode", "tip.label", "maps", "mapped.edge", "Q"]
    np.testing.assert_array_equal(v["edge"], m.tree.edge)
    assert v["edge"].dtype == np.int32
    np.testing.assert_array_equal(v["edge.length"], m.tree.edge_length)
    assert int(v["Nnode"][0]) == 2 and v["tip.label"] == ["t1", "t2", "t3"]
    assert len(v["maps"]) == 4
    np.testing.assert_array_equal(v["maps"][2].value, [1.0, 1.5, 0.5])
    assert v["maps"][2].attributes["names"] == ["a", "b", "a"]
    me = v["mapped.edge"]
    np.testing.assert_array_equal(me.value, m.mapped_edge()[0])
    assert me.attributes["dimnames"] == [["4,5", "5,1", "5,2", "4,3"], ["a", "b", "c"]]
    np.testing.assert_array_equal(v["Q"].value, Q)
    assert v["Q"].attributes["dimnames"] == [["a", "b", "c"], ["a", "b", "c"]]

    path = str(tmp_path / "multi.rds")
    rds.write_rds(path, multi_simmap([m.to_simmap(i) for i in range(len(m))]))
    got = rds.read_rds(path)
    assert got.attributes["class"] == ["multiSimmap", "multiPhylo"]
    assert len(got.value) == 2
    for i, s in enumerate(got.value):
        assert s.attributes["class"] == ["simmap", "phylo"]
        assert "Q" not in s.value
        assert s.value["mapped.edge"].attributes["dimnames"][1] == ["1", "2", "3"]
        for e in range(4):
            ln, st = m.path(i, e)
            np.testing.assert_array_equal(s.value["maps"][e].value, ln)
            assert s.value["maps"][e].attributes["names"] == [str(x + 1) for x in st]


def test_to_tree_is_the_phylomap_input_layout():
    m = _maps()
    t = m.to_tree(1)
    back = pb.PhyloTree.from_mapping(t.to_mapping())
    np.testing.assert_array_equal(back.edge, m.tree.edge)
    np.testing.assert_array_equal(back.states, [2, 2, 1])
    assert [list(x) for x in back.mapnames] == [[2], [2], [2], [2, 3]]
    assert [list(x) for x in back.maps] == [[1.0], [2.0], [3.0], [1.0, 3.0]]
    order = back.order()
    flat, _ = back.flat(*order)                  # what a new chain would be created from
    assert flat.n_sites == 1 and flat.n_edges == 4


def test_maps_entry_refuses_to_run_without_a_b200():
    """No chain can be created without a usable sm_100 device (PM_ERR_CUDA), and the entry itself rejects a missing chain
    without touching a device."""
    L = capi.lib()
    off = np.full(5, -1, dtype=np.int64)
    sel = np.zeros(1, dtype=np.int64)
    err = C.create_string_buffer(256)
    assert L.pm_chain_get_maps(None, 0, capi.ptr(sel), 1, capi.ptr(off), None, None, 0, err, 256) == capi.PM_ERR_ARG
    if L.pm_device_count() > 0:
        pytest.skip("a B200 is present")
    z = cases.tree2(T=8)
    with pytest.raises(capi.PhylomapError) as e:
        pb.Chain(capi.PM_V_PLAIN, z, np.asfortranarray(cases.Q2), cases.PID2, 0.2, 2)
    assert e.value.code == capi.PM_ERR_CUDA

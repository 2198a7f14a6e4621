"""Sampled stochastic maps of a resident chain (`Chain.maps`) and their phylomap / phytools layouts.

A stochastic map is the history of one character on every branch of the tree: the runs (length, state) from the parent
end of a branch to its child end.  `Chain.maps` decodes the histories the chain holds after its last sweep on the device
and returns them as CSR arrays; everything here is host arithmetic over those arrays.

    m = chain.maps(sites=[0, 5])     # StochasticMaps of local sites 0 and 5
    m.path(1, e)                     # runs of site 5 on branch e: (lengths, 0-based states)
    m.mapped_edge()                  # [k, E, n] time per state per branch
    m.transitions()                  # [k, n, n] changes between consecutive runs, summed over branches
    m.to_tree(0)                     # PhyloTree with site 0's history as its maps (a new chain's initial maps)
    rds.write_rds(path, multi_simmap([m.to_simmap(i) for i in range(2)]))   # phytools' multiSimmap
"""
import numpy as np

from .rds import RObject
from .tree import PhyloTree


class StochasticMaps:
    """The histories of the selected sites on every branch of `tree`, in CSR form: the runs of the i-th selected site on
    branch e (edge-row order) are `length[off[i*E + e]:off[i*E + e + 1]]` and `state[...]` (0-based), parent end first.
    `sites` are the chain's local site indices, `n` its number of states."""

    def __init__(self, sites, off, length, state, n, tree):
        self.sites = np.asarray(sites, dtype=np.int64)
        self.off = np.asarray(off, dtype=np.int64)
        self.length = np.asarray(length, dtype=np.float64)
        self.state = np.asarray(state, dtype=np.int32)
        self.n = int(n)
        self.tree = tree
        self.E = tree.E
        if self.off.shape != (len(self.sites) * self.E + 1,) or self.off[-1] != len(self.length) or len(self.state) != len(self.length):
            raise ValueError("inconsistent CSR arrays")

    def __len__(self):
        return len(self.sites)

    def path(self, i, e):
        """(lengths, 0-based states) of the i-th selected site on branch e, parent end first."""
        a, b = self.off[i * self.E + e], self.off[i * self.E + e + 1]
        return self.length[a:b], self.state[a:b]

    def _group(self):
        """(site, branch) group of every run: i * E + e."""
        return np.repeat(np.arange(len(self.off) - 1, dtype=np.int64), np.diff(self.off))

    def mapped_edge(self):
        """[k, E, n]: time spent in each state on each branch, per selected site (phytools' mapped.edge)."""
        k, E, n = len(self.sites), self.E, self.n
        g = self._group()
        return np.bincount(g * n + self.state, weights=self.length, minlength=k * E * n).reshape(k, E, n)

    def transitions(self):
        """[k, n, n]: number of changes from state a to state b between consecutive runs of a branch, summed over the
        branches, per selected site."""
        k, E, n = len(self.sites), self.E, self.n
        g = self._group()
        same = g[1:] == g[:-1]
        a, b, site = self.state[:-1][same], self.state[1:][same], g[:-1][same] // E
        return np.bincount((site * n + a) * n + b, minlength=k * n * n).reshape(k, n, n)

    def _tip_states(self, i):
        st = self.tree.states
        if st is None:
            return None
        st = np.asarray(st)
        return st.copy() if st.ndim == 1 else st[self.sites[i]].copy()

    def to_tree(self, i):
        """PhyloTree of the i-th selected site in the phylomap input layout: its history as `maps` / `mapnames` (1-based
        states) and its tip data as `states`, so that it can seed a new chain."""
        E = self.E
        maps, names = [], []
        for e in range(E):
            ln, st = self.path(i, e)
            maps.append(ln.copy())
            names.append((st + 1).astype(np.int32))
        t = self.tree
        return PhyloTree(t.edge, t.edge_length, self._tip_states(i), maps, names, t.tip_label)

    def to_simmap(self, i, Q=None, labels=None):
        """The i-th selected site as phytools' class c("simmap", "phylo") (what describe.simmap, densityMap and plotSimmap
        read), for `rds.write_rds`: edge, edge.length, Nnode, tip.label (t1..tT when the tree has none), maps (per branch
        the run lengths named by state label, parent end first), mapped.edge (E x n, rownames "parent,child", colnames the
        labels) and Q when given.  labels: the state names, by default "1".."n" (phylomap's 1-based states)."""
        t, n = self.tree, self.n
        labels = [str(s + 1) for s in range(n)] if labels is None else [str(x) for x in labels]
        if len(labels) != n:
            raise ValueError("need %d state labels" % n)
        maps = []
        for e in range(self.E):
            ln, st = self.path(i, e)
            maps.append(RObject(ln.copy(), {"names": [labels[s] for s in st]}))
        rown = ["%d,%d" % (p, c) for p, c in t.edge]
        obj = {"edge": t.edge.astype(np.int32), "edge.length": t.edge_length.copy(),
               "Nnode": np.array([t.Nnode], dtype=np.int32),
               "tip.label": list(t.tip_label) if t.tip_label is not None else ["t%d" % (j + 1) for j in range(t.T)],
               "maps": maps,
               "mapped.edge": RObject(self._site_mapped_edge(i), {"dimnames": [rown, list(labels)]})}
        if Q is not None:
            obj["Q"] = RObject(np.array(Q, dtype=np.float64).reshape(n, n), {"dimnames": [list(labels), list(labels)]})
        return RObject(obj, {"class": ["simmap", "phylo"]})

    def _site_mapped_edge(self, i):
        """[E, n]: mapped_edge() of the i-th selected site alone."""
        E, n = self.E, self.n
        a, b = self.off[i * E], self.off[(i + 1) * E]
        g = np.repeat(np.arange(E, dtype=np.int64), np.diff(self.off[i * E:(i + 1) * E + 1]))
        return np.bincount(g * n + self.state[a:b], weights=self.length[a:b], minlength=E * n).reshape(E, n)


def multi_simmap(simmaps):
    """phytools' class c("multiSimmap", "multiPhylo"): a list of `StochasticMaps.to_simmap` objects."""
    return RObject(list(simmaps), {"class": ["multiSimmap", "multiPhylo"]})

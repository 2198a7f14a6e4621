"""Host-side mirror of the reference's R-facing API (same function names, argument order and return layout),
calling the B200 library through its C ABI.

    R/sumstatMCMC.R:21          sumstatMCMC(z, Q, pid, Omega, N)
    R/SPARSEsumstatMCMC.R:21    SPARSEsumstatMCMC(z, Q, pid, Omega, N)
    R/sumstatMCMC_bigtree.R:21  sumstatMCMC_bigtree(z, Q, pid, Omega, N)
    R/sumstatMCMCbf.R:21        sumstatMCMCbf(z, Q, pid, Omega, N, prior)      -> named columns, ss[,1:9]
    R/sumstatMCMCks.R:21        sumstatMCMCks(z, Q, pid, Omega, N, prior)
    R/sumstatMCMCmt.R:21        sumstatMCMCmt(treelist, Q, pid, Omega, N, prior)
    R/sumstatMCMCksmt.R:21      sumstatMCMCksmt(treelist, Q, pid, Omega, N, prior)
    R/sumstatEXP.R:21           sumstatEXP(z, Q, pid, N)                           -> independent samples
    R/sumstatMCMC2sDICt.R       sumstatMCMC2sDICt(z, Q, pid, Omega, N, prior)      -> bf columns + log p(y|Q)
    R/sumstatMCMCksDICt.R       sumstatMCMCksDICt(z, Q, pid, Omega, N, prior)      -> ks columns + log p(y|Q)
    R/RcppExports.R:4-50        maketreelist*(x, Q, pid, B, Omega, nen, nodelist, root, N[, prior])

Like the reference, the rate-updating samplers rewrite `Q` (and `B` in the maketreelist* forms) IN PLACE; pass
Fortran-ordered float64 arrays to observe that (other arrays are copied and the caller's object is left alone,
which is what R does for non-double input).  Extra keyword-only arguments (`n_gpu` sharding aside) select the
device arithmetic; their defaults come from PHYLOMAP_B200_{PRECISION,MODE,SEED,DEVICE} so that the positional
signatures stay those of the R functions.
"""
import ctypes as C
import os

import numpy as np

from . import capi
from .simmap import StochasticMaps
from .tree import PhyloTree

BF_COLNAMES = ["time_0", "time_1", "n00", "n01", "n10", "n11", "l01", "l10", "root_state"]
MT_COLNAMES = ["time_0", "time_1", "n00", "n01", "n10", "n11", "l01", "l10", "tree_number"]


def _options(precision=None, mode=None, seed=None, device=None, rng=None, table=None, host_table=None,
             site_offset=0, path_capacity=0, power_capacity=0, allreduce=None, stream=None, progress=False, nccl=None):
    o = capi.default_options()
    env = os.environ
    precision = precision if precision is not None else env.get("PHYLOMAP_B200_PRECISION", "f64")
    mode = mode if mode is not None else env.get("PHYLOMAP_B200_MODE", "production")
    o.precision = {"f64": capi.PM_F64, "f32": capi.PM_F32}[str(precision).lower()]
    o.mode = {"production": capi.PM_MODE_PRODUCTION, "deterministic": capi.PM_MODE_DETERMINISTIC}[str(mode).lower()]
    o.seed = int(seed if seed is not None else env.get("PHYLOMAP_B200_SEED", "1"))
    o.device = int(device if device is not None else env.get("PHYLOMAP_B200_DEVICE", "0"))
    o.site_offset = int(site_offset)
    o.path_capacity, o.power_capacity = int(path_capacity), int(power_capacity)
    o.progress = int(bool(progress))
    keep = []
    if table is not None:
        off = np.ascontiguousarray(table[0], dtype=np.int64)
        u = np.ascontiguousarray(table[1], dtype=np.float64)
        keep += [off, u]
        o.rng, o.tab_off, o.tab_u = capi.PM_RNG_TABLE, capi.ptr(off), capi.ptr(u)
        if host_table is not None:
            ht = np.ascontiguousarray(host_table, dtype=np.float64)
            keep.append(ht)
            o.host_tab, o.host_tab_n = capi.ptr(ht), len(ht)
    if allreduce is not None:
        cb = capi.ALLREDUCE_FN(allreduce)
        keep.append(cb)
        o.allreduce = cb
    if stream is not None:
        o.cuda_stream = int(stream)
    if nccl is not None:   # (unique id bytes, rank, world): the library joins the clique and all-reduces itself
        uid, rank, world = nccl
        buf = np.frombuffer(bytes(uid), dtype=np.uint8).copy()
        assert buf.size == 128
        keep.append(buf)
        o.nccl_id, o.nccl_rank, o.nccl_world = capi.ptr(buf), int(rank), int(world)
    return o, keep


def _inplace(a, n):
    """float64 Fortran-ordered n x n view of `a` if it already is one (so in-place updates are visible), else a copy."""
    if isinstance(a, np.ndarray) and a.dtype == np.float64 and a.shape == (n, n) and (a.flags.f_contiguous):
        return a
    return np.asfortranarray(np.array(a, dtype=np.float64))


def _trees(x):
    if isinstance(x, (list, tuple)):
        return [PhyloTree.from_mapping(t) for t in x]
    return [PhyloTree.from_mapping(x)]


class Chain:
    """Resident chain (pm_chain_*): what the one-call entries are built from; used by bench.py and the tests."""

    def __init__(self, variant, x, Q, pid, Omega, N, prior=None, B=None, order=None, **opts):
        L = capi.lib()
        trees = _trees(x)
        n = np.asarray(Q).shape[0]
        self.n, self.N, self.variant = n, int(N), variant
        self.Q = _inplace(Q, n)
        self.B = _inplace(np.eye(n) + self.Q / Omega if B is None else B, n)
        self.pid = np.ascontiguousarray(pid, dtype=np.float64)
        self.prior = None if prior is None else np.ascontiguousarray(prior, dtype=np.float64)
        self._keep = []
        arr = (capi.PmTree * len(trees))()
        for i, t in enumerate(trees):
            o = order[i] if order is not None else (None, None, None)
            arr[i], keep = t.flat(*o)
            self._keep.append(keep)
        self.trees = trees
        self.opt, keep = _options(**opts)
        self._keep.append(keep)
        self.ncols = L.pm_ncols(variant, n)
        h = C.c_void_p()
        err = C.create_string_buffer(512)
        rc = L.pm_chain_create(variant, C.byref(arr), len(trees), n, capi.ptr(self.Q), capi.ptr(self.pid),
                               capi.ptr(self.B), float(Omega), capi.ptr(self.prior),
                               0 if self.prior is None else len(self.prior), self.N, C.byref(self.opt), C.byref(h),
                               err, 512)
        capi.check(rc, err)
        self.h = h
        self.done = 0

    def run(self, count=None, out=None):
        count = self.N - self.done if count is None else count
        if out is None:
            out = np.zeros((count, self.ncols), dtype=np.float64, order="F")
        err = C.create_string_buffer(512)
        rc = capi.lib().pm_chain_run(self.h, count, capi.ptr(out), out.shape[0], err, 512)
        capi.check(rc, err)
        self.done += count
        return out

    def export_state(self):
        """Checkpoint: the chain state as a byte array (pm_chain_export_state)."""
        L = capi.lib()
        buf = np.empty(int(L.pm_chain_state_bytes(self.h)), dtype=np.uint8)
        err = C.create_string_buffer(512)
        capi.check(L.pm_chain_export_state(self.h, capi.ptr(buf), buf.size, err, 512), err)
        return buf

    def import_state(self, buf):
        """Resume from `export_state()` of a chain created with the same arguments; Q and B are restored in place."""
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        err = C.create_string_buffer(512)
        capi.check(capi.lib().pm_chain_import_state(self.h, capi.ptr(buf), buf.size, err, 512), err)
        self.done = int(np.frombuffer(buf[:64].tobytes(), dtype=np.int32)[9])  # StateHeader.iters_done

    def time_prune(self, reps=10, tree=0):
        ms = C.c_float(0)
        err = C.create_string_buffer(512)
        capi.check(capi.lib().pm_chain_time_prune(self.h, tree, reps, C.byref(ms), err, 512), err)
        return float(ms.value)

    def enable_timing(self, on=True):
        capi.lib().pm_chain_enable_timing(self.h, int(on))

    def kernel_times(self):
        ms = (C.c_double * 4)()
        n = C.c_int64(0)
        capi.lib().pm_chain_kernel_times(self.h, ms, C.byref(n))
        return {"prune": ms[0], "sample_nodes": ms[1], "resample_paths": ms[2], "reduce": ms[3]}, int(n.value)

    def overheads(self):
        """(all-reduce device ms, host rate-update ms) accumulated while timing was enabled (rate-updating samplers)."""
        ms = (C.c_double * 2)()
        capi.lib().pm_chain_overheads(self.h, ms)
        return float(ms[0]), float(ms[1])

    def device_bytes(self):
        return int(capi.lib().pm_chain_device_bytes(self.h))

    def acceptance(self):
        """(proposed, accepted) per rate parameter in trace-column order (l01, l10, kappa->, kappa<-, gamma)."""
        prop = np.zeros(64, dtype=np.int64)
        acc = np.zeros(64, dtype=np.int64)
        k = capi.lib().pm_chain_acceptance(self.h, capi.ptr(prop), capi.ptr(acc), 64)
        return prop[:k].copy(), acc[:k].copy()

    def node_states(self, tree=0):
        t = self.trees[tree]
        out = np.zeros((t.n_sites(), 2 * t.T - 1), dtype=np.int32)
        rc = capi.lib().pm_chain_get_node_states(self.h, tree, capi.ptr(out))
        if rc:
            raise capi.PhylomapError(rc, "get_node_states")
        return out

    def piece_counts(self, tree=0):
        t = self.trees[tree]
        out = np.zeros((t.n_sites(), t.E), dtype=np.int32)
        rc = capi.lib().pm_chain_get_piece_counts(self.h, tree, capi.ptr(out))
        if rc:
            raise capi.PhylomapError(rc, "get_piece_counts")
        return out

    def path(self, site, e, tree=0, cap=256):
        ln = np.zeros(cap)
        st = np.zeros(cap, dtype=np.int32)
        k = capi.lib().pm_chain_get_path(self.h, tree, site, e, capi.ptr(ln), capi.ptr(st), cap)
        if k < 0:
            raise capi.PhylomapError(-k, "get_path")
        return ln[:k].copy(), st[:k].copy()

    def maps(self, sites=None, tree=0):
        """Stochastic maps of the current state (pm_chain_get_maps): the history every selected site holds on every branch of
        tree `tree` after the last sweep, decoded on the device, as a `simmap.StochasticMaps`.  `sites` are LOCAL site
        indices (default: all); under site sharding the global index is `site_offset` + local.  Repeated and unsorted
        indices are allowed.  Does not modify the chain."""
        L = capi.lib()
        t = self.trees[tree]
        sel = np.arange(t.n_sites(), dtype=np.int64) if sites is None else np.ascontiguousarray(sites, dtype=np.int64).reshape(-1)
        off = np.zeros(len(sel) * t.E + 1, dtype=np.int64)
        err = C.create_string_buffer(512)
        capi.check(L.pm_chain_get_maps(self.h, tree, capi.ptr(sel), len(sel), capi.ptr(off), None, None, 0, err, 512), err)
        total = int(off[-1])
        length = np.empty(total, dtype=np.float64)
        state = np.empty(total, dtype=np.int32)
        capi.check(L.pm_chain_get_maps(self.h, tree, capi.ptr(sel), len(sel), capi.ptr(off), capi.ptr(length), capi.ptr(state),
                                       total, err, 512), err)
        return StochasticMaps(sel, off, length, state, self.n, t)

    def sample_maps(self, count, every, sites=None, tree=0):
        """Run `count` sweeps in blocks of `every` and export the maps after each block: (rows, [StochasticMaps, ...]).  The
        rows are those one run(count) returns (device uniforms are keyed by sweep index, so a chain resumes bit for bit)."""
        if every < 1:
            raise ValueError("every must be >= 1")
        rows, maps = [], []
        done = 0
        while done < count:
            k = min(every, count - done)
            rows.append(self.run(k))
            maps.append(self.maps(sites, tree))
            done += k
        out = np.concatenate(rows, axis=0) if rows else np.zeros((0, self.ncols))
        return np.asfortranarray(out), maps

    def partials(self, site=0, tree=0):
        t = self.trees[tree]
        out = np.zeros((2 * t.T - 1, self.n))
        rc = capi.lib().pm_chain_get_partials(self.h, tree, site, capi.ptr(out))
        if rc:
            raise capi.PhylomapError(rc, "get_partials")
        return out

    def close(self):
        if getattr(self, "h", None):
            capi.lib().pm_chain_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_ENTRY = {capi.PM_V_PLAIN: "pm_maketreelistMCMC", capi.PM_V_SPARSE: "pm_SPARSEmaketreelistMCMC",
          capi.PM_V_BIGTREE: "pm_maketreelistMCMC_bigtree", capi.PM_V_BF: "pm_maketreelistMCMCbf",
          capi.PM_V_KS: "pm_maketreelistMCMCks", capi.PM_V_MT: "pm_maketreelistMCMCmt",
          capi.PM_V_KSMT: "pm_maketreelistMCMCksmt", capi.PM_V_DIC2S: "pm_maketreelistMCMC2sDICt",
          capi.PM_V_DICKS: "pm_maketreelistMCMCksDICt"}


def _call(variant, x, Q, pid, B, Omega, order, N, prior=None, **opts):
    """One blocking call of the C-ABI entry that replaces the reference's `.Call('phylomap_<fn>', ...)`."""
    L = capi.lib()
    trees = _trees(x)
    n = np.asarray(Q).shape[0]
    Qf, Bf = _inplace(Q, n), _inplace(B, n)
    pidc = np.ascontiguousarray(pid, dtype=np.float64)
    arr = (capi.PmTree * len(trees))()
    keep = []
    for i, t in enumerate(trees):
        arr[i], k = t.flat(*order[i])
        keep.append(k)
    opt, k2 = _options(**opts)
    ncols = L.pm_ncols(variant, n)
    out = np.zeros((int(N), ncols), dtype=np.float64, order="F")
    err = C.create_string_buffer(512)
    fn = getattr(L, _ENTRY[variant])
    if variant in (capi.PM_V_PLAIN, capi.PM_V_SPARSE, capi.PM_V_BIGTREE):
        rc = fn(C.byref(arr), n, capi.ptr(Qf), capi.ptr(pidc), capi.ptr(Bf), float(Omega), int(N), C.byref(opt),
                capi.ptr(out), err, 512)
    else:
        pr = np.ascontiguousarray(prior, dtype=np.float64)
        if variant in (capi.PM_V_BF, capi.PM_V_KS, capi.PM_V_DIC2S, capi.PM_V_DICKS):
            rc = fn(C.byref(arr), n, capi.ptr(Qf), capi.ptr(pidc), capi.ptr(Bf), float(Omega), int(N), capi.ptr(pr),
                    len(pr), C.byref(opt), capi.ptr(out), err, 512)
        else:
            rc = fn(C.byref(arr), len(trees), n, capi.ptr(Qf), capi.ptr(pidc), capi.ptr(Bf), float(Omega), int(N),
                    capi.ptr(pr), len(pr), C.byref(opt), capi.ptr(out), err, 512)
    capi.check(rc, err)
    return out


# ---- R/RcppExports.R:4-50 -------------------------------------------------------------------------------------
def maketreelistMCMC(x, Q, pid, B, Omega, nen, nodelist, root, N, **opts):
    return _call(capi.PM_V_PLAIN, x, Q, pid, B, Omega, [(nen, nodelist, root)], N, **opts)


def SPARSEmaketreelistMCMC(x, Q, pid, B, Omega, nen, nodelist, root, N, **opts):
    return _call(capi.PM_V_SPARSE, x, Q, pid, B, Omega, [(nen, nodelist, root)], N, **opts)


def maketreelistMCMC_bigtree(x, Q, pid, B, Omega, nen, nodelist, root, N, **opts):
    return _call(capi.PM_V_BIGTREE, x, Q, pid, B, Omega, [(nen, nodelist, root)], N, **opts)


def maketreelistMCMCbf(x, Q, pid, B, Omega, nen, nodelist, root, N, prior, **opts):
    return _call(capi.PM_V_BF, x, Q, pid, B, Omega, [(nen, nodelist, root)], N, prior, **opts)


def maketreelistMCMCks(x, Q, pid, B, Omega, nen, nodelist, root, N, prior, **opts):
    return _call(capi.PM_V_KS, x, Q, pid, B, Omega, [(nen, nodelist, root)], N, prior, **opts)


def maketreelistEXP(x, Q, pid, nen, nodelist, root, N, lefts, rights, d, **opts):
    """R/RcppExports.R: maketreelistEXP(x, Q, pid, nen, nodelist, root, N, lefts, rights, d) -> src/phylomap.cpp:3001."""
    L = capi.lib()
    t = PhyloTree.from_mapping(x)
    n = np.asarray(Q).shape[0]
    Qf = _inplace(Q, n)
    pidc = np.ascontiguousarray(pid, dtype=np.float64)
    lf, rf, df = [np.asfortranarray(np.array(m, dtype=np.float64)) for m in (lefts, rights, d)]
    arr = (capi.PmTree * 1)()
    arr[0], keep = t.flat(nen, nodelist, root)
    opts.setdefault("precision", "f64")
    opt, k2 = _options(**opts)
    out = np.zeros((int(N), L.pm_ncols(capi.PM_V_EXP, n)), dtype=np.float64, order="F")
    err = C.create_string_buffer(512)
    rc = L.pm_maketreelistEXP(C.byref(arr), n, capi.ptr(Qf), capi.ptr(pidc), int(N), capi.ptr(lf), capi.ptr(rf), capi.ptr(df),
                              C.byref(opt), capi.ptr(out), err, 512)
    capi.check(rc, err)
    return out


def maketreelistMCMC2sDICt(x, Q, pid, B, Omega, nen, nodelist, root, N, prior, **opts):
    return _call(capi.PM_V_DIC2S, x, Q, pid, B, Omega, [(nen, nodelist, root)], N, prior, **opts)


def maketreelistMCMCksDICt(x, Q, pid, B, Omega, nen, nodelist, root, N, prior, **opts):
    return _call(capi.PM_V_DICKS, x, Q, pid, B, Omega, [(nen, nodelist, root)], N, prior, **opts)


def maketreelistMCMCmt(x, Q, pid, B, Omega, nen, nodelist_m, roots, N, prior, **opts):
    order = [(np.asarray(nen)[i], np.asarray(nodelist_m)[i], int(roots[i])) for i in range(len(x))]
    return _call(capi.PM_V_MT, x, Q, pid, B, Omega, order, N, prior, **opts)


def maketreelistMCMCksmt(x, Q, pid, B, Omega, nen, nodelist_m, roots, N, prior, **opts):
    order = [(np.asarray(nen)[i], np.asarray(nodelist_m)[i], int(roots[i])) for i in range(len(x))]
    return _call(capi.PM_V_KSMT, x, Q, pid, B, Omega, order, N, prior, **opts)


# ---- R/sumstatMCMC.R:1-18 -------------------------------------------------------------------------------------
def pruningwiseedgeorder(x):
    return PhyloTree.from_mapping(x).order()[0]


def makenodelist(x):
    return PhyloTree.from_mapping(x).order()[1]


def myreorder(x):
    return PhyloTree.from_mapping(x).order()[2]


# ---- the sumstat* wrappers ------------------------------------------------------------------------------------
def _single(fn, z, Q, pid, Omega, N, prior=None, **opts):
    z = PhyloTree.from_mapping(z)
    nen, nodelist, root = z.order()
    n = np.asarray(Q).shape[0]
    B = np.asfortranarray(np.eye(n) + np.asarray(Q, dtype=np.float64) / Omega)
    if prior is None:
        return fn(z, Q, pid, B, Omega, nen, nodelist, root, N, **opts)
    return fn(z, Q, pid, B, Omega, nen, nodelist, root, N, prior, **opts)


def sumstatMCMC(z, Q, pid, Omega, N, **opts):
    return _single(maketreelistMCMC, z, Q, pid, Omega, N, **opts)


def SPARSEsumstatMCMC(z, Q, pid, Omega, N, **opts):
    return _single(SPARSEmaketreelistMCMC, z, Q, pid, Omega, N, **opts)


def sumstatMCMC_bigtree(z, Q, pid, Omega, N, **opts):
    return _single(maketreelistMCMC_bigtree, z, Q, pid, Omega, N, **opts)


def sumstatMCMCbf(z, Q, pid, Omega, N, prior, **opts):
    ss = _single(maketreelistMCMCbf, z, Q, pid, Omega, N, prior, **opts)
    return ss[:, 0:9]  # R/sumstatMCMCbf.R:33-34 names the columns BF_COLNAMES and returns ss[,1:9]


def sumstatMCMCks(z, Q, pid, Omega, N, prior, **opts):
    return _single(maketreelistMCMCks, z, Q, pid, Omega, N, prior, **opts)


def sumstatEXP(z, Q, pid, N, **opts):
    """R/sumstatEXP.R:21-33: eigendecompose Q (eigen / solve), then maketreelistEXP."""
    z = PhyloTree.from_mapping(z)
    nen, nodelist, root = z.order()
    w, V = np.linalg.eig(np.asarray(Q, dtype=np.float64))
    if np.iscomplexobj(w) and np.abs(w.imag).max() > 1e-12 * max(1.0, np.abs(w).max()):
        # R's eigen() would hand complex matrices to maketreelistEXP, whose NumericMatrix arguments reject them
        raise ValueError("sumstatEXP needs a generator with real eigenvalues (the reference passes eigen(Q) as real matrices)")
    return maketreelistEXP(z, Q, pid, nen, nodelist, root, N, V.real, np.linalg.inv(V).real, np.diag(w.real), **opts)


def sumstatMCMC2sDICt(z, Q, pid, Omega, N, prior, **opts):
    """R/sumstatMCMC2sDICt.R: the bf chain plus log p(y|Q) in the last column."""
    return _single(maketreelistMCMC2sDICt, z, Q, pid, Omega, N, prior, **opts)


def sumstatMCMCksDICt(z, Q, pid, Omega, N, prior, **opts):
    """R/sumstatMCMCksDICt.R: the ks chain plus log p(y|Q) in the last column."""
    return _single(maketreelistMCMCksDICt, z, Q, pid, Omega, N, prior, **opts)


def colnames(fn, n=None):
    """Column names of a sampler's result, where the reference assigns any: `sumstatMCMCbf` (R/sumstatMCMCbf.R:33),
    `sumstatMCMCmt` (R/sumstatMCMCmt.R:39) and the two DIC traces as make_12_chains labels them (R/sourceme.R:532, 547) --
    the names `make2stateDIC` / `make4stateDIC` index by.  `fn` is the function or its name; n the number of states."""
    name = fn if isinstance(fn, str) else fn.__name__
    name = name.replace("maketreelist", "sumstat")
    two = ["n00", "n01", "n10", "n11", "l01", "l10"]
    if name == "sumstatMCMCbf":
        return ["time 0", "time 1"] + two + ["root_state"]
    if name == "sumstatMCMCmt":
        return ["time_0", "time_1"] + two + ["tree_number"]
    if name == "sumstatMCMC2sDICt":
        return ["t0", "t1"] + two + ["root_state", "log(p(y|Q))"]
    if name == "sumstatMCMCksDICt":
        n = 4 if n is None else n
        k = n // 2 - 1
        rates = ["l01", "l10"] + (["k01", "k10", "gamma"] if k == 1 else ["k01_%d" % i for i in range(1, k + 1)] +
                                  ["k10_%d" % i for i in range(1, k + 1)] + ["gamma_%d" % i for i in range(1, k + 1)])
        return ["t%d" % i for i in range(1, n + 1)] + ["n%d%d" % (a, b) for a in range(1, n + 1) for b in range(1, n + 1)] + \
            rates + ["root_state", "log(p(y|Q))"]
    raise KeyError("the reference names no columns for %s" % name)


def loglik(z, Q, pid, parity_tips=False, order=None, **opts):
    """log p(y | Q) summed over the sites of `z` (pm_loglik): pruning with exp(Q t_e) on the GPU."""
    L = capi.lib()
    z = PhyloTree.from_mapping(z)
    n = np.asarray(Q).shape[0]
    Qf = np.asfortranarray(np.asarray(Q, dtype=np.float64))
    pidc = np.ascontiguousarray(pid, dtype=np.float64)
    tree, keep = z.flat(*(order if order is not None else (None, None, None)))
    opt, keep2 = _options(**opts)
    out = C.c_double(0.0)
    err = C.create_string_buffer(512)
    rc = L.pm_loglik(C.byref(tree), n, capi.ptr(Qf), capi.ptr(pidc), int(bool(parity_tips)), C.byref(opt), C.byref(out), err, 512)
    capi.check(rc, err)
    return float(out.value)


class ExpectedSumstats:
    """Exact posterior expectations under a fixed Q (`expected_sumstats`).  Columns of a statistic follow the fixed-Q
    sampler rows: n dwell times, then the n(n-1) changes i -> j, row-major with the diagonal skipped.
        stats           [S, n^2]           per site
        loglik          [S]                log p(y_s | Q)
        sites           [k]                the selected local sites
        branch_stats    [k, E, n^2]        per selected site and branch (edge-row order)
        node_marginals  [k, 2T-1, n]       P(X_v = s | y), 0-based node ids (tips 0..T-1)"""

    def __init__(self, n, stats, loglik, sites, branch_stats, node_marginals):
        self.n, self.stats, self.loglik, self.sites = n, stats, loglik, sites
        self.branch_stats, self.node_marginals = branch_stats, node_marginals

    def mapped_edge(self):
        """[k, E, n]: expected time in each state on each branch (the mean of `StochasticMaps.mapped_edge()`)."""
        return self.branch_stats[:, :, :self.n]

    def transitions(self):
        """[k, n, n]: expected number of changes a -> b summed over the branches (the mean of `StochasticMaps.transitions()`)."""
        n = self.n
        tot = self.branch_stats[:, :, n:].sum(axis=1)
        out = np.zeros((len(self.sites), n, n))
        off = np.ones((n, n), dtype=bool)
        np.fill_diagonal(off, False)
        out[:, off] = tot
        return out


def expected_sumstats(z, Q, pid, parity_tips=False, sites=None, order=None, **opts):
    """Exact posterior expected dwell times and transition counts of every site of `z` given its tip data under a fixed Q,
    and log p(y_s | Q) per site (pm_expected_sumstats): no sampling.  For the local `sites` (repeats and any order allowed)
    also per branch and the marginal state probabilities of every node.  Returns an `ExpectedSumstats`."""
    L = capi.lib()
    z = PhyloTree.from_mapping(z)
    n = np.asarray(Q).shape[0]
    Qf = np.asfortranarray(np.asarray(Q, dtype=np.float64))
    pidc = np.ascontiguousarray(pid, dtype=np.float64)
    tree, keep = z.flat(*(order if order is not None else (None, None, None)))
    opt, keep2 = _options(**opts)
    S, E, NK = z.n_sites(), z.E, n * n
    sel = np.zeros(0, dtype=np.int64) if sites is None else np.ascontiguousarray(sites, dtype=np.int64).reshape(-1)
    stats = np.zeros((S, NK), dtype=np.float64, order="F")
    ll = np.zeros(S, dtype=np.float64)
    bs = np.zeros((len(sel), E, NK), dtype=np.float64)
    nm = np.zeros((len(sel), 2 * z.T - 1, n), dtype=np.float64)
    err = C.create_string_buffer(512)
    rc = L.pm_expected_sumstats(C.byref(tree), n, capi.ptr(Qf), capi.ptr(pidc), int(bool(parity_tips)), capi.ptr(sel), len(sel),
                                C.byref(opt), capi.ptr(stats), capi.ptr(ll), capi.ptr(bs) if len(sel) else None,
                                capi.ptr(nm) if len(sel) else None, err, 512)
    capi.check(rc, err)
    return ExpectedSumstats(n, stats, ll, sel, bs, nm)


def _col(mat, name, pos):
    """Column of a sampler output by the reference's name (a pandas frame) or by its position (a plain matrix)."""
    if hasattr(mat, "columns"):
        return np.asarray(mat[name], dtype=np.float64)
    if hasattr(mat, "attributes") and hasattr(mat, "value"):  # rds.RObject: a matrix read back with its dimnames
        names = (mat.attributes.get("dimnames") or [None, None])[1]
        a = np.asarray(mat.value, dtype=np.float64)
        return a[:, list(names).index(name)] if names else a[:, pos]
    return np.asarray(mat, dtype=np.float64)[:, pos]


def _dic(mat, D):
    ll = _col(mat, "log(p(y|Q))", -1)
    pD = np.mean(-2.0 * ll) - D            # R/sourceme.R:169-173
    return D + 2.0 * pD


def make2stateDIC(mat, atree, pid, **opts):
    """R/sourceme.R:141-177: DIC of the 2-state model from a sumstatMCMC2sDICt trace: D(Q-hat) at the posterior-mean
    rates (columns l01, l10 = 6, 7) plus 2 pD with pD = mean(-2 log p(y|Q)) - D(Q-hat)."""
    l01, l10 = _col(mat, "l01", 6).mean(), _col(mat, "l10", 7).mean()
    Q = np.array([[-l01, l01], [l10, -l10]])
    return _dic(mat, -2.0 * loglik(atree, Q, pid, parity_tips=False, **opts))


def make4stateDIC(mat, atree, pid, **opts):
    """R/sourceme.R:248-284: the same for the hidden-rate model from a sumstatMCMCksDICt trace (columns l01, l10, k01,
    k10, gamma = 20..24); tips enter as (1,0,1,0) / (0,1,0,1)."""
    from .synth import make2sQ
    r = [_col(mat, nm, 20 + i).mean() for i, nm in enumerate(("l01", "l10", "k01", "k10", "gamma"))]
    return _dic(mat, -2.0 * loglik(atree, make2sQ(*r), pid, parity_tips=True, **opts))


def make2stateDICbig(mat, atree, pid, ne=None, **opts):
    """R/sourceme.R:445-474: the rescaled ("big tree") form; the GPU pruning always rescales, so this is make2stateDIC
    with the caller's pruning-wise edge order."""
    return make2stateDIC(mat, atree, pid, **opts)


def make4stateDICbig(mat, atree, pid, ne=None, **opts):
    """R/sourceme.R:476-516."""
    return make4stateDIC(mat, atree, pid, **opts)


def _multi(fn, treelist, Q, pid, Omega, N, prior, **opts):
    trees = _trees(treelist)
    orders = [t.order() for t in trees]
    nen_m = np.stack([o[0] for o in orders])
    nodelist_m = np.stack([o[1] for o in orders])
    roots = [o[2] for o in orders]
    n = np.asarray(Q).shape[0]
    B = np.asfortranarray(np.eye(n) + np.asarray(Q, dtype=np.float64) / Omega)
    return fn(trees, Q, pid, B, Omega, nen_m, nodelist_m, roots, N, prior, **opts)


def sumstatMCMCmt(treelist, Q, pid, Omega, N, prior, **opts):
    return _multi(maketreelistMCMCmt, treelist, Q, pid, Omega, N, prior, **opts)


def sumstatMCMCksmt(treelist, Q, pid, Omega, N, prior, **opts):
    return _multi(maketreelistMCMCksmt, treelist, Q, pid, Omega, N, prior, **opts)

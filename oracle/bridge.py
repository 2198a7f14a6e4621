"""TEST INFRASTRUCTURE ONLY: ctypes bridge to the CPU oracle (oracle/libphylomap_oracle.so).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this module.
The product package (phylomap_b200) never does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

PLAIN, SPARSE, BIGTREE, BF, KS, MT, KSMT, EXP, DIC2S, DICKS = range(10)
SEQUENTIAL, KEYED, TABLE = range(3)


class _Tree(C.Structure):
    _fields_ = [("T", C.c_int32), ("E", C.c_int32), ("edge", C.c_void_p), ("nen", C.c_void_p),
                ("nodelist", C.c_void_p), ("root", C.c_int32), ("maps_off", C.c_void_p),
                ("maps_len", C.c_void_p), ("maps_state", C.c_void_p), ("states", C.c_void_p),
                ("S", C.c_int64), ("edge_length", C.c_void_p)]


class _Config(C.Structure):
    _fields_ = [("variant", C.c_int32), ("n", C.c_int32), ("N", C.c_int32), ("ntrees", C.c_int32),
                ("Omega", C.c_double), ("prior", C.c_void_p), ("nprior", C.c_int32),
                ("rng_mode", C.c_int32), ("seed", C.c_uint64), ("want_log", C.c_int32),
                ("tab_off", C.c_void_p), ("tab_u", C.c_void_p), ("host_tab", C.c_void_p),
                ("host_tab_n", C.c_int64), ("lefts", C.c_void_p), ("rights", C.c_void_p), ("d", C.c_void_p),
                ("site_offset", C.c_int64)]


def build(force=False):
    so = os.path.join(_HERE, "libphylomap_oracle.so")
    srcs = [os.path.join(_HERE, f) for f in ("phylomap_oracle.cpp", "r_rng.hpp")]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return so


def lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(_HERE, "libphylomap_oracle.so")
        if not os.path.exists(so):
            build()
        L = C.CDLL(so)
        L.orc_create.restype = C.c_void_p
        L.orc_create.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_char_p, C.c_int]
        L.orc_run.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_int]
        L.orc_ncols.argtypes = [C.c_void_p]
        L.orc_destroy.argtypes = [C.c_void_p]
        L.orc_set_fast_lookup.argtypes = [C.c_void_p, C.c_int]
        L.orc_get_node_states.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.orc_get_piece_counts.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.orc_get_path.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        L.orc_get_pieces.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        L.orc_get_pl.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p]
        for f in ("orc_log_nslots", "orc_log_total", "orc_hostlog_n"):
            getattr(L, f).restype = C.c_int64
            getattr(L, f).argtypes = [C.c_void_p]
        L.orc_log_export.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_hostlog_export.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_rng_probe.argtypes = [C.c_uint32, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p]
        L.orc_philox.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_keyed_uniform.restype = C.c_double
        L.orc_keyed_uniform.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
        L.orc_sample.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_char_p, C.c_int]
        _LIB = L
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


_REF = None


def ref_path():
    return os.path.join(_HERE, "_ref", "libphylomap_ref.so")


def ref_lib():
    """oracle/_ref/libphylomap_ref.so: the UNMODIFIED reference sources (src/phylomap.cpp + RcppExports.cpp) compiled
    against the stand-in headers of oracle/standin/ (oracle/Makefile, target `ref`).  Built here when /root/reference
    exists; on the GPU box the prebuilt file travels with the repo.  Returns None when neither is available."""
    global _REF
    if _REF is None:
        so = ref_path()
        if os.path.exists("/root/reference/src/phylomap.cpp"):
            subprocess.check_call(["make", "-C", _HERE, "-s", "ref"])
        if not os.path.exists(so):
            return None
        L = C.CDLL(so)
        L.ref_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_char_p, C.c_int]
        L.ref_ncols.argtypes = [C.c_int, C.c_int]
        L.ref_rng_probe.argtypes = [C.c_uint32, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p]
        _REF = L
    return _REF


def _pack_trees(trees, keep):
    arr = (_Tree * len(trees))()
    for i, t in enumerate(trees):
        edge = np.asfortranarray(t["edge"], dtype=np.int32)
        nen = np.ascontiguousarray(t["nen"], dtype=np.int32)
        nodelist = np.ascontiguousarray(t["nodelist"], dtype=np.int32)
        mo = np.ascontiguousarray(t["maps_off"], dtype=np.int64)
        ml = np.ascontiguousarray(t["maps_len"], dtype=np.float64)
        ms = np.ascontiguousarray(t["maps_state"], dtype=np.int32)
        st = np.ascontiguousarray(t["states"], dtype=np.int32)
        if st.ndim == 1:
            st = st[None, :]
        el = None if t.get("edge_length") is None else np.ascontiguousarray(t["edge_length"], dtype=np.float64)
        keep += [edge, nen, nodelist, mo, ml, ms, st, el]
        arr[i] = _Tree(st.shape[1], edge.shape[0], _p(edge), _p(nen), _p(nodelist), int(t["root"]), _p(mo), _p(ml), _p(ms),
                       _p(st), st.shape[0], _p(el))
    return arr


_SHIM = None


def shim_path():
    return os.path.join(_HERE, "_ref", "libphylomap_shim.so")


def shim_lib():
    """oracle/_ref/libphylomap_shim.so: the package's `.Call` glue (oracle/shim_glue.cpp) + shim/phylomap_b200_shim.cpp
    (the drop-in replacement of src/phylomap.cpp on the product's C ABI) + the same driver, against the stand-in headers
    (oracle/Makefile, target `shim`; make relinks it when a source or libphylomap_b200.so is newer).  The `.Call`
    symbols of the package, served by libphylomap_b200.so.  This is the one place where test infrastructure loads the
    PRODUCT through the reference's boundary; nothing of the oracle restatement is involved."""
    global _SHIM
    if _SHIM is None:
        subprocess.check_call(["make", "-C", _HERE, "-s", "shim"])
        L = C.CDLL(shim_path())
        L.ref_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_char_p, C.c_int]
        L.ref_ncols.argtypes = [C.c_int, C.c_int]
        L.ref_rng_probe.argtypes = [C.c_uint32, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p]
        L.shim_tree_order.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_char_p, C.c_int]
        _SHIM = L
    return _SHIM


def shim_run(variant, trees, Q, pid, Omega, N, prior=None, seed=1, B=None, eig=None):
    """The same call as ref_run, answered by the product through the shim (any number of sites: states become an
    ntips x nsites matrix).  Precision / mode / device come from the PHYLOMAP_B200_* environment like in an R session."""
    return _lib_run(shim_lib(), variant, trees, Q, pid, Omega, N, prior, seed, B, eig)


def shim_seed(seed):
    """The 64-bit seed the shim derives from R's stream after set.seed(seed): two unif_rand() draws (shim/phylomap_b200_shim.cpp)."""
    u = ref_rng_probe(seed, "unif", 2, lib_=shim_lib())
    return (int(u[0] * 4294967296.0) << 32) | int(u[1] * 4294967296.0)


def ref_run(variant, trees, Q, pid, Omega, N, prior=None, seed=1, B=None, eig=None):
    """One call of the reference's own `.Call` entry point for `variant` (phylomap_maketreelistMCMC ... ksDICt) with R's
    generator seeded like set.seed(seed).  One site per tree (the reference has no site axis).  Returns (rows, Q, B):
    Q and B as the call left them (the rate-updating drivers rewrite them in place)."""
    L = ref_lib()
    if L is None:
        raise OracleError("oracle/_ref is not built (no /root/reference here and no prebuilt library)")
    return _lib_run(L, variant, trees, Q, pid, Omega, N, prior, seed, B, eig)


def _lib_run(L, variant, trees, Q, pid, Omega, N, prior, seed, B, eig):
    keep = []
    n = Q.shape[0]
    Qf = np.asfortranarray(np.array(Q, dtype=np.float64))
    Bf = np.asfortranarray(np.eye(n) + Qf / Omega) if B is None else np.asfortranarray(np.array(B, dtype=np.float64))
    pidc = np.ascontiguousarray(pid, dtype=np.float64)
    arr = _pack_trees(trees, keep)
    pr = None if prior is None else np.ascontiguousarray(prior, dtype=np.float64)
    cfg = _Config()
    cfg.variant, cfg.n, cfg.N, cfg.ntrees, cfg.Omega = variant, n, N, len(trees), float(Omega)
    cfg.prior, cfg.nprior = _p(pr), 0 if pr is None else len(pr)
    cfg.rng_mode, cfg.seed = SEQUENTIAL, seed
    if eig is not None:
        lefts, rights, d = [np.asfortranarray(x, dtype=np.float64) for x in eig]
        keep += [lefts, rights, d]
        cfg.lefts, cfg.rights, cfg.d = _p(lefts), _p(rights), _p(d)
    out = np.zeros((N, L.ref_ncols(variant, n)), dtype=np.float64, order="F")
    err = C.create_string_buffer(512)
    rc = L.ref_run(C.byref(arr), C.byref(cfg), _p(Qf), _p(pidc), _p(Bf), _p(out), err, 512)
    if rc:
        raise OracleError(err.value.decode())
    return out, Qf, Bf


def ref_rng_probe(seed, kind, n, a=0.0, b=0.0, lib_=None):
    out = np.zeros(n)
    (lib_ or ref_lib()).ref_rng_probe(seed, {"unif": 0, "exp": 1, "norm": 2, "gamma": 3, "rexp": 4}[kind], n, a, b, _p(out))
    return out


class OracleError(RuntimeError):
    pass


class OracleRun:
    """One oracle chain.  `trees` is a list of dicts with numpy arrays:
    edge [E,2] int32 (1-based), nen [E], nodelist [T-2], root, maps_off [E+1] int64, maps_len, maps_state,
    states [S,T] int32 (1-based), edge_length [E] (EXP only).  Q and B are float64 [n,n]; they are copied to
    column-major buffers (self.Q / self.B) which the bf/ks/mt variants mutate like the reference does."""

    def __init__(self, variant, trees, Q, pid, Omega, N, prior=None, rng_mode=KEYED, seed=1, want_log=False,
                 table=None, host_table=None, B=None, eig=None, site_offset=0):
        L = lib()
        self._keep = []
        n = Q.shape[0]
        self.n, self.N, self.variant = n, N, variant
        self.Q = np.asfortranarray(np.array(Q, dtype=np.float64))
        self.B = np.asfortranarray(np.eye(n) + self.Q / Omega) if B is None else np.asfortranarray(np.array(B, dtype=np.float64))
        self.pid = np.ascontiguousarray(pid, dtype=np.float64)
        arr = (_Tree * len(trees))()
        for i, t in enumerate(trees):
            edge = np.asfortranarray(t["edge"], dtype=np.int32)
            nen = np.ascontiguousarray(t["nen"], dtype=np.int32)
            nodelist = np.ascontiguousarray(t["nodelist"], dtype=np.int32)
            mo = np.ascontiguousarray(t["maps_off"], dtype=np.int64)
            ml = np.ascontiguousarray(t["maps_len"], dtype=np.float64)
            ms = np.ascontiguousarray(t["maps_state"], dtype=np.int32)
            st = np.ascontiguousarray(t["states"], dtype=np.int32)
            if st.ndim == 1:
                st = st[None, :]
            el = None if t.get("edge_length") is None else np.ascontiguousarray(t["edge_length"], dtype=np.float64)
            self._keep += [edge, nen, nodelist, mo, ml, ms, st, el]
            T = st.shape[1]
            arr[i] = _Tree(T, edge.shape[0], _p(edge), _p(nen), _p(nodelist), int(t["root"]), _p(mo), _p(ml), _p(ms),
                           _p(st), st.shape[0], _p(el))
        self._trees = arr
        self.S = [int(a.S) for a in arr]
        self.T = [int(a.T) for a in arr]
        self.E = [int(a.E) for a in arr]
        pr = None if prior is None else np.ascontiguousarray(prior, dtype=np.float64)
        cfg = _Config()
        cfg.variant, cfg.n, cfg.N, cfg.ntrees, cfg.Omega = variant, n, N, len(trees), float(Omega)
        cfg.prior, cfg.nprior = _p(pr), 0 if pr is None else len(pr)
        cfg.rng_mode, cfg.seed, cfg.want_log = rng_mode, seed, int(want_log)
        cfg.site_offset = int(site_offset)
        if table is not None:
            off = np.ascontiguousarray(table[0], dtype=np.int64)
            u = np.ascontiguousarray(table[1], dtype=np.float64)
            self._keep += [off, u]
            cfg.tab_off, cfg.tab_u = _p(off), _p(u)
        if host_table is not None:
            ht = np.ascontiguousarray(host_table, dtype=np.float64)
            self._keep.append(ht)
            cfg.host_tab, cfg.host_tab_n = _p(ht), len(ht)
        if eig is not None:
            lefts, rights, d = [np.asfortranarray(x, dtype=np.float64) for x in eig]
            self._keep += [lefts, rights, d]
            cfg.lefts, cfg.rights, cfg.d = _p(lefts), _p(rights), _p(d)
        self._keep += [pr, cfg]
        err = C.create_string_buffer(512)
        self.h = L.orc_create(C.byref(arr), C.byref(cfg), _p(self.Q), _p(self.pid), _p(self.B), err, 512)
        if not self.h:
            raise OracleError(err.value.decode())
        self.ncols = L.orc_ncols(self.h)

    def set_fast_lookup(self, on=True):
        """bench.py's "optimised CPU" leg: parent-edge table instead of the reference's O(E) search per node (:643)."""
        lib().orc_set_fast_lookup(self.h, int(on))

    def run(self):
        out = np.zeros((self.N, self.ncols), dtype=np.float64, order="F")
        err = C.create_string_buffer(512)
        rc = lib().orc_run(self.h, _p(out), err, 512)
        if rc:
            raise OracleError(err.value.decode())
        return out

    def node_states(self, tree=0):
        out = np.zeros((self.S[tree], 2 * self.T[tree] - 1), dtype=np.int32)
        lib().orc_get_node_states(self.h, tree, _p(out))
        return out

    def piece_counts(self, tree=0):
        out = np.zeros((self.S[tree], self.E[tree]), dtype=np.int32)
        lib().orc_get_piece_counts(self.h, tree, _p(out))
        return out

    def path(self, site, e, tree=0, cap=4096):
        ln = np.zeros(cap)
        st = np.zeros(cap, dtype=np.int32)
        k = lib().orc_get_path(self.h, tree, site, e, _p(ln), _p(st), cap)
        return ln[:k].copy(), st[:k].copy()

    def pieces(self, site, e, tree=0, cap=65536):
        ln = np.zeros(cap)
        st = np.zeros(cap, dtype=np.int32)
        k = lib().orc_get_pieces(self.h, tree, site, e, _p(ln), _p(st), cap)
        return ln[:k].copy(), st[:k].copy()

    def partials(self, site=0, tree=0):
        out = np.zeros((2 * self.T[tree] - 1, self.n))
        lib().orc_get_pl(self.h, tree, site, _p(out))
        return out

    def export_log(self):
        L = lib()
        ns, tot = L.orc_log_nslots(self.h), L.orc_log_total(self.h)
        off = np.zeros(ns + 1, dtype=np.int64)
        u = np.zeros(max(tot, 1), dtype=np.float64)
        L.orc_log_export(self.h, _p(off), _p(u))
        nh = L.orc_hostlog_n(self.h)
        hu = np.zeros(max(nh, 1), dtype=np.float64)
        L.orc_hostlog_export(self.h, _p(hu))
        return (off, u[:tot]), hu[:nh]

    def close(self):
        if self.h:
            lib().orc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def rng_probe(seed, kind, n, a=0.0, b=0.0):
    out = np.zeros(n)
    lib().orc_rng_probe(seed, {"unif": 0, "exp": 1, "norm": 2, "gamma": 3, "rexp": 4}[kind], n, a, b, _p(out))
    return out


def philox(ctr, key):
    c = np.asarray(ctr, dtype=np.uint32)
    k = np.asarray(key, dtype=np.uint32)
    o = np.zeros(4, dtype=np.uint32)
    lib().orc_philox(_p(c), _p(k), _p(o))
    return o


def keyed_uniform(seed, site, it, slot, k):
    return lib().orc_keyed_uniform(seed, site, it, slot, k)


def sample(w, u):
    w = np.ascontiguousarray(w, dtype=np.float64)
    err = C.create_string_buffer(256)
    r = lib().orc_sample(_p(w), len(w), u, err, 256)
    if r < 0:
        raise OracleError(err.value.decode())
    return r

#!/usr/bin/env python
"""Headline benchmark: sampled branch-site histories / second (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

`--dump-outputs DIR` writes the statistics row the last timed sweep returned (dwell times, then transition counts, float64)
to DIR/rows.npy.  The inputs are seeded, so two builds run with the same arguments can be compared output for output.

Workload (config.workload): BASELINE.json configs[3] — sumstatMCMC_bigtree on a 10 000-tip Yule tree, 4-state
hidden-rate model make2sQ(.1,.1,.2,.2,10), 1 000 000 sites site-sharded over 8 GPUs = 125 000 sites per GPU, weak
scaling (every rank always holds 125 000 sites).  One step = one MCMC sweep (prune, node draws, path resampling,
reduction) over all local sites = E x S_local branch-site histories.  Production arithmetic: FP32, Philox.

`value`   : device-timed sweeps on the resident chain (CUDA events on the chain's stream), max over ranks.
`e2e`     : the same sweeps through the drop-in entry pm_maketreelistMCMC_bigtree with HOST buffers: tip states
            uploaded from pinned host memory, chain built, K sweeps, result matrix copied back — all inside the timer.
`roofline`: pruning pass K1 (k_prune) timed alone with CUDA events; algorithmic bytes per site from SURVEY.md §8(d).
`rate_sampler`: sumstatMCMCks (hidden-rate model, Q updated every sweep) on the same tree and sites: ms per sweep, and
            per sweep the device time of the one small NCCL all-reduce and the host time of the replicated rate update --
            the part of the design that has a collective in it (the fixed-Q headline all-reduces once per run).
`one_character`: BASELINE configs[0] (one binary trait, 100 tips, 1 000 sweeps: the reference's literal usage) -- microseconds
            per sweep on the GPU (whole call / resident chain) beside the reference's code and the optimised port on one core.
`cpu_baseline` / `--impl reference`: the reference's own code -- oracle/_ref = the unmodified src/phylomap.cpp compiled
            against stand-in Rcpp / Armadillo headers (R is absent) -- on a bounded site sample, one process per host
            core; beside it the in-repo port in "faithful" mode (keeps the reference's O(E) edge search per node, :643) and in
            "optimised" mode (parent-edge table): the honest CPU context for the GPU number.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TIPS = int(os.environ.get("PM_BENCH_TIPS", 10000))
SITES_PER_GPU = int(os.environ.get("PM_BENCH_SITES", 125000))
OMEGA = 2.4
METRIC = "sampled branch-site histories/sec (4-state, 10k-tip tree)"
UNIT = "histories/s"


def workload_tree():
    from phylomap_b200 import synth
    Q = synth.make2sQ(0.1, 0.1, 0.2, 0.2, 10.0)
    qmax = float(np.max(-np.diag(Q)))
    tree = synth.yule_tree(TIPS, seed=4, mean_branch=0.1 / qmax)
    return tree, Q, np.full(4, 0.25)


def config(n_gpus, sites):
    return {"workload": "sumstatMCMC_bigtree, %d-tip Yule tree (seed 4, mean branch 0.1/max|Qii|), 4-state make2sQ(.1,.1,.2,.2,10), "
                        "Omega=2.4, %d sites per GPU x %d GPU(s), site-sharded" % (TIPS, sites, n_gpus),
            "tips": TIPS, "branches": 2 * TIPS - 2, "states": 4, "sites_per_gpu": sites, "sites_total": sites * n_gpus,
            "precision": "f32", "rng": "philox4x32-10",
            "l2": "per-sweep working set (partials + jump counts, >30 GB at the default size) exceeds the 126 MB L2"}


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run_nvml(self):
        """NVML directly (a sample costs well under a millisecond): the same fields as the nvidia-smi query below."""
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = (0x8, 0x40, 0x20, 0x4)  # hw_slowdown, hw_thermal_slowdown, sw_thermal_slowdown, sw_power_cap
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        while not self.stop.is_set():
            r = int(get_reasons(h))
            self.rows.append([str(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), str(mx)] +
                             ["Active" if r & b else "Not Active" for b in bits])
            self.stop.wait(0.05)

    def _run(self):
        try:
            self._run_nvml()
            return
        except Exception:
            pass
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=3)

    def summary(self):
        sm = [int(r[0]) for r in self.rows if len(r) == 6 and r[0].isdigit()]
        mx = [int(r[1]) for r in self.rows if len(r) == 6 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) == 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": int(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
# CPU legs.  Nothing here touches the product library: the tree order is computed in numpy so that the reference arm's
# process maps no libphylomap_b200.so (the driver checks which native libraries a process loaded).
def tree_order_numpy(edge, T):
    """A valid (nen, nodelist, root) for the reference's samplers (R/sumstatMCMC.R:1-18): nen lists the two child edges of
    every internal node, children before parents; nodelist lists the internal nodes below the root, parents first."""
    E = edge.shape[0]
    kids = {}
    for r in range(E):
        kids.setdefault(int(edge[r, 0]), []).append(r)
    root = (set(kids) - set(int(c) for c in edge[:, 1])).pop()
    nen, nodelist, stack = [], [], [(root, 0)]
    while stack:
        v, k = stack.pop()
        rows = kids[v]
        if k == 0 and v != root:
            nodelist.append(v)
        if k < len(rows):
            stack.append((v, k + 1))
            c = int(edge[rows[k], 1])
            if c > T:
                stack.append((c, 0))
        else:
            nen += [r + 1 for r in rows]
    return np.array(nen, dtype=np.int32), np.array(nodelist, dtype=np.int32), root


def _cpu_worker(args):
    """One process: `kind` on a slice of sites.  Returns (histories, seconds)."""
    kind, tree_d, Q, pid, N, seed = args
    from oracle import bridge
    E, S = tree_d["edge"].shape[0], tree_d["states"].shape[0]
    t0 = time.perf_counter()
    if kind == "reference":   # the reference handles one character per call: one call per site
        for s in range(S):
            d = dict(tree_d)
            d["states"] = tree_d["states"][s:s + 1]
            bridge.ref_run(bridge.BIGTREE, [d], Q, pid, OMEGA, N, seed=seed + s)
    else:
        run = bridge.OracleRun(bridge.BIGTREE, [tree_d], Q, pid, OMEGA, N, rng_mode=bridge.SEQUENTIAL, seed=seed)
        run.set_fast_lookup(kind == "port_optimised")
        run.run()
    return E * S * N, time.perf_counter() - t0


CPU_SITES = {"reference": 3, "port_faithful": 6, "port_optimised": 80}   # sites per core: a few seconds of work each


def cpu_leg(kind, tree, Q, pid, steps, order, sites_per_core=None, cores=None):
    """`kind` on all host cores: sites are independent for fixed Q, so each core gets its own slice -- the most favourable
    way to run the single-threaded reference on this host."""
    import multiprocessing as mp
    from phylomap_b200 import synth
    cores = cores or os.cpu_count() or 1
    spc = sites_per_core or int(os.environ.get("PM_BENCH_CPU_SITES", CPU_SITES[kind]))
    st = synth.simulate_tip_states(tree, Q, pid, cores * spc, seed=99).numpy()
    jobs = []
    for c in range(cores):
        z = tree.with_states(st[c * spc:(c + 1) * spc], segments=2)
        jobs.append((kind, z.oracle_dict(*order), Q.copy(), pid, steps, 1000 + 97 * c))
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(cores) as pool:
        res = pool.map(_cpu_worker, jobs)
    wall = time.perf_counter() - t0
    what = {"reference": "oracle/_ref: the unmodified src/phylomap.cpp (maketreelistMCMC_bigtree) compiled against stand-in Rcpp / Armadillo headers",
            "port_faithful": "in-repo port, keeps the reference's O(E) edge search per node (:643)",
            "port_optimised": "in-repo port with a parent-edge table"}[kind]
    return {"value": sum(r[0] for r in res) / wall, "unit": UNIT, "cores": cores, "kind": "reference" if kind == "reference" else "port",
            "sample": "%s; %d sites x %d cores x %d sweeps of the same tree/model, one process per core, wall %.1f s"
                      % (what, spc, cores, steps, wall)}, wall


def cpu_baseline(tree, Q, pid, steps=6):
    """The reported CPU context: the reference's own code where oracle/_ref exists, and the port in both modes."""
    from oracle import bridge
    bridge.build()
    order = tree_order_numpy(tree.edge, tree.T)
    have_ref = bridge.ref_lib() is not None
    main, _ = cpu_leg("reference" if have_ref else "port_faithful", tree, Q, pid, steps, order)
    for k in ("port_faithful", "port_optimised"):
        leg, _ = cpu_leg(k, tree, Q, pid, steps, order)
        main[k] = {"value": leg["value"], "sample": leg["sample"]}
    return main


def one_character(opts):
    """BASELINE configs[0], the reference's literal usage: ONE binary character on a 100-tip tree, sumstatMCMC, 1 000 sweeps
    (tutorial sec. 2).  GPU: the whole drop-in call with host buffers (chain built, sweeps, result matrix back) and the
    sweeps alone on a chain that already exists -- at this size the library runs a block per site with the site's state in
    shared memory and every sweep of the call inside one launch (pm_small.cuh).  CPU, one core: the reference's own code
    (oracle/_ref) and the in-repo port with a parent-edge table."""
    import torch
    import phylomap_b200 as pb
    from phylomap_b200 import capi, synth
    from oracle import bridge
    Q2, pid2, Om, N = np.array([[-0.1, 0.1], [0.1, -0.1]]), np.array([0.5, 0.5]), 0.2, 1000
    z = synth.simulate_2_state_tree(101, synth.yule_tree(100, seed=1, mean_branch=5.0), Q2, pid2)
    kw = {k: v for k, v in opts.items() if k in ("precision", "device")}

    def best(fn, reps=3):
        fn()
        b = 1e30
        for _ in range(reps):
            torch.cuda.synchronize(); t = time.perf_counter(); fn(); torch.cuda.synchronize()
            b = min(b, time.perf_counter() - t)
        return b
    call = best(lambda: pb.sumstatMCMC(z, Q2, pid2, Om, N, seed=5, **kw))
    ch = pb.Chain(capi.PM_V_PLAIN, z, Q2, pid2, Om, 5 * N, seed=5, **kw)
    res = best(lambda: ch.run(N))
    _, launches = ch.kernel_times()
    ch.close()
    out = {"workload": "BASELINE configs[0]: sumstatMCMC, 100-tip tree, one binary character, Omega = 0.2, 1 000 sweeps",
           "gpu_us_per_sweep_whole_call": 1e6 * call / N, "gpu_us_per_sweep_resident_chain": 1e6 * res / N,
           "gpu_launches_per_call": int(launches // 4), "cpu_cores": 1}
    run = bridge.OracleRun(bridge.PLAIN, [z.oracle_dict()], Q2, pid2, Om, N, rng_mode=bridge.SEQUENTIAL, seed=3)
    run.set_fast_lookup(True)
    t = time.perf_counter(); run.run()
    out["cpu_port_optimised_us_per_sweep"] = 1e6 * (time.perf_counter() - t) / N
    if bridge.ref_lib() is not None:
        t = time.perf_counter(); bridge.ref_run(bridge.PLAIN, [z.oracle_dict()], Q2, pid2, Om, N, seed=3)
        out["cpu_reference_us_per_sweep"] = 1e6 * (time.perf_counter() - t) / N
    return out


def run_reference(a, rank, world):
    if rank != 0:
        return
    from oracle import bridge
    bridge.build()
    tree, Q, pid = workload_tree()
    order = tree_order_numpy(tree.edge, tree.T)
    kind = "reference" if bridge.ref_lib() is not None else "port_faithful"
    for _ in range(min(a.warmup, 1)):   # a tiny run so that page-in / fork costs stay out of the measurement
        cpu_leg(kind, tree, Q, pid, 1, order, sites_per_core=1)
    cb, wall = cpu_leg(kind, tree, Q, pid, a.steps, order)
    cfg = config(a.gpus, SITES_PER_GPU)
    cfg["precision"] = "f64"
    cfg["rng"] = "R Mersenne-Twister (sequential)"
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": min(a.warmup, 1), "ms_per_step": 1e3 * wall / a.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
            "cpu_baseline": cb, "gpu_launches": 0,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "each step is one sweep over a bounded site sample of the workload (%s)" % cb["sample"]}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------
def run_ours(a, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    import phylomap_b200 as pb
    from phylomap_b200 import capi, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the sampler has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    tree, Q, pid = workload_tree()
    S = SITES_PER_GPU
    E = tree.E
    # synthetic tip data for this rank's site block, generated on the GPU, staged in pinned host memory
    st_dev = synth.simulate_tip_states(tree, Q, pid, S, seed=101 + rank, device="cuda:%d" % local_rank,
                                       batch_sites=min(S, 32768))
    st_host = torch.empty((S, tree.T), dtype=torch.uint8, pin_memory=True)
    st_host.copy_(st_dev)
    del st_dev
    torch.cuda.empty_cache()
    z = tree.with_states(st_host.numpy(), segments=2)
    order = [z.order()]
    stream = torch.cuda.Stream()
    opts = dict(precision="f32", mode="production", seed=2026, device=local_rank, site_offset=rank * S,
                stream=stream.cuda_stream)
    if world > 1:  # the one collective of the path: the library's own ncclAllReduce of the statistics rows
        from phylomap_b200 import dist as pdist
        opts["nccl"] = pdist.nccl_clique(rank, world)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    total = a.warmup + a.steps
    chain = pb.Chain(capi.PM_V_BIGTREE, z, Q.copy(), pid, OMEGA, total + 2, order=order, **opts)
    chain.run(a.warmup)
    barrier()
    _, launches0 = chain.kernel_times()
    chain.enable_timing(True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        with torch.cuda.stream(stream):
            ev0.record(stream)
            rows = chain.run(a.steps)
            ev1.record(stream)
        barrier()
    ms = ev0.elapsed_time(ev1)
    chain.enable_timing(False)
    ktimes, launches = chain.kernel_times()
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = E * S * world * a.steps / (ms_max * 1e-3)

    # sanity: total dwell time per sweep == sites x tree length
    tot = rows[:, :4].sum(1)
    expect = S * world * tree.edge_length.sum()
    if not np.allclose(tot, expect, rtol=1e-3):
        raise SystemExit("bench sanity check failed: dwell %r vs %r" % (tot[:3], expect))
    if a.dump_outputs and rank == 0:   # the rows are already summed over ranks
        os.makedirs(a.dump_outputs, exist_ok=True)
        np.save(os.path.join(a.dump_outputs, "rows.npy"), np.ascontiguousarray(rows[-1:], dtype=np.float64))

    # roofline of the pruning pass (K1, SURVEY.md 8(d)).  In the step it is the first pass of the fused launch
    # k_prune_nodes_clade (prune the block's 32 sites, then draw their node states): the launch is timed with CUDA events
    # and split between the two passes by the block-nanoseconds (%globaltimer) the blocks report for each; the same pass
    # launched alone (phases = 1), five times back to back, is the cross-check `ms_per_launch_isolated`.
    K1_NAME = "k_prune_nodes_clade<float,4,8,3>"
    k1_ms = chain.time_prune(reps=5)
    T = tree.T
    bytes_site = (T - 1) * 16 + (T - 2) * 16 + T * 1 + E * 4
    bytes_site_k2 = (T - 2) * 16 + E * 4 + (2 * T - 1) * 2      # DESIGN.md section 3: partials and jump counts once, node states r/w
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    traffic = traffic_fused = None  # dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed ncu captures
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        if S == 125000 and TIPS == 10000:
            k1 = tj[K1_NAME + " (pruning pass alone)"]
            traffic = k1["dram_bytes_read"] + k1["dram_bytes_write"]
            kf = tj[K1_NAME]
            traffic_fused = kf["dram_bytes_read"] + kf["dram_bytes_write"]
    except Exception:
        pass
    k1_iso_ms = k1_ms                                  # the pruning pass launched alone, five times back to back
    k1_ms = ktimes["prune"] / a.steps                  # the pruning pass inside the timed region (share of the fused launch)
    fused_ms = (ktimes["prune"] + ktimes["sample_nodes"]) / a.steps   # the fused launch itself (CUDA events)
    ach = bytes_site * S / (k1_ms * 1e-3) / 1e9
    ach_fused = (bytes_site + bytes_site_k2) * S / (fused_ms * 1e-3) / 1e9
    roof = {"bound": "hbm", "kernel": K1_NAME + ", pruning pass (K1)", "achieved": ach, "peak": peak, "unit": "GB/s",
            "frac": ach / peak, "traffic": traffic, "traffic_source": "profiles/r2_traffic.json (ncu capture of this workload)" if traffic else None,
            "algorithmic_bytes_per_launch": bytes_site * S, "peak_source": "MEASURED_PEAKS.json (measured)" if peaks else "fallback 6650",
            "ms_per_launch": k1_ms, "ms_per_launch_isolated": k1_iso_ms, "frac_isolated": bytes_site * S / (k1_iso_ms * 1e-3) / 1e9 / peak,
            "algorithmic_bytes_per_site": bytes_site,
            "dram_gbs_actual": (traffic / (k1_ms * 1e-3) / 1e9) if traffic else None,
            "note": "K1 is the first pass of the fused prune + node-draw launch: ms_per_launch = the launch's CUDA-event time x the "
                    "share of block-nanoseconds its blocks spent pruning; ms_per_launch_isolated = the same pass launched alone.  The "
                    "clade-order walk hands a child's partial to its parent through registers / L2, so its DRAM traffic is below the "
                    "algorithmic bytes (which count every partial once written and once read)",
            "fused_launch": {"kernel": K1_NAME, "ms_per_launch": fused_ms, "algorithmic_bytes_per_site": bytes_site + bytes_site_k2,
                             "achieved": ach_fused, "frac": ach_fused / peak, "traffic": traffic_fused,
                             "dram_gbs_actual": (traffic_fused / (fused_ms * 1e-3) / 1e9) if traffic_fused else None},
            "in_step_ms": {k: v / a.steps for k, v in ktimes.items()}}
    dev_bytes = chain.device_bytes()
    chain.close()
    del chain
    torch.cuda.empty_cache()

    # end to end through the drop-in entry with host buffers: once with the library's device-buffer cache emptied (what a
    # single call in a fresh R session pays: cudaMalloc of the whole state), once more with the cache warm (a session that
    # calls the sampler repeatedly on the same tree)
    def e2e_call():
        barrier()
        t0 = time.perf_counter()
        res = pb.maketreelistMCMC_bigtree(z, Q.copy(), pid, np.asfortranarray(np.eye(4) + Q / OMEGA), OMEGA, *order[0], a.steps,
                                          **opts)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), res
    capi.lib().pm_release_cached_memory()
    first_s, res = e2e_call()
    e2e_s, res = e2e_call()
    e2e = {"value": E * S * world * a.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(S * tree.T / a.steps),
           "d2h_bytes_per_step": int(res.nbytes / a.steps), "seconds": e2e_s, "first_call_seconds": first_s,
           "first_call_value": E * S * world * a.steps / first_s,
           "what": "pm_maketreelistMCMC_bigtree(host tree + pinned u8 tip states): upload, chain build, %d sweeps, read-back. "
                   "`value` / `seconds`: a repeated call (device buffers come from the library's cache); `first_call_*`: the same "
                   "call with the cache emptied first (cudaMalloc of the whole state included)" % a.steps}

    # the rate-updating sampler on the same tree and site count: one small all-reduce + replicated host update per sweep
    rate = None
    if not a.no_rate:
        capi.lib().pm_release_cached_memory()
        zk = z  # same tips read as observed parity (1 / 2) of the hidden-rate model
        par = torch.from_numpy(z.states)
        par = ((par - 1) % 2 + 1).to(torch.uint8).numpy()     # observed trait of the 4 hidden states: 1,3 -> 1; 2,4 -> 2
        zk = tree.with_states(par, segments=2)
        Qk = np.asfortranarray(Q.copy())
        n_ks = max(4, min(a.steps, 12))
        prior_ks = np.array([1.0, 10.0, 2.0, 10.0, 20.0, 2.0])  # phylomap_tutorial.Rnw:261
        ks_opts = {k: v for k, v in opts.items() if k != "nccl"}
        if world > 1:
            ks_opts["nccl"] = pdist.nccl_clique(rank, world)
        ch = pb.Chain(capi.PM_V_KS, zk, Qk, pid, 4.0, n_ks + 3, prior=prior_ks, order=order, **ks_opts)
        ch.run(3)
        barrier()
        ch.enable_timing(True)
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record(stream)
        t0 = time.perf_counter()
        ch.run(n_ks)
        k1.record(stream)
        torch.cuda.synchronize()
        wall_ms = 1e3 * (time.perf_counter() - t0)
        comm_ms, host_ms = ch.overheads()
        kt, _ = ch.kernel_times()
        t = torch.tensor([wall_ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        rate = {"sampler": "sumstatMCMCks (4-state hidden-rate model, Omega = 4, prior c(1,10,2,10,20,2)), %d sites per GPU" % S,
                "sweeps": n_ks, "ms_per_sweep": float(t.item()) / n_ks, "value": E * S * world * n_ks / (float(t.item()) * 1e-3),
                "unit": UNIT, "allreduce_us_per_sweep": 1e3 * comm_ms / n_ks, "host_update_us_per_sweep": 1e3 * host_ms / n_ks,
                "allreduce_doubles": 4 + 16 + 1 + 1, "collective": "ncclAllReduce issued by the library on the chain's stream" if world > 1 else "none (1 rank)",
                "in_sweep_ms": {k: v / n_ks for k, v in kt.items()},
                "limits": "kernel time; the collective + D2H + host update + model upload are serialised with the sweep "
                          "(the next sweep's kernels need the new Q)"}
        ch.close()
        del ch

    cb = one = None
    if rank == 0 and world == 1 and not a.no_cpu:
        cb = cpu_baseline(tree, Q, pid)
        one = one_character(opts)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": ms_max / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config(world, S), "clocks": clk.summary(), "e2e": e2e,
                "gpu_launches": int(launches - launches0), "roofline": roof, "cpu_baseline": cb, "rate_sampler": rate, "one_character": one,
                "device_bytes": dev_bytes, "device_bytes_per_branch_site": dev_bytes / (E * S)}
        print(json.dumps(line))


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=None,
                   help="timed sweeps (default 10; for --impl reference PM_BENCH_CPU_STEPS, else 6)")
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours")
    p.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    p.add_argument("--no-rate", action="store_true", help="skip the rate_sampler block")
    p.add_argument("--dump-outputs", metavar="DIR", help="write the last timed sweep's statistics row to DIR/rows.npy")
    a = p.parse_args()
    if a.steps is None:
        a.steps = int(os.environ.get("PM_BENCH_CPU_STEPS", 6)) if a.impl == "reference" else 10
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        sys.stderr.write("bench.py: --dump-outputs ignored: the reference arm runs on the CPU and returns no GPU outputs\n")
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if a.impl == "reference":
        run_reference(a, rank, world)
    else:
        run_ours(a, rank, local_rank, world)


if __name__ == "__main__":
    main()

"""Cost of one exact posterior-expectation call (pb.expected_sumstats) against one MCMC sweep of the same data.

    python scripts/expected_sumstats.py [--out profiles/r3_expected_sumstats.log] [--skip-big]

Workloads: BASELINE configs[1] (1 000-tip Yule tree, 10 000 sites, 4-state JC, sumstatMCMC Omega 0.6), the benchmark size
(10 000 tips x 125 000 sites, 4-state make2sQ(.1,.1,.2,.2,10), sumstatMCMC_bigtree Omega 2.4), one binary character on the
100-tip tree of configs[0], and 8 states at configs[1]'s size.  Per workload and precision: the CUDA-event times of the
three kernel groups (P(t) + branch integrals, inside pass, outside pass; PHYLOMAP_B200_TRACE=1 prints them), the whole call
from host buffers (best of 3 after a warm-up, trace off), FMAs and bytes counted from the shapes, and the time of one sweep
of the fixed-Q sampler on the same data in the same process.  The card's name, power limit and maximum SM clock are read in
the same process.
"""
import argparse
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import phylomap_b200 as pb  # noqa: E402
from phylomap_b200 import capi, synth  # noqa: E402

HBM_BPS = 7.7e12  # HGX B200 data sheet, per GPU


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, pl, clk = [x.strip() for x in q.split(",")]
    return name, float(pl), float(clk)


def traced(fn):
    """Run fn() with PHYLOMAP_B200_TRACE=1 and return the library's expect lines from stderr."""
    os.environ["PHYLOMAP_B200_TRACE"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as f:
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["PHYLOMAP_B200_TRACE"]
        f.seek(0)
        lines = [ln for ln in f.read().splitlines() if "expect:" in ln]
    tot = np.zeros(3)
    for ln in lines:
        tot += [float(x) for x in re.findall(r"([0-9.]+) ms", ln)]
    return tot


def counts(z, n, S, rsz):
    """(FMAs, HBM bytes) of the three kernel groups from the shapes."""
    T, E, NK = z.T, z.E, n * n
    internal_children = T - 2
    tip_children = T
    Q_sq = 3  # squarings of the scaled block exponential are a few on these trees; the Taylor part dominates
    branch = E * NK * (18 * 3 * n ** 3 + Q_sq * 3 * n ** 3) + E * (18 + Q_sq) * n ** 3
    inside = S * (T - 1) * 2 * n * n
    outside = S * ((T - 1) * (2 * n * n + n) + internal_children * (n ** 4 + 2 * n * n) + tip_children * n ** 3)
    b_branch = E * NK * NK * rsz + E * n * n * rsz
    b_inside = S * ((T - 1) * n * rsz + internal_children * n * rsz + T) + S * 8
    b_outside = S * ((T - 1) * n * rsz * 2 + internal_children * n * rsz * 2 + T) + S * NK * 8
    return (branch, inside, outside), (b_branch, b_inside, b_outside)


def workload(name):
    if name == "configs[1]":
        Q, pid = np.full((4, 4), 0.1) - np.eye(4) * 0.4, np.full(4, 0.25)
        tree = synth.yule_tree(1000, seed=2, mean_branch=1.0)
        S, om, sampler = 10000, 0.6, capi.PM_V_PLAIN
    elif name == "n=8 at configs[1]":
        Q, pid = np.full((8, 8), 0.1 / 7) - np.eye(8) * 0.1 * 8 / 7, np.full(8, 0.125)
        tree = synth.yule_tree(1000, seed=2, mean_branch=1.0)
        S, om, sampler = 10000, 0.3, capi.PM_V_PLAIN
    elif name == "one character":
        Q, pid = np.array([[-0.1, 0.1], [0.1, -0.1]]), np.full(2, 0.5)
        z = synth.simulate_2_state_tree(101, synth.yule_tree(100, seed=1, mean_branch=5.0), Q, pid)
        return z, Q, pid, 0.2, capi.PM_V_PLAIN
    else:
        Q, pid = synth.make2sQ(0.1, 0.1, 0.2, 0.2, 10.0), np.full(4, 0.25)
        tree = synth.yule_tree(10000, seed=4, mean_branch=0.1 / float(np.max(-np.diag(Q))))
        S, om, sampler = 125000, 2.4, capi.PM_V_BIGTREE
    import torch
    st = synth.simulate_tip_states(tree, Q, pid, S, seed=101, device="cuda", batch_sites=32768).to("cpu").to(torch.uint8).numpy()
    return tree.with_states(st, segments=2), Q, pid, om, sampler


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--skip-big", action="store_true")
    a = ap.parse_args()
    name, plim, clk = card()
    fp32 = 148 * 128 * clk * 1e6  # FMA/s: 148 SMs x 128 FP32 (64 FP64) FMA lanes per clock at the maximum SM clock
    fp64 = 148 * 64 * clk * 1e6
    lines = ["card: %s, power limit %.0f W, max SM clock %.0f MHz; %s" % (name, plim, clk, pb.capi.lib().pm_version().decode()),
             "FMA rates used for the bounds: %.1f T FP32 / %.1f T FP64 FMA/s (148 SMs x 128 / 64 lanes x max clock); HBM %.1f TB/s"
             % (fp32 / 1e12, fp64 / 1e12, HBM_BPS / 1e12), ""]
    names = ["configs[1]", "benchmark size", "one character", "n=8 at configs[1]"]
    if a.skip_big:
        names.remove("benchmark size")
    for wl in names:
        z, Q, pid, om, sampler = workload(wl)
        n, S = Q.shape[0], z.n_sites()
        for prec in ("f32", "f64"):
            rsz = 4 if prec == "f32" else 8
            pb.expected_sumstats(z, Q, pid, precision=prec)   # warm-up (module load, pool)
            ms = traced(lambda: pb.expected_sumstats(z, Q, pid, precision=prec))
            best = 1e9
            for _ in range(3):
                t0 = time.perf_counter()
                r = pb.expected_sumstats(z, Q, pid, precision=prec)
                best = min(best, time.perf_counter() - t0)
            assert np.allclose(r.stats[:, :n].sum(1), z.edge_length.sum(), rtol=1e-4)
            fmas, byts = counts(z, n, S, rsz)
            rate = fp32 if prec == "f32" else fp64
            ch = pb.Chain(sampler, z, Q.copy(), pid, om, 8, precision=prec, seed=1)
            ch.run(3)
            t0 = time.perf_counter()
            ch.run(5)
            sweep = (time.perf_counter() - t0) / 5
            ch.close()
            lines.append("%s, %s: T=%d tips, S=%d sites, n=%d" % (wl, prec, z.T, S, n))
            for k, what in enumerate(("P(t) + branch integrals", "inside pass (k_loglik)", "outside pass (k_expect)")):
                t_c, t_m = fmas[k] / rate, byts[k] / HBM_BPS
                bound = "compute" if t_c > t_m else "memory"
                lines.append("  %-26s %9.3f ms   %.3g FMA  %.3g B   %s-bound floor %.3f ms (%.0f %% of it reached)"
                             % (what, ms[k], fmas[k], byts[k], bound, 1e3 * max(t_c, t_m), 100 * 1e3 * max(t_c, t_m) / max(ms[k], 1e-9)))
            lines.append("  whole call from host buffers %.3f ms; one sampler sweep %.3f ms; one exact call = %.1f sweeps"
                         % (1e3 * best, 1e3 * sweep, best / sweep))
            lines.append("")
            print("\n".join(lines[-6:]), flush=True)
        del z
    text = "\n".join(lines) + "\n"
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)
    print(text)


if __name__ == "__main__":
    main()

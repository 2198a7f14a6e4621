"""The DIC samplers' sweep (PM_V_DIC2S / PM_V_DICKS: the rate-updating chains with a log-likelihood column) at sizes
where the one-block-per-site kernel is not chosen, FP32 and FP64: ms per sweep (rate update and log-likelihood pass
included), kernel launches per sweep and the in-sweep split of kernel_times().  With --dump DIR every row the chains
returned is written to DIR/<config>_<precision>.npy, so that two builds can be compared bit for bit.

    python scripts/dic_sweep.py [--sweeps K] [--warmup W] [--reps R] [--dump DIR]
"""
import argparse, json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import bench
import phylomap_b200 as pb
from phylomap_b200 import capi, synth

PRIOR_BF = np.array([0.55, 1.0, 0.56, 1.01])            # phylomap_tutorial.Rnw:218
PRIOR_KS = np.array([1.0, 10.0, 2.0, 10.0, 20.0, 2.0])  # phylomap_tutorial.Rnw:261
Q2, PID2 = np.array([[-0.1, 0.1], [0.1, -0.1]]), np.array([0.5, 0.5])


def configs():
    """name -> (variant, tree with states, Q, pid, Omega, prior): the 4096-site hidden-rate case of the test suite and
    the benchmark's 10 000-tip tree with 32 768 sites, for both samplers."""
    small = synth.yule_tree(200, seed=6, mean_branch=0.4)
    big, Q4, pid4 = bench.workload_tree()
    S = 32768
    return {
        "dicks_T200_S4096": (capi.PM_V_DICKS, synth.simulate_4_state_tree(9, small, Q4, pid4, n_sites=4096, device="cuda", segments=2),
                             Q4, pid4, 4.0, PRIOR_KS),
        "dicks_bench_S32768": (capi.PM_V_DICKS, synth.simulate_4_state_tree(9, big, Q4, pid4, n_sites=S, device="cuda", segments=2),
                               Q4, pid4, 4.0, PRIOR_KS),
        "dic2s_bench_S32768": (capi.PM_V_DIC2S, synth.simulate_2_state_tree(9, big, Q2, PID2, n_sites=S, device="cuda", segments=2),
                               Q2, PID2, 1.0, PRIOR_BF),
    }


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--sweeps", type=int, default=10, help="timed sweeps per repetition")
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--reps", type=int, default=3, help="timed repetitions per chain")
    p.add_argument("--dump", metavar="DIR", help="write every row of each chain to DIR/<config>_<precision>.npy")
    a = p.parse_args()
    timed_sweeps = 5  # with per-kernel timing on, after the timed repetitions
    for name, (v, z, Q, pid, Om, prior) in configs().items():
        for prec in ("f32", "f64"):
            N = a.warmup + a.reps * a.sweeps + timed_sweeps
            ch = pb.Chain(v, z, np.asfortranarray(Q.copy()), pid, Om, N, prior=prior, precision=prec, seed=5)
            rows = [ch.run(a.warmup)]
            ms = []
            for _ in range(a.reps):
                torch.cuda.synchronize(); t0 = time.perf_counter()
                rows.append(ch.run(a.sweeps))
                torch.cuda.synchronize(); ms.append(1e3 * (time.perf_counter() - t0) / a.sweeps)
            _, l0 = ch.kernel_times()
            ch.enable_timing(True)
            rows.append(ch.run(timed_sweeps))
            kt, l1 = ch.kernel_times()
            rows = np.concatenate(rows)
            if a.dump:
                os.makedirs(a.dump, exist_ok=True)
                np.save(os.path.join(a.dump, "%s_%s.npy" % (name, prec)), rows)
            print(json.dumps({"config": name, "precision": prec, "sites": z.n_sites(), "tips": z.T,
                              "ms_per_sweep": [round(x, 3) for x in ms],
                              "launches_per_sweep": (l1 - l0) / timed_sweeps,
                              "kernel_ms_per_sweep": {k: round(x / timed_sweeps, 3) for k, x in kt.items()},
                              "loglik_last": rows[-1, -1]}), flush=True)
            ch.close(); del ch
            capi.lib().pm_release_cached_memory()


if __name__ == "__main__":
    main()

"""Cost of exporting stochastic maps (Chain.maps / pm_chain_get_maps) from the benchmark chain: the 10 000-tip tree of
bench.py (19 998 branches), 125 000 resident sites, FP32, after a few sweeps.

For contiguous selections of 1 024 and 8 192 sites and for 1 024 scattered sites: the decode kernels' device time
(torch.profiler, CUDA activities: k_maps_count, the CUB scan, k_maps_write), their algorithmic bytes over that time as a
share of the device-to-device copy bandwidth measured in the same run (6 B of state words read and 8 B of offsets written
per branch-site, 12 B written per run, the stored records read: sizeof(Real) + 1 B per record, header records included),
the device-to-host copy time, and the end-to-end Chain.maps time (host clock, both calls, host allocation included);
for scale one sweep's time (CUDA events) and path() over every branch of one site (host clock).  Prints the card's name
and power limit first.

    python scripts/maps_export.py [--sites 125000] [--reps 5]
"""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import phylomap_b200 as pb  # noqa: E402
from phylomap_b200 import capi, synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def copy_bandwidth(nbytes=4 << 30, reps=20):
    """Device-to-device copy of a 4 GiB buffer (larger than L2): bytes read + written per second."""
    a = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    s = e0.elapsed_time(e1) / 1e3 / reps
    del a, b
    torch.cuda.empty_cache()
    return 2 * nbytes / s


def algorithmic_bytes(m, real_bytes):
    """What the decode must move: state words and offsets per branch-site, the runs, the stored records it reads."""
    runs = np.diff(m.off)
    bs = len(runs)
    rec = runs[runs >= 3]                      # production: paths with two or more real jumps are stored as records
    headers = int(np.count_nonzero(rec >= 64))  # ... 64 runs or more behind a header record
    return bs * (6 + 8) + int(runs.sum()) * 12 + (int(rec.sum()) + headers) * (real_bytes + 1)


def profiled(fn):
    """(kernel ms by name, device-to-host copy ms) of one call of fn."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    kern, d2h = {}, 0.0
    for ev in prof.events():
        if ev.device_type != DeviceType.CUDA:
            continue
        t = ev.time_range.elapsed_us() / 1e3
        if ev.name.startswith("Memcpy DtoH"):
            d2h += t
        elif "k_maps_" in ev.name or "DeviceScan" in ev.name:
            key = "k_maps_count" if "k_maps_count" in ev.name else "k_maps_write" if "k_maps_write" in ev.name else "cub scan"
            kern[key] = kern.get(key, 0.0) + t
    return kern, d2h


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=bench.SITES_PER_GPU)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("maps_export.py needs a B200")
    print("card (name, power limit, max SM clock):", card())
    tree, Q, pid = bench.workload_tree()
    S, E = a.sites, tree.E
    st = synth.simulate_tip_states(tree, Q, pid, S, seed=101, device="cuda", batch_sites=min(S, 32768)).cpu().numpy()
    torch.cuda.empty_cache()
    z = tree.with_states(st, segments=2)
    ch = pb.Chain(capi.PM_V_BIGTREE, z, Q.copy(), pid, bench.OMEGA, 64, precision="f32", seed=2026)
    ch.run(4)
    torch.cuda.synchronize()
    print("workload: %d tips, %d branches, %d resident sites, FP32, after 4 sweeps" % (tree.T, E, S))
    bw = copy_bandwidth()
    print("device-to-device copy bandwidth (4 GiB buffer, read + write): %.0f GB/s" % (bw / 1e9))

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ch.run(a.reps)
    e1.record()
    torch.cuda.synchronize()
    sweep_ms = e0.elapsed_time(e1) / a.reps
    print("one sweep (CUDA events, mean of %d): %.2f ms" % (a.reps, sweep_ms))

    t0 = time.perf_counter()
    for e in range(E):
        ch.path(7, e)
    path_s = time.perf_counter() - t0
    print("path() over the %d branches of one site: %.2f s" % (E, path_s))

    rng = np.random.default_rng(5)
    selections = [("contiguous 1024", np.arange(1000, 1000 + 1024)), ("contiguous 8192", np.arange(20000, 20000 + 8192)),
                  ("scattered 1024", np.sort(rng.choice(S, size=1024, replace=False)))]
    for name, sel in selections:
        m = ch.maps(sel)                        # warm-up (module load, scratch pool)
        ts = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            m = ch.maps(sel)
            ts.append(time.perf_counter() - t0)
        kern, d2h = profiled(lambda: ch.maps(sel))
        kms = sum(kern.values())
        ab = algorithmic_bytes(m, 4)
        runs = int(m.off[-1])
        print("%s: %d branch-sites, %d runs (%.3f per branch-site)" % (name, len(m) * E, runs, runs / (len(m) * E)))
        print("  decode kernels (device time of one Chain.maps, both calls): %.3f ms  [%s]"
              % (kms, ", ".join("%s %.3f" % kv for kv in sorted(kern.items()))))
        print("  algorithmic bytes of one decode: %.1f MB" % (ab / 1e6))
        # Chain.maps calls the entry twice: sizes (count + scan), then data (count + scan + write); the data call's kernels
        data_ms = kern.get("k_maps_write", 0.0) + 0.5 * (kern.get("k_maps_count", 0.0) + kern.get("cub scan", 0.0))
        print("  kernels of the data call %.3f ms: %.0f GB/s = %.0f%% of the measured copy bandwidth"
              % (data_ms, ab / (data_ms / 1e3) / 1e9, 100 * ab / (data_ms / 1e3) / bw))
        print("  device-to-host copies: %.3f ms (%.1f MB of offsets and runs)" % (d2h, (2 * (len(m) * E + 1) * 8 + runs * 12) / 1e6))
        print("  end-to-end Chain.maps: median %.1f ms, min %.1f ms over %d calls" % (1e3 * np.median(ts), 1e3 * min(ts), a.reps))
        del m
    print("done")


if __name__ == "__main__":
    main()

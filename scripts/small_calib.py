"""Where the one-block-per-site chain kernel (pm_small.cuh) stops paying: microseconds per sweep of a resident chain, one
character, against the 32-sites-per-warp kernels, as the work of a site (branches + jump points) grows."""
import os, sys, time, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np, torch
import cases
import phylomap_b200 as pb
from phylomap_b200 import capi, synth

def resident(z, Q, pid, Om, n_sweeps, prec="f32"):
    ch = pb.Chain(capi.PM_V_BIGTREE, z, Q, pid, Om, 5 * n_sweeps, precision=prec, seed=5)
    ch.run(n_sweeps)
    best = 1e30
    for _ in range(3):
        torch.cuda.synchronize(); t = time.perf_counter(); ch.run(n_sweeps); torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t)
    ch.close()
    return round(1e6 * best / n_sweeps, 2)

out = {}
Q4 = cases.q4(); pid4 = np.full(4, 0.25)
os.environ["PHYLOMAP_B200_SMALL_WORK"] = "1e15"
os.environ["PHYLOMAP_B200_SMALL_SITES"] = "100000"
for name, T, mb, Om, S, n_sw in [("T100_Om2.4", 100, 1.0, 2.4, 1, 400), ("T100_Om24", 100, 1.0, 24.0, 1, 200), ("T300_Om2.4", 300, 1.0, 2.4, 1, 300),
                                 ("T1000_Om2.4", 1000, 0.5, 2.4, 1, 200), ("T1000_Om12", 1000, 0.5, 12.0, 1, 100), ("T3000_Om2.4", 3000, 0.3, 2.4, 1, 100),
                                 ("T1000_Om2.4_S148", 1000, 0.5, 2.4, 148, 60), ("T300_Om2.4_S592", 300, 1.0, 2.4, 592, 60)]:
    z = cases.tree_n(Q4, T=T, S=S, seed=3, mean_branch=mb, segments=2)
    work = z.E + 1.5 * Om * float(np.sum(z.edge_length)) + 2 * z.E
    row = {"work_per_site": round(work)}
    for small in ("1", "0"):
        os.environ["PHYLOMAP_B200_SMALL"] = small
        row["one_block_per_site" if small == "1" else "wide"] = resident(z, Q4.copy(), pid4, Om, n_sw)
    out[name] = row
print(json.dumps(out))

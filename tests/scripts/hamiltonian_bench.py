"""What Hamiltonian replica exchange costs in the fused step kernel: a Hamiltonian ladder and a temperature ladder, each with
a swap round at every measure, against the scalar kernel on the same workload, the three arms alternating in one process.

  c2: 65,536 xy-well chains x 10^5 steps, measure every 10, R = 8: well depths k_r geometric 1.0 .. 0.05 at T = 0.1 /
      temperatures geometric 0.05 .. 1.0 / temp = 0.1
  c3: 262,144 mixed 3r+4c chains x 10^3 steps, measure every 10, R = 8: k[1] from -1.0 to -0.2 at T = 0.1 /
      temperatures as c2 / temp = 0.1

Prints the card, its power limit and SM clock, then per arm the best and the spread (max - min) of the repeats in ms,
chain-steps/s, and the ladder's swap acceptance per neighbour pair.  record=False: the time series is not part of either arm.

usage: python tests/scripts/hamiltonian_bench.py [repeats, default 5] [output json]
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    import numpy as np
    import torch
    import metropolisengine_b200 as me
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    out = dict(card=card(), results={})
    print("card:", out["card"], flush=True)
    work = {
        "c2": (lambda t, k, kr=None: me.MetropolisEngine(("xy_well", 1.0), initial_real_params=np.zeros(2), temp=t,
                                                         n_chains=65536, seed=7, record=False, replica_exchange=k,
                                                         rung_consts=kr), 10000, 10,
               np.geomspace(1.0, 0.05, 8)[:, None]),
        "c3": (lambda t, k, kr=None: me.MetropolisEngine(("mixed_well", 1.0, -1.0, 0.5, 1.0), initial_real_params=np.zeros(3),
                                                         initial_complex_params=np.zeros(4, dtype=complex), temp=t,
                                                         n_chains=262144, seed=7, record=False, replica_exchange=k,
                                                         rung_consts=kr), 100, 10,
               np.array([[1.0, k1, 0.5, 1.0] for k1 in np.linspace(-1.0, -0.2, 8)])),
    }
    ladder = list(np.geomspace(0.05, 1.0, 8))
    for name, (make, M, spm, kr) in work.items():
        arms = {"scalar": make(0.1, 0), "ladder_R8": make(ladder, 1), "hamiltonian_R8": make(0.1, 1, kr)}
        for e in arms.values():                      # warm-up: module load, first launch
            e.run(10, spm)
        times = {k: [] for k in arms}
        for _ in range(reps):
            for k, e in arms.items():                # alternate the arms
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                a.record()
                e.run(M, spm)
                b.record()
                torch.cuda.synchronize()
                times[k].append(a.elapsed_time(b))
        n = arms["scalar"].n_chains
        for k, ts in times.items():
            best = min(ts)
            r = dict(best_ms=best, spread_ms=max(ts) - best, chain_steps_per_s=n * M * spm / best * 1e3,
                     grid=arms[k]._grid, block=arms[k]._block)
            if k != "scalar":
                r["swap_acceptance"] = [float(v) for v in arms[k].swap_acceptance_rate]
            out["results"]["%s_%s" % (name, k)] = r
            print("%s %-10s best %9.3f ms  spread %.3f ms  %.4e chain-steps/s  grid %d x %d %s" % (
                name, k, best, max(ts) - best, r["chain_steps_per_s"], r["grid"], r["block"],
                ("swap acceptance " + " ".join("%.3f" % v for v in r["swap_acceptance"])) if "swap_acceptance" in r
                else ""), flush=True)
        s, l = out["results"][name + "_scalar"]["best_ms"], out["results"][name + "_ladder_R8"]["best_ms"]
        h = out["results"][name + "_hamiltonian_R8"]["best_ms"]
        print("%s temperature-ladder overhead: %+.2f %%, Hamiltonian-ladder overhead: %+.2f %%" % (
            name, 100 * (l / s - 1), 100 * (h / s - 1)), flush=True)
    if len(sys.argv) > 2:
        os.makedirs(os.path.dirname(os.path.abspath(sys.argv[2])), exist_ok=True)
        with open(sys.argv[2], "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()

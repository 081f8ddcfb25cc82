"""What a free-energy profile costs on the device (csrc/me_mbar.cuh k_mbar_hist, me_mbar_hist_pass) against the plain
MBAR pass (k_mbar, me_mbar_pass) over the same recorded rows.

  c2: xy-well temperature ladder, R = 8 (T geometric 0.05 .. 1.0), 65,536 chains, 2,000 recorded measures: 1.31e8
      samples; profiles of x with 100 bins and of (x, y) with 40 x 40 bins at a target between the rungs
  c3: mixed 3r+4c Hamiltonian ladder, R = 8 (k[1] from -1.0 to -0.2 at T = 0.1), 65,536 chains, 500 recorded measures:
      3.3e7 samples; profile of |c_0| with 100 bins

Each pass is timed with CUDA events after a warm-up, best and spread of the repeats; the plain pass and the histogram
passes alternate in one process, repeat by repeat.  Both evaluate R + 1 energies and exponentials per sample (the plain
pass without targets evaluates R).  The host algebra of ``pmf()`` (Theta over R + 1,600 states) is timed on the 40 x 40
sums.  The card, its power limit and SM clock are read in the same run.  The recorded rows exceed the 126 MB L2.

usage: python tests/scripts/pmf_bench.py [repeats, default 5] [output json]
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def timed(fn):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()                                          # includes the read-back of the sums
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def main():
    import numpy as np
    import torch
    import metropolisengine_b200 as me
    from metropolisengine_b200 import mbar as mb
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    out = dict(card=card(), results={})
    print("card:", out["card"], flush=True)
    R = 8
    work = {
        "c2": dict(make=lambda: me.MetropolisEngine(("xy_well", 1.0), initial_real_params=np.zeros(2),
                                                    temp=list(np.geomspace(0.05, 1.0, R)), replica_exchange=1,
                                                    n_chains=65536, seed=1, device="cuda:0"),
                   measures=2000, target=(0.3, None),
                   hists={"x_100": ([0], [0], [-1.0], [1.0], [100]),
                          "xy_40x40": ([0, 0], [0, 1], [-1.0, -1.0], [1.0, 1.0], [40, 40])}),
        "c3": dict(make=lambda: me.MetropolisEngine(me.BuiltinEnergy("mixed_well", 1.0, -1.0, 0.5, 1.0),
                                                    initial_real_params=np.full(3, 0.5),
                                                    initial_complex_params=np.full(4, 0.1 + 0.1j), temp=0.1,
                                                    rung_consts=np.stack([np.ones(R), np.linspace(-1.0, -0.2, R),
                                                                          np.full(R, 0.5), np.ones(R)], axis=1),
                                                    replica_exchange=1, n_chains=65536, seed=1, device="cuda:0"),
                   measures=500, target=(0.1, np.array([1.0, -0.6, 0.5, 1.0])),
                   hists={"abs_c0_100": ([1], [0], [0.0], [1.5], [100])}),
    }
    for name, w in work.items():
        eng = w["make"]()
        eng.reserve_rows(w["measures"])
        eng.run(w["measures"], 10)
        torch.cuda.synchronize()
        n = eng._ts_rows * eng.n_chains
        f = eng.mbar(burn_in=0.0).free_energies
        tt, kt = w["target"]
        calls = {"plain": lambda: eng._mbar_sums(f, np.zeros(0), None, False, 0, 1)}
        for label, (kinds, idx, lo, hi, nb) in w["hists"].items():
            calls[label] = (lambda kinds=kinds, idx=idx, lo=lo, hi=hi, nb=nb:
                            eng._mbar_hist_sums(f, tt, kt, kinds, idx, lo, hi, nb, 0, 1))
        for fn in calls.values():                        # warm-up: modules, shared-memory attributes, buffers
            fn()
            fn()
        times = {k: [] for k in calls}
        last = {}
        for _ in range(reps):                            # alternate the passes repeat by repeat
            for k, fn in calls.items():
                ms, last[k] = timed(fn)
                times[k].append(ms)
        res = {"samples": n, "D": eng._d}
        for k, t in times.items():
            res[k] = dict(ms=min(t), spread_ms=max(t) - min(t), samples_per_s=n / (min(t) * 1e-3))
            print(name, k, res[k], flush=True)
        if "xy_40x40" in last:
            s = last["xy_40x40"]
            G = eng._mbar_sums(f, np.zeros(0), None, False, 0, 1)["G"]
            t0 = time.perf_counter()
            mb.profile(s["h"], s["q"], s["c"], s["w_out"], G, n // R)
            res["host_profile_1600_bins_s"] = time.perf_counter() - t0
            print(name, "host profile algebra, 1,600 bins:", res["host_profile_1600_bins_s"], "s on",
                  os.cpu_count(), "host cores", flush=True)
        out["results"][name] = res
        del eng
        torch.cuda.empty_cache()
    if len(sys.argv) > 2:
        with open(sys.argv[2], "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()

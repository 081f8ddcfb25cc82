"""What the uncertainties of reweighted expectations cost on the device (csrc/me_mbar.cuh, me_mbar_cov_pass), beside the
plain ``evaluate()`` they extend.  The workloads are those of tests/scripts/mbar_bench.py:

  c2: xy-well temperature ladder, R = 8 (T geometric 0.05 .. 1.0), 65,536 chains, 2,000 recorded measures (every 10
      steps): 1.31e8 samples of D = 2 words; 20 targets between the rungs (S = 28, m = 6 observables)
  c3: mixed 3r+4c Hamiltonian ladder, R = 8 (k[1] from -1.0 to -0.2 at T = 0.1), 65,536 chains, 500 recorded measures:
      3.3e7 samples of D = 11 words; 2 targets (S = 10, m = 24)

Per workload, after a full ``mbar()`` solve: ``evaluate()`` and ``evaluate(uncertainty=True)`` alternating in one
process, then each covariance pass of the split the library asked for on its own.  Every call sits between two CUDA
events and a synchronise (best and spread of the repeats after a warm-up) and includes the host algebra and the
read-back of the sums.  The card, its power limit and SM clock are read in the same run.  The recorded rows (4.2 GB for
c2) exceed the 126 MB L2, so every pass reads HBM.

usage: python tests/scripts/expectation_bench.py [repeats, default 5] [output json]
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


def _events(fn, reps):
    """Best and spread (ms) of fn() over reps calls, each between two CUDA events and a synchronise."""
    import torch
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return min(times), max(times) - min(times)


def uncertainty_arm(eng, r, tt, kt, reps):
    """evaluate() and evaluate(uncertainty=True) alternating, then each covariance pass of the split on its own."""
    import numpy as np
    plain = lambda: r.evaluate(temp=tt, consts=kt)
    full = lambda: r.evaluate(temp=tt, consts=kt, uncertainty=True)
    plain(), full()                                                    # warm-up of both
    tp, tf = [], []
    for _ in range(reps):
        tp.append(_events(plain, 1)[0])
        tf.append(_events(full, 1)[0])
    R, m = r.free_energies.size, 2 * eng._d + 2
    ev = full()
    cen = np.concatenate([ev["x_mean"], ev["x2_mean"], ev["E_mean"][:, None], ev["E2_mean"][:, None]], axis=1)
    passes = eng._mbar_cov_sums(r.free_energies, tt, kt, R, tt.size, cen, *r._sample)["passes"]
    per = []
    for first, count in passes:
        c = cen[first - R:first - R + count]
        one = lambda: eng._mbar_cov_sums(r.free_energies, tt, kt, first, count, c, *r._sample)
        one()
        best, spread = _events(one, reps)
        per.append(dict(first=first, count=count, ms=best, spread_ms=spread))
    return dict(targets=int(tt.size), m=m, evaluate_ms=min(tp), evaluate_spread_ms=max(tp) - min(tp),
                evaluate_uncertainty_ms=min(tf), evaluate_uncertainty_spread_ms=max(tf) - min(tf),
                n_cov_passes=len(passes), cov_passes=per, max_dE_mean=float(np.max(ev["dE_mean"])),
                heat_capacity=ev["heat_capacity"].tolist(), dheat_capacity=ev["dheat_capacity"].tolist())


def main():
    import numpy as np
    import torch
    import metropolisengine_b200 as me
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    out = dict(card=card(), results={})
    print("card:", out["card"], flush=True)
    R = 8
    kt3 = np.array([[1.0, -0.6, 0.5, 1.0], [1.0, -0.3, 0.5, 1.0]])
    work = {
        "c2": dict(make=lambda: me.MetropolisEngine(("xy_well", 1.0), initial_real_params=np.zeros(2),
                                                    temp=list(np.geomspace(0.05, 1.0, R)), replica_exchange=1,
                                                    n_chains=65536, seed=1, device="cuda:0"),
                   measures=2000, targets=(np.geomspace(0.06, 0.9, 20), None)),
        "c3": dict(make=lambda: me.MetropolisEngine(me.BuiltinEnergy("mixed_well", 1.0, -1.0, 0.5, 1.0),
                                                    initial_real_params=np.full(3, 0.5),
                                                    initial_complex_params=np.full(4, 0.1 + 0.1j), temp=0.1,
                                                    rung_consts=np.stack([np.ones(R), np.linspace(-1.0, -0.2, R),
                                                                          np.full(R, 0.5), np.ones(R)], axis=1),
                                                    replica_exchange=1, n_chains=65536, seed=1, device="cuda:0"),
                   measures=500, targets=(np.array([0.1, 0.1]), kt3)),
    }
    for name, w in work.items():
        eng = w["make"]()
        eng.reserve_rows(w["measures"])
        eng.run(w["measures"], 10)
        torch.cuda.synchronize()
        r = eng.mbar(burn_in=0.0)
        res = dict(samples=eng._ts_rows * eng.n_chains, D=eng._d, converged=r.converged,
                   uncertainty=uncertainty_arm(eng, r, *w["targets"], reps))
        print(name, res, flush=True)
        out["results"][name] = res
        del eng
        torch.cuda.empty_cache()
    if len(sys.argv) > 2:
        with open(sys.argv[2], "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()

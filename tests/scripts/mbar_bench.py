"""What an MBAR pass over recorded ladder rows costs on the device (csrc/me_mbar.cuh, me_mbar_pass).

  c2: xy-well temperature ladder, R = 8 (T geometric 0.05 .. 1.0), 65,536 chains, 2,000 recorded measures (every 10
      steps): 1.31e8 samples of D = 2 words
  c3: mixed 3r+4c Hamiltonian ladder, R = 8 (k[1] from -1.0 to -0.2 at T = 0.1), 65,536 chains, 500 recorded measures:
      3.3e7 samples of D = 11 words

Per workload: one pass timed with CUDA events after a warm-up (best and spread of the repeats), without observables
(s, G and sum L: the Gram product is always formed) and with observables (+ 2 targets), then a full ``mbar()`` solve
and its Newton iterations.  Reports samples/s per pass and the two bounds: the x columns read (D x 8 B per sample) over
7.7 TB/s, and the static FP64 instruction count of the pass kernel's SASS (cuobjdump).  The numpy oracle's per-sample
rate on the host cores is measured on a 10^6-sample subset of the c2 rows.  The card, its power limit and SM clock are
read in the same run.  The recorded rows (4.2 GB for c2) exceed the 126 MB L2, so every pass reads HBM.

usage: python tests/scripts/mbar_bench.py [repeats, default 5] [output json]
"""
import json
import os
import re
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


def fp64_sass_counts():
    """Static counts of FP64 instructions in the fast build's k_mbar instantiations (None if cuobjdump is missing)."""
    obj = os.path.join(ROOT, "metropolisengine_b200", "csrc", "build", "me_aot_fast.o")
    try:
        txt = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, timeout=300).stdout
    except (OSError, subprocess.SubprocessError):
        return None
    out, cur = {}, None
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1) if "k_mbar" in m.group(1) else None
            if cur:
                out[cur] = {}
            continue
        if cur:
            m = re.search(r"\*/\s+(?:@!?U?P\w+\s+)?(D[A-Z]+|MUFU\.\w+)", line)
            if m and m.group(1) in ("DFMA", "DADD", "DMUL", "DSETP", "DMMA", "MUFU.RCP64H", "MUFU.RSQ64H"):
                out[cur][m.group(1)] = out[cur].get(m.group(1), 0) + 1
    return out


def time_pass(eng, f, tt, kt, obs, row0, reps):
    import torch
    for _ in range(2):
        eng._mbar_sums(f, tt, kt, obs, row0, 1)
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng._mbar_sums(f, tt, kt, obs, row0, 1)        # includes the read-back of the sums (a few hundred bytes)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return min(times), max(times) - min(times)


def main():
    import numpy as np
    import torch
    import metropolisengine_b200 as me
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    out = dict(card=card(), results={}, fp64_sass=fp64_sass_counts())
    print("card:", out["card"], flush=True)
    R = 8
    work = {
        "c2": dict(make=lambda: me.MetropolisEngine(("xy_well", 1.0), initial_real_params=np.zeros(2),
                                                    temp=list(np.geomspace(0.05, 1.0, R)), replica_exchange=1,
                                                    n_chains=65536, seed=1, device="cuda:0"),
                   measures=2000, targets=(np.array([0.1, 0.5]), None)),
        "c3": dict(make=lambda: me.MetropolisEngine(me.BuiltinEnergy("mixed_well", 1.0, -1.0, 0.5, 1.0),
                                                    initial_real_params=np.full(3, 0.5),
                                                    initial_complex_params=np.full(4, 0.1 + 0.1j), temp=0.1,
                                                    rung_consts=np.stack([np.ones(R), np.linspace(-1.0, -0.2, R),
                                                                          np.full(R, 0.5), np.ones(R)], axis=1),
                                                    replica_exchange=1, n_chains=65536, seed=1, device="cuda:0"),
                   measures=500, targets=(np.array([0.1, 0.1]), np.array([[1.0, -0.6, 0.5, 1.0], [1.0, -0.3, 0.5, 1.0]]))),
    }
    for name, w in work.items():
        eng = w["make"]()
        eng.reserve_rows(w["measures"])
        eng.run(w["measures"], 10)
        torch.cuda.synchronize()
        n = eng._ts_rows * eng.n_chains
        d = eng._d
        f = np.zeros(R)
        res = {"samples": n, "D": d}
        for label, tt, kt, obs in (("sums", np.zeros(0), None, False),
                                   ("obs_targets", w["targets"][0], w["targets"][1], True)):
            best, spread = time_pass(eng, f, tt, kt, obs, 0, reps)
            res[label] = dict(ms=best, spread_ms=spread, samples_per_s=n / (best * 1e-3),
                              hbm_bound_ms=n * d * 8 / 7.7e12 * 1e3)
            print(name, label, res[label], flush=True)
        t0 = time.perf_counter()
        r = eng.mbar(burn_in=0.0)
        torch.cuda.synchronize()
        res["solve"] = dict(s=time.perf_counter() - t0, iterations=r.n_iterations, converged=r.converged,
                            f=r.free_energies.tolist())
        print(name, "solve", res["solve"], flush=True)
        if name == "c2":
            from oracle import mbar_oracle as mo
            ts = eng.time_series()[:16].cpu().numpy()
            x = ts[:, :d, :].transpose(0, 2, 1).reshape(-1, d)[:1000000]
            temps = eng.temperatures
            t0 = time.perf_counter()
            E, walled = mo.energies(lambda xx, k: mo.energy("xy_well", xx, k), x, np.ones((R, 1)))
            mo.pass_sums(mo.reduced(E, walled, temps), f, x.shape[0] // R, R)
            dt = time.perf_counter() - t0
            res["numpy_oracle_samples_per_s"] = x.shape[0] / dt
            print(name, "numpy oracle samples/s", x.shape[0] / dt, "on", os.cpu_count(), "host cores", flush=True)
        out["results"][name] = res
        del eng
        torch.cuda.empty_cache()
    print(json.dumps(out["fp64_sass"], indent=1))
    if len(sys.argv) > 2:
        with open(sys.argv[2], "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py — ensemble chain-steps/sec of the step_all()/measure() hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c1|c3|c4]
                    [--dump-outputs DIR]

Headline workload (N=1 and per rank for N>1, weak scaling): BASELINE.json configs[1] — demo/toymodel_xypotentialwell:
2 real params, E = x^2+y^2, T = 0.1, 65,536 chains x 10^5 steps, measure every 10 steps (DXY:39-44), FP64.
One bench "step" = ONE pass of that whole job: 10^4 x (10 x step_all() + measure()) for every chain, i.e.
6.5536e9 chain-steps and 10^4 time-series rows per chain (21 GB written to HBM per pass, larger than L2).

value  : chain-steps/s, device-timed (CUDA events on the launching stream, barrier + synchronize on both sides,
         max over ranks), state resident in HBM.
e2e    : the same metric through the public Python API with HOST buffers: per step the initial parameters of all
         chains are copied from pinned host memory (H2D), the job runs, and the final per-chain state, the pooled
         statistics and chain 0's time series are read back to the host (D2H), all inside the timed region.
roofline: the step kernel is FP64-pipe bound (SURVEY.md §8d): `achieved` = algorithmic flops (20 flop per
         chain-step for the xy-well, special functions not counted) / kernel time, `peak` = FP64 FMA throughput
         measured live by me_probe_fp64 (MEASURED_PEAKS.json has no FP64 figure); the HBM side (time-series bytes
         / kernel time vs the measured copy bandwidth) is reported next to it.
workloads: short device-timed passes of the other BASELINE configs in the same line — c1 (README x^2), c3 (mixed
         3r+4c, 262,144 chains), c4 (1r+64c shared covariance on the tensor cores, with its per-measure moment
         all-reduce when N > 1) and c5 (config 5: 2^20 xy-well chains in TOTAL sharded over the N ranks, pooled-moment
         all-reduce after every 100-step launch, CUDA-graph launches) — each with its own kernel time and roofline.
check.invariance: SHA-256 of the state block of global chains 0..255 after one pass from the initial state; the Philox
         counter carries the global chain id, so the digest must be the same at every N.
cpu_baseline / --impl reference: the UNMODIFIED reference (baseline/_ref, or /root/reference in the build container;
         kind "reference") driven by its own README loop on the host cores, one chain per process; if neither copy is on
         the box, the numpy port of the same loop (oracle/py_port.py, pinned bit-for-bit against the reference; kind "port").
--dump-outputs DIR: after the timed steps, what the timed path handed its caller in its last step as float64 DIR/<name>.npy
         (see dump_outputs), so that two builds can be compared output for output on identical seeded inputs.
"""
import argparse
import json
import os
import sys
import threading
import time

sys.dont_write_bytecode = True        # the tree may be read-only: the bench writes nothing into it

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# SURVEY.md §8(d): algorithmic work per chain-step / bytes per chain-measure (x[D], E, sigma stored in FP64).
# inst / fp64_inst / wide_inst / dmma_inst: instructions, FP64 instructions, IMAD.WIDE and FP64 tensor-core MMAs per
# chain-step over one whole MEASURE PERIOD (spm steps + the measure block + the per-measure prologue) in the SASS of the
# shipped library (tests/scripts/sass_period.py <kernel> <spm>) — the inputs of the pipe-level roofline below.  The step
# loops alone (tests/scripts/sass_loop.py) are 126.5 / 40 / 12 (C2), 636 / 257 / 52 (C3).  C1's period alternates between two
# paths (one Philox call and one Box-Muller pair per TWO steps, me_device.cuh ShareCall), so its counts are the dynamic
# ones of an ncu capture of one bench pass (profiles/r02_ncu_c1_k_run.csv: smsp__inst_executed.sum / warp-steps = 210.1,
# sm__pipe_fp64_cycles_active -> 65.8 FP64 instructions, 14 IMAD.WIDE per pair of steps).
WORKLOADS = {
    "c1": dict(name="README x^2: 1 real param, T=0.01, measure every step", energy=("x2",), n_r=1, n_c=0, temp=0.01,
               chains=65536, measures=10000, short_measures=10000, spm=1, flop=10, sf=3, inst=210.1, fp64_inst=65.8, wide_inst=7.0, dmma_inst=0.0),
    "c2": dict(name="demo/toymodel_xypotentialwell: 2 real params, E=x^2+y^2, T=0.1, 65,536 chains x 1e5 steps, "
                    "measure every 10", energy=("xy_well", 1.0), n_r=2, n_c=0, temp=0.1, chains=65536,
               measures=10000, short_measures=2000, spm=10, flop=20, sf=5, inst=146.3, fp64_inst=48.2, wide_inst=12.3, dmma_inst=0.0),
    "c3": dict(name="mixed 3 real + 4 complex (bounded demo-style well), T=0.1, 262,144 chains, measure every 10",
               energy=("mixed_well", 1.0, -1.0, 0.5, 1.0), n_r=3, n_c=4, temp=0.1, chains=262144, measures=100,
               short_measures=100, spm=10, flop=170, sf=23, inst=787.3, fp64_inst=305.4, wide_inst=54.1, dmma_inst=4.0),
}
# the CPU arm also knows config 4 (1 real + 64 complex, the reference's own per-chain covariance: 128x128 SVD per step)
CPU_WORKLOADS = dict(WORKLOADS)
CPU_WORKLOADS["c4"] = dict(name="cylinder-style Fourier-mode field: 1 real + 64 complex (reference: per-chain covariance)",
                           temp=0.1, spm=10)
NCU_C2_CAPTURE = "profiles/r02_ncu_c2_k_run_stream_v3.csv"


C4_NAME = ("cylinder-style Fourier-mode field: 1 real + 64 complex, shared proposal covariance (tensor-core L.Z), "
           "32,768 chains per GPU, measure + covariance adaptation every 10 steps")


def _ncu_traffic_per_chain_measure():
    """DRAM bytes per chain-measure of the step kernel from the committed ncu --set full capture
    (profiles/r01_ncu_c2_k_run_v5.csv: a launch of 300 measures x 65,536 chains)."""
    try:
        rd = wr = None
        for line in open(os.path.join(ROOT, NCU_C2_CAPTURE)):
            f = line.strip().split(",")
            if f[0] == "dram__bytes_read.sum":
                rd = float(f[2]) * {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}[f[1]]
            if f[0] == "dram__bytes_write.sum":
                wr = float(f[2]) * {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}[f[1]]
        return (rd + wr) / (300.0 * 65536.0)
    except Exception:
        return None


def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


# ------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU while the timed region runs (NVML)."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            uuid = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(index).uuid)
            except Exception:
                pass
            self.h = None
            if uuid:
                for cand in ("GPU-" + uuid, uuid):
                    try:
                        self.h = pynvml.nvmlDeviceGetHandleByUUID(cand.encode() if hasattr(cand, "encode") else cand)
                        break
                    except Exception:
                        continue
            if self.h is None:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:                               # pragma: no cover
            self.nv, self.err = None, repr(e)

    def _loop(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thr is not None:
            self._thr.join(2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------ CPU baseline
REFERENCE_ROOTS = ("/root/reference", os.path.join(ROOT, "baseline", "_ref"))


def find_reference():
    """Directory holding the unmodified reference package (metropolisengine/metropolis_engine.py), or None."""
    for root in REFERENCE_ROOTS:
        if os.path.exists(os.path.join(root, "metropolisengine", "metropolis_engine.py")):
            return root
    return None


def _import_reference(root):
    """SURVEY.md Appendix C: the reference imports matplotlib / pymbar at module top (statistics.py:2,4) although the
    hot path never uses them; empty stand-ins let the UNMODIFIED package import."""
    import types
    for name in ("matplotlib", "matplotlib.pyplot", "pymbar", "pymbar.timeseries"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.modules["pymbar"].timeseries = sys.modules["pymbar.timeseries"]
    sys.path.insert(0, root)                     # ahead of this repository's own `metropolisengine` import shim
    sys.modules.pop("metropolisengine", None)
    import metropolisengine as ref
    assert os.path.abspath(ref.__file__).startswith(os.path.abspath(root)), ref.__file__
    return ref


def _cpu_chain(wl_key, ref_root):
    """One chain of the workload: the reference's own class when a copy is on the box, else the numpy port."""
    import contextlib
    import io
    import numpy as np
    from oracle import energies as en
    wl = CPU_WORKLOADS[wl_key]
    if wl_key == "c1":
        fn, kw = en.x2, dict(initial_real_params=[0.0], temp=wl["temp"])
    elif wl_key == "c2":
        fn, kw = en.xy_well, dict(initial_real_params=np.array([0., 0.]), temp=wl["temp"])
    elif wl_key == "c3":
        fn, kw = en.mixed_3r4c_bounded, dict(initial_real_params=np.zeros(3),
                                             initial_complex_params=np.zeros(4, dtype=complex), temp=wl["temp"])
    else:                                        # c4: cylinder energy with its hard wall, per-chain covariance (ME:274-302)
        fn, kw = en.make_cylinder(64), dict(initial_real_params=np.array([0.0]),
                                            initial_complex_params=np.zeros(64, dtype=complex), temp=wl["temp"])
    if ref_root is not None:
        ref = _import_reference(ref_root)
        with contextlib.redirect_stdout(io.StringIO()):
            ch = ref.MetropolisEngine(fn, **kw)
        if wl_key == "c4":
            ch.set_reject_condition(en.cylinder_reject)
        return ch, ch.step_all
    from oracle.py_port import PortChain
    ch = PortChain(fn, reject_condition=en.cylinder_reject if wl_key == "c4" else None, **kw)
    return ch, ch.step


def _cpu_worker(args):
    """One process = one chain of the reference's loop (README.md:39-44), timed for `seconds` after a warm-up."""
    wl_key, seed, seconds, fixed_steps, ref_root = args
    os.environ["OMP_NUM_THREADS"] = "1"
    import random
    import numpy as np
    np.random.seed(seed)
    random.seed(seed)
    ch, step = _cpu_chain(wl_key, ref_root)
    spm = CPU_WORKLOADS[wl_key]["spm"]
    for _ in range(3 if wl_key == "c4" else 20):          # warm-up
        for _ in range(spm):
            step()
        ch.measure()
    steps = 0
    series = []                                # first coordinate after every step (for the ESS estimate)
    first = (lambda: float(ch.real_params[0])) if len(ch.real_params) else (lambda: float(ch.complex_params[0].real))
    t0 = time.perf_counter()
    if fixed_steps:
        for _ in range(max(1, fixed_steps // spm)):
            for _ in range(spm):
                step()
                series.append(first())
            ch.measure()
        steps = max(1, fixed_steps // spm) * spm
    else:
        while time.perf_counter() - t0 < seconds:
            for _ in range(spm):
                step()
                series.append(first())
            ch.measure()
            steps += spm
    dt = time.perf_counter() - t0
    from oracle.py_port import statistical_inefficiency
    g = statistical_inefficiency(series[len(series) // 5:]) if len(series) > 2000 else float("nan")
    return steps, dt, g


def cpu_baseline(wl_key, seconds=10.0, fixed_steps=0, procs=None, ref_root="auto"):
    import multiprocessing as mp
    if ref_root == "auto":
        ref_root = find_reference()
    procs = procs or os.cpu_count() or 1
    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    with ctx.Pool(procs) as pool:
        res = pool.map(_cpu_worker, [(wl_key, s, seconds, fixed_steps, ref_root) for s in range(procs)])
    wall = time.perf_counter() - t0
    steps = sum(r[0] for r in res)
    busy = max(r[1] for r in res)
    gs = sorted(r[2] for r in res if r[2] == r[2])
    cpu_baseline.last_g = gs[len(gs) // 2] if gs else float("nan")
    return steps, busy, wall, procs


def _cpu_kind(ref_root):
    if ref_root is not None:
        return "reference", "the unmodified reference class (%s) driven by its README loop" % ref_root
    return "port", "reference not on box: numpy port of the reference loop (oracle/py_port.py, bit-identical to it)"


def c_oracle_rate(wl_key, steps=2_000_000):
    """Single-core throughput of the C restatement (Philox mode) — a much stronger CPU figure than the python loop."""
    import numpy as np
    from oracle import c_oracle as co
    wl = WORKLOADS[wl_key]
    n_r, n_c = wl["n_r"], wl["n_c"]
    o = co.CChain(n_r, n_c, wl["energy"][0], consts=wl["energy"][1:], temp=wl["temp"], x0=np.zeros(n_r + 2 * n_c))
    spm = wl["spm"]
    o.run(100, spm, True, seed=1, chain_id=0)
    t0 = time.perf_counter()
    o.run(steps // spm, spm, True, seed=1, chain_id=0, step0=100 * spm)
    return (steps // spm) * spm / (time.perf_counter() - t0)


# ------------------------------------------------------------------------------------------ reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wl = CPU_WORKLOADS[args.workload]
    ref_root = find_reference()
    kind, what = _cpu_kind(ref_root)
    procs = os.cpu_count() or 1
    # chain-steps per process per bench step: a bounded sample of the workload's own schedule
    per_step = {"c1": 1000, "c2": 1000, "c3": 1000, "c4": 60}[args.workload]
    for _ in range(args.warmup):
        cpu_baseline(args.workload, fixed_steps=per_step, procs=procs, ref_root=ref_root)
    total, t_sum = 0, 0.0
    for _ in range(args.steps):
        steps, busy, wall, _ = cpu_baseline(args.workload, fixed_steps=per_step, procs=procs, ref_root=ref_root)
        total += steps
        t_sum += busy
    value = total / t_sum
    sample = "%d processes x %d chain-steps of the %s schedule per bench step (one chain per process, " \
             "OMP_NUM_THREADS=1); %s" % (procs, per_step, args.workload, what)
    line = {
        "impl": "reference", "metric": "ensemble chain-steps/sec", "value": value, "unit": "chain-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_sum / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["name"], "arm": what},
        "cpu_baseline": {"value": value, "unit": "chain-steps/s", "cores": procs, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "chain-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------ our arm
class Ctx:
    """Process-wide bench context: ranks, device, barrier, max-over-ranks timing."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a GPU: the hot path is CUDA-only (no CPU fallback)")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
        self.stream = torch.cuda.current_stream(self.dev)
        self.n_sm = torch.cuda.get_device_properties(self.dev).multi_processor_count

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()

    def event(self):
        return self.torch.cuda.Event(enable_timing=True)

    def timed(self, fn, steps, warmup):
        """warmup untimed calls, then `steps` calls bracketed by barrier + synchronize; ms (max over ranks)."""
        for _ in range(warmup):
            fn()
        self.barrier()
        a, b = self.event(), self.event()
        a.record(self.stream)
        for _ in range(steps):
            fn()
        b.record(self.stream)
        self.barrier()
        return self.max_over_ranks(a.elapsed_time(b))

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def pipe_model(wl, chains, steps_per_chain, ker_ms, sm_hz, n_sm):
    """Issue-port roofline of the fused step kernel (DESIGN.md §3 "What bounds the step kernel").  Measured on B200: once an
    SM sub-partition holds >= 3 warps of this kernel its throughput no longer grows with the warp count
    (tests/scripts/scale_probe.py) and the time per warp-step follows   inst + fp64_inst + 2.5 * wide_inst + 15 * dmma_inst
    cycles of the sub-partition's issue port — every instruction takes one issue cycle, a warp-wide FP64 instruction holds
    the port a second cycle (64 FP64 lanes per clock and SM = 2 cycles per warp), an IMAD.WIDE (Philox round) about 3.5
    cycles in all (tests/scripts/issue_mix.cu), an FP64 tensor-core mma.m8n8k4 (256 FMA) 16.  The counts cover the whole
    measure period (steps + measure block + per-measure prologue, tests/scripts/sass_period.py), per chain-step.  The
    bound is that cost times the average number of warps per sub-partition."""
    warps = -(-chains // 32) / (4.0 * n_sm)
    cyc = wl["inst"] + wl["fp64_inst"] + 2.5 * wl["wide_inst"] + 15.0 * wl["dmma_inst"]
    bound_ms = 1e3 * warps * steps_per_chain * cyc / sm_hz
    fp64_cycles = 2.0 * wl["fp64_inst"] + 16.0 * wl["dmma_inst"]
    return {"inst_per_chain_step": wl["inst"], "fp64_inst_per_chain_step": wl["fp64_inst"],
            "imad_wide_per_chain_step": wl["wide_inst"], "fp64_mma_per_chain_step": wl["dmma_inst"],
            "issue_cycles_per_warp_step_lower_bound": cyc,
            "warps_per_subpartition": warps, "bound_ms": bound_ms, "frac": bound_ms / ker_ms,
            "fp64_pipe_frac": 1e3 * warps * steps_per_chain * fp64_cycles / sm_hz / ker_ms,
            "how": "issue-port cycles the SASS of one measure period needs, per chain-step (1 per instruction + 1 more per "
                   "FP64 instruction + 2.5 more per IMAD.WIDE + 15 more per FP64 tensor-core MMA; counts from "
                   "tests/scripts/sass_period.py on the shipped library, rarely taken fallback spans left out) x average "
                   "warps per SM sub-partition / measured kernel time; fp64_pipe_frac = FP64-pipe cycles (2 per FP64 "
                   "instruction, 16 per MMA) / measured kernel time, the quantity ncu reports as "
                   "sm__pipe_fp64_cycles_active"}


def fp64_peak_tflops(ctx, lib):
    """FP64 FMA throughput of this GPU, measured now (roofline denominator of the step kernels)."""
    import ctypes
    torch = ctx.torch
    probe_out = torch.empty(ctx.n_sm * 8 * 256, dtype=torch.float64, device=ctx.dev)
    flops = ctypes.c_int64()
    best = None
    for it in range(6):
        a, b = ctx.event(), ctx.event()
        a.record(ctx.stream)
        rc = lib.me_probe_fp64(ctx.local_rank, 20000, ctypes.c_void_p(probe_out.data_ptr()), probe_out.numel(),
                               ctypes.c_void_p(ctx.stream.cuda_stream), ctypes.byref(flops))
        b.record(ctx.stream)
        torch.cuda.synchronize(ctx.dev)
        assert rc == 0
        if it > 0:
            best = a.elapsed_time(b) if best is None else min(best, a.elapsed_time(b))
    return flops.value / (best * 1e-3) / 1e12


def make_engine(ctx, wl, chains_total, record=True, measures=None, seed=2024):
    import numpy as np
    import metropolisengine_b200 as me
    n_r, n_c = wl["n_r"], wl["n_c"]
    d = n_r + 2 * n_c
    ts_cols = d + (3 if (n_r and n_c) else 2)
    per_rank = chains_total // ctx.world
    kw = dict(temp=wl["temp"], n_chains=chains_total, seed=seed, distributed=(ctx.world > 1), device=ctx.dev,
              record=record, ts_chunk_bytes=max(1, (measures or 1) * ts_cols * per_rank * 8))
    if n_r:
        kw["initial_real_params"] = np.zeros(n_r)
    if n_c:
        kw["initial_complex_params"] = np.zeros(n_c, dtype=complex)
    return me.MetropolisEngine(wl["energy"], **kw), ts_cols


def short_fused_pass(ctx, wl_key, fp64_peak, hbm_peak, sm_hz, steps=3, warmup=3):
    """Device-timed passes of one of the other fused BASELINE configs (c1, c3) at its full chain count per GPU."""
    wl = WORKLOADS[wl_key]
    chains, M, spm = wl["chains"], wl["short_measures"], wl["spm"]
    eng, ts_cols = make_engine(ctx, wl, chains * ctx.world, measures=M)
    eng.reserve_rows(M)
    ker = []

    def one():
        eng.clear_time_series(keep_storage=True)
        a, b = ctx.event(), ctx.event()
        a.record(ctx.stream)
        eng.run(M, spm)
        b.record(ctx.stream)
        ker.append((a, b))

    ms = ctx.timed(one, steps, warmup)
    ker_ms = sum(a.elapsed_time(b) for a, b in ker[-steps:]) / steps
    value = chains * ctx.world * M * spm * steps / (ms * 1e-3)
    ts_bytes = M * ts_cols * chains * 8
    tf = chains * M * spm * wl["flop"] / (ker_ms * 1e-3) / 1e12
    rec = {"workload": wl["name"], "value": value, "unit": "chain-steps/s", "ms_per_pass": ms / steps,
           "chains_per_gpu": chains, "steps_per_chain_per_pass": M * spm, "measure_every": spm,
           "kernel": "me::k_run", "kernel_ms": ker_ms, "launch": {"grid": eng._grid, "block": eng._block},
           "roofline": {"bound": "fp64", "achieved": tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac": tf / fp64_peak,
                        "algorithmic": "%d flop + %d special functions per chain-step (SURVEY.md §8d)" % (wl["flop"], wl["sf"]),
                        "pipe": pipe_model(wl, chains, M * spm, ker_ms, sm_hz, ctx.n_sm),
                        "hbm": {"achieved": ts_bytes / (ker_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                "frac": ts_bytes / (ker_ms * 1e-3) / 1e9 / hbm_peak,
                                "bytes_per_chain_measure": 8 * ts_cols}},
           "acceptance_rate": eng.acceptance_rate}
    del eng
    ctx.torch.cuda.empty_cache()
    return rec


def per_chain_large_pass(ctx, hbm_peak, steps=3, warmup=2, chains=32768, measures=10):
    """The reference's OWN algorithm at the cylinder shape: 1 real + 64 complex with a covariance per chain (ME:274-302), the
    runtime-shape kernel (me_generic.cu, gk_run: one launch per schedule).  HBM-bound: every step streams the chain's 64 x 64
    complex factor (8 n_c^2 = 32,768 B) plus the parameter / proposal / normal vectors."""
    import numpy as np
    import metropolisengine_b200 as me
    spm, nc = 10, 64
    eng = me.MetropolisEngine(me.BuiltinEnergy("cylinder", 10.0, -1.0, 0.05, 1.0, reject=True),
                              initial_real_params=np.array([0.0]), initial_complex_params=np.zeros(nc, dtype=complex),
                              temp=.1, n_chains=chains * ctx.world, seed=5, record=False, distributed=(ctx.world > 1),
                              device=ctx.dev, sampling_width=0.02)
    eng.run(55, 2)                       # past the 50th measure: per-chain covariances and their Cholesky factors are live
    ms = ctx.timed(lambda: eng.run(measures, spm), steps, warmup)
    value = chains * ctx.world * measures * spm * steps / (ms * 1e-3)
    d = 1 + 2 * nc
    bytes_step = 8.0 * (nc * nc + 7 * d)             # factor + x, z (w+r), proposal (w+r+r), state write-back on accept
    gbs = chains * measures * spm * steps * bytes_step / (ms * 1e-3) / 1e9
    rec = {"workload": "1 real + 64 complex, PER-CHAIN covariance (the reference's algorithm at the cylinder shape), %d chains "
                       "per GPU, measure (64 x 64 complex Cholesky per chain) every 10 steps" % chains,
           "value": value, "unit": "chain-steps/s", "ms_per_pass": ms / steps, "kernel": "gk_run",
           "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                        "traffic": None,
                        "algorithmic": "%d B per chain-step (8 n_c^2 factor stream + 7 vectors of D doubles); the per-measure "
                                       "Cholesky (O(n_c^3) per chain, operands in global memory) is inside the timed pass"
                                       % int(bytes_step)},
           "acceptance_rate": eng.acceptance_rate}
    del eng
    ctx.torch.cuda.empty_cache()
    return rec


def c4_pass(ctx, peaks, steps=3, warmup=3, measures=100, dump=None):
    """BASELINE config 4: 1 real + 64 complex, shared proposal covariance, 32,768 chains per GPU; tcgen05 path.  One pass =
    `measures` x (10 x step_all() + measure()), the pooled-covariance update (and, for N > 1, its moment all-reduce)
    at every measure.  `dump`: directory for dump_outputs() after the timed passes."""
    import metropolisengine_b200 as me
    torch = ctx.torch
    chains, M, spm = 32768, measures, 10
    eng = me.SharedCovarianceEngine(energy_consts=(10.0, -1.0, 0.05, 1.0), temp=.1, n_chains=chains * ctx.world, seed=2024,
                                    record=False, distributed=(ctx.world > 1), device=ctx.dev)
    eng.run(60, spm)                      # past the 50th measure: the shared covariance is live
    l0 = [0]

    def one():
        eng.run(M, spm)

    for _ in range(warmup):
        one()
    ctx.barrier()
    l0[0] = eng.launch_count
    ms = ctx.timed(one, steps, 0)
    launches = eng.launch_count - l0[0]
    if dump:
        dump_outputs(dump, eng, {"covariance_matrix_real": eng.covariance_matrix_real,
                                 "covariance_matrix_complex": eng.covariance_matrix_complex})
    value = chains * ctx.world * M * spm * steps / (ms * 1e-3)
    a, b = ctx.event(), ctx.event()
    a.record(ctx.stream)
    eng.step(200)
    b.record(ctx.stream)
    torch.cuda.synchronize(ctx.dev)
    ker_ms = a.elapsed_time(b)
    tf_peak = peaks.get("bf16_tflops", 1590.0)
    tf = chains * 200 * 2.0 * 128 * 128 / (ker_ms * 1e-3) / 1e12
    rec = {"workload": C4_NAME, "value": value, "unit": "chain-steps/s", "ms_per_pass": ms / steps,
           "chains_per_gpu": chains, "measures_per_pass": M, "measure_every": spm, "gpu_launches": launches,
           "dtype": "f64 state/energy/accept, bf16 proposal contraction (fp32 accumulate)",
           "kernel": "k4_steps", "kernel_ms_per_step": ker_ms / 200,
           "step_kernel_only_chain_steps_per_s": chains * 200 / (ker_ms * 1e-3),
           "roofline": {"bound": "tensor", "achieved": tf, "peak": tf_peak, "unit": "TFLOP/s", "frac": tf / tf_peak,
                        "traffic": None,
                        "algorithmic": "2*128*128 flop per chain-step in the L.Z contraction (SURVEY.md §8d C4); the step "
                                       "kernel is bound by in-kernel Gaussian generation and the FP64 epilogue, not by "
                                       "the tensor pipe",
                        "peak_source": "MEASURED_PEAKS.json bf16_tflops" if peaks else "fallback 1590"},
           "parallelism": "chains sharded over %d GPU(s); 8,328-double moment all-reduce at every measure" % ctx.world,
           "acceptance_rate": eng.acceptance_rate}
    del eng
    torch.cuda.empty_cache()
    return rec


def c5_pass(ctx, steps=3, warmup=3, total_chains=1 << 20, launches=20):
    """BASELINE config 5 (strong scaling): 2^20 xy-well chains in TOTAL sharded over the ranks, 100 steps per launch
    (10 x (10 steps + measure)), pooled-moment reduction + all-reduce across ranks after EVERY launch, issued inside
    the library; each launch is one CUDA-graph replay (run_graphed)."""
    from metropolisengine_b200 import parallel
    wl = WORKLOADS["c2"]
    eng, _ = make_engine(ctx, wl, total_chains, record=False, seed=7)
    M, spm = 10, 10
    eng.run_graphed(M, spm, launches)        # eager (allocations, communicator)
    eng.run_graphed(M, spm, launches)        # capture + first replay

    def one():
        eng.run_graphed(M, spm, launches)

    ms = ctx.timed(one, steps, warmup)
    value = total_chains * M * spm * launches * steps / (ms * 1e-3)
    ps = eng.pooled_statistics()

    def eager():
        for _ in range(launches):
            eng.run(M, spm)
            eng._flush_pool()

    ms_e = ctx.timed(eager, steps, 1)
    rec = {"workload": "config 5: %d xy-well chains in total over %d GPU(s), 100 steps per launch, pooled-moment "
                       "all-reduce after every launch" % (total_chains, ctx.world),
           "scaling": "strong", "value": value, "unit": "chain-steps/s", "us_per_launch": 1e3 * ms / (steps * launches),
           "chains_total": total_chains, "chains_per_gpu": total_chains // ctx.world, "launches_per_pass": launches,
           "how": "one CUDA graph per pass: %d x [me_run -> me_reduce_stats (fixed-order reduction of the per-CTA rows) -> "
                  "me_accumulate_stats on a side stream (NCCL all-reduce inside the library, device-resident totals), which "
                  "overlaps the next me_run]; one D2H of the totals at the end" % launches,
           "collective": ("one-shot sum over NVLink peer windows (me_comm_peer_*)" if parallel.peer_windows_on(eng._library_comm())
                          else ("NCCL all-reduce inside the library" if ctx.world > 1 else "none (one rank)")),
           "eager_value": total_chains * M * spm * launches * steps / (ms_e * 1e-3),
           "pooled_var_x0": float(ps["cov_real"][0, 0]), "pooled_count": ps["count"]}
    del eng
    ctx.torch.cuda.empty_cache()
    return rec


# per-chain state and time-series samples; with the pooled statistics the dump stays well under 64 MB
DUMP_STATE_BYTES, DUMP_TS_BYTES = 24 << 20, 32 << 20


def _sorted_sample(rng, n, k):
    import numpy as np
    return np.arange(n) if k >= n else np.sort(rng.choice(n, k, replace=False))


def dump_outputs(out_dir, eng, extra):
    """Write what the timed path handed its caller after its last step as float64 ``out_dir/<name>.npy``: the per-chain
    state block ``state`` [words, chains] (parameters, energy, widths, means, covariances, counters), the recorded rows
    ``time_series`` [rows, columns, chains] and the arrays of ``extra`` (complex values get a trailing [re, im] axis,
    scalars become shape (1,), empty arrays are not written).
    Chains (and, for very long series, rows) are a fixed seeded sample sized to the byte budgets above; the sampled
    indices are written beside the arrays (``state_chains``, ``time_series_chains``, ``time_series_rows``)."""
    import numpy as np
    import torch
    rng = np.random.default_rng(0)
    words, n = eng.state.shape
    chains = _sorted_sample(rng, n, DUMP_STATE_BYTES // (8 * words))
    out = {"state": eng.state[:, torch.as_tensor(chains, device=eng.state.device)], "state_chains": chains}
    ts = eng.time_series()
    if ts.shape[0]:
        rows, row_bytes = ts.shape[0], 8 * ts.shape[1]
        ts_chains = chains[_sorted_sample(rng, len(chains), max(1, DUMP_TS_BYTES // (row_bytes * rows)))]
        ts_rows = _sorted_sample(rng, rows, DUMP_TS_BYTES // (row_bytes * len(ts_chains)))
        sub = ts.index_select(2, torch.as_tensor(ts_chains, device=ts.device))
        out.update(time_series=sub[torch.as_tensor(ts_rows, device=ts.device)], time_series_chains=ts_chains,
                   time_series_rows=ts_rows)
    out.update(extra)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        a = np.atleast_1d(np.asarray(a.cpu() if isinstance(a, torch.Tensor) else a))
        if a.size == 0:                   # e.g. complex statistics of an all-real workload: nothing was computed
            continue
        if np.iscomplexobj(a):
            a = np.stack([a.real, a.imag], axis=-1)
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def run_ours(args):
    import ctypes
    import hashlib
    import numpy as np
    import metropolisengine_b200 as me  # noqa: F401

    ctx = Ctx()
    torch, dist = ctx.torch, ctx.dist
    world, rank, dev, stream = ctx.world, ctx.rank, ctx.dev, ctx.stream
    if args.gpus != world and rank == 0:
        print("bench.py: --gpus %d but WORLD_SIZE=%d; the launcher's world size is used" % (args.gpus, world),
              file=sys.stderr)

    wl = WORKLOADS[args.workload]
    chains, M, spm = wl["chains"], wl["measures"], wl["spm"]
    if args.measures:
        M = args.measures
    n_r, n_c = wl["n_r"], wl["n_c"]
    d = n_r + 2 * n_c
    eng, ts_cols = make_engine(ctx, wl, chains * world, measures=M)
    ts_bytes = M * ts_cols * chains * 8
    eng.reserve_rows(M)
    lay = eng._lay

    def one_pass():
        """One pass of the job on resident state: fused step/measure launch + pooled-moment reduction and its
        all-reduce across ranks (the path's only collective, inside the library: me_allreduce_stats)."""
        eng.clear_time_series(keep_storage=True)
        eng.run(M, spm)
        eng._flush_pool()

    # ---- value: device-timed, inputs resident
    for _ in range(args.warmup):
        one_pass()
    ctx.barrier()
    launches0 = eng.launch_count
    ker_ev = []
    ev0, ev1 = ctx.event(), ctx.event()
    with ClockSampler(ctx.local_rank) as clocks:
        ctx.barrier()      # the sampler's NVML start-up takes milliseconds and differs per process: line the ranks up
        ev0.record(stream) # again so that no rank's timed region contains another rank's start-up
        for _ in range(args.steps):
            a, b = ctx.event(), ctx.event()
            eng.clear_time_series(keep_storage=True)
            a.record(stream)
            eng.run(M, spm)
            b.record(stream)
            ker_ev.append((a, b))
            eng._flush_pool()
        ev1.record(stream)
        ctx.barrier()
    launches = eng.launch_count - launches0
    if args.dump_outputs:
        ps = eng.pooled_statistics()          # collective when sharded: every rank must call it
        if rank == 0:
            dump_outputs(args.dump_outputs, eng, {"pooled_" + k: v for k, v in ps.items()})
    ms_total = ctx.max_over_ranks(ev0.elapsed_time(ev1))
    chain_steps_per_pass = chains * world * M * spm
    value = chain_steps_per_pass * args.steps / (ms_total * 1e-3)
    ker_ms = sum(a.elapsed_time(b) for a, b in ker_ev) / len(ker_ev)
    # per-rank view of the timed region (a straggler GPU — e.g. one that is power-capped when all eight run FP64 flat
    # out — sets the job's time through the per-step all-reduce): kernel time and clocks of every rank
    rank_view = None
    if world > 1:
        mine = {"rank": rank, "kernel_ms": ker_ms, "clocks": clocks.summary()}
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        rank_view = gathered

    # ---- e2e: public API with host buffers, copies inside the timed region
    pin_r = torch.zeros((chains, n_r), dtype=torch.float64).pin_memory() if n_r else None
    pin_c = torch.zeros((chains, n_c), dtype=torch.complex128).pin_memory() if n_c else None
    host_state = torch.empty((lay.WORDS, chains), dtype=torch.float64).pin_memory()
    host_ts0 = torch.empty((M, ts_cols), dtype=torch.float64).pin_memory()
    h2d = (pin_r.numel() * 8 if n_r else 0) + (pin_c.numel() * 16 if n_c else 0)
    d2h = host_state.numel() * 8 + host_ts0.numel() * 8 + (lay.POOL_WORDS + 1) * 8

    def e2e_pass():
        eng.reset(initial_real_params=pin_r, initial_complex_params=pin_c)        # H2D + re-initialisation
        eng.run(M, spm)
        ps = eng.pooled_statistics()                                               # reduce (+all-reduce) + D2H
        host_state.copy_(eng.state, non_blocking=True)                            # final per-chain state D2H
        host_ts0.copy_(eng.time_series()[:, :, 0], non_blocking=True)             # chain 0 series (df) D2H
        torch.cuda.synchronize(dev)
        return ps

    e2e_steps = max(1, min(args.steps, 3 if args.steps > 3 else args.steps))
    e2e_pass()
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ps = e2e_pass()
    ctx.barrier()
    e2e_s = ctx.max_over_ranks(time.perf_counter() - t0)
    e2e_value = chain_steps_per_pass * e2e_steps / e2e_s
    # invariance digest: global chains 0..255 (always on rank 0) after exactly one pass from the initial state
    digest = hashlib.sha256(host_state[:, :256].contiguous().numpy().tobytes()).hexdigest() if rank == 0 else None

    fp64_peak = fp64_peak_tflops(ctx, eng._lib)
    acc_rate = eng.acceptance_rate            # collective when sharded: every rank must call it

    # ---- ESS: statistical inefficiency per STEP from a side ensemble measured at every step (device kernel)
    g_steps = None
    if rank == 0:
        import metropolisengine_b200 as me2
        kw2 = dict(temp=wl["temp"], n_chains=4096, seed=2024, device=dev, ts_chunk_bytes=4096 * ts_cols * 8 * 6000)
        if n_r:
            kw2["initial_real_params"] = np.zeros(n_r)
        if n_c:
            kw2["initial_complex_params"] = np.zeros(n_c, dtype=complex)
        side = me2.MetropolisEngine(wl["energy"], **kw2)
        side.record = False
        side.run(300, 10)                     # sigma / covariance adaptation
        side.record = True
        side.run(6000, 1)
        gq = torch.stack([side.statistical_inefficiency(column=c, n_chains=1024, burn_in=0.2) for c in range(d)])
        g_steps = float(gq.max(dim=0).values.median().item())      # worst coordinate per chain, median over chains
        del side

    peaks = _peaks() or {}
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    clk = clocks.summary()
    sm_hz = 1e6 * (clk.get("sm_mhz") or 1965)
    grid_block = {"grid": eng._grid, "block": eng._block}
    del eng, host_ts0
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs, short passes in the same line (every rank takes part)
    sub = {}
    if not args.no_workloads:
        for key in ("c1", "c3"):
            if key != args.workload:
                sub[key] = short_fused_pass(ctx, key, fp64_peak, hbm_peak, sm_hz)
        sub["c4"] = c4_pass(ctx, peaks)
        sub["c4_per_chain_covariance"] = per_chain_large_pass(ctx, hbm_peak)
        sub["c5_2^20_chains_total"] = c5_pass(ctx)

    if rank != 0:
        ctx.close()
        return 0

    per_launch_steps = chains * M * spm
    achieved_tf = per_launch_steps * wl["flop"] / (ker_ms * 1e-3) / 1e12
    ts_gbs = ts_bytes / (ker_ms * 1e-3) / 1e9
    pipe = pipe_model(wl, chains, M * spm, ker_ms, sm_hz, ctx.n_sm)
    tpm = _ncu_traffic_per_chain_measure() if args.workload == "c2" else None
    line = {
        "metric": "ensemble chain-steps/sec", "value": value, "unit": "chain-steps/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["name"], "chains_per_gpu": chains, "steps_per_chain_per_bench_step": M * spm,
                   "measure_every": spm, "chain_steps_per_bench_step": chain_steps_per_pass,
                   "time_series_bytes_per_bench_step_per_gpu": ts_bytes,
                   "l2": "outputs (%.1f GB per step) exceed L2; state is register-resident" % (ts_bytes / 1e9),
                   "parallelism": "chains sharded over %d GPU(s); pooled-moment all-reduce per bench step "
                                  "(me_allreduce_stats: NCCL inside the library)" % world,
                   "launch": grid_block},
        "e2e": {"value": e2e_value, "unit": "chain-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps, "what": "reset() from pinned host params, run(), pooled_statistics(), D2H of the "
                                            "final per-chain state and of chain 0's time series (the 21 GB of rows of "
                                            "the other chains stay on the device)"},
        "gpu_launches": launches,
        "roofline": {"bound": "fp64", "achieved": achieved_tf, "peak": fp64_peak, "unit": "TFLOP/s",
                     "frac": achieved_tf / fp64_peak,
                     "traffic": None,
                     "traffic_ncu_capture": ({"bytes_per_chain_measure": tpm, "algorithmic_bytes_per_chain_measure": 8 * ts_cols,
                                              "source": NCU_C2_CAPTURE + ": dram__bytes_read.sum + dram__bytes_write.sum of one "
                                                        "ncu --set full capture of this kernel (300 measures x 65,536 chains); "
                                                        "NOT measured in this run, hence traffic = null"} if tpm else None),
                     "pipe": pipe,
                     "kernel": "me::k_run", "kernel_ms": ker_ms,
                     "algorithmic": "%d flop + %d special functions per chain-step (SURVEY.md §8d); special functions "
                                    "and Philox integer work are NOT counted in achieved" % (wl["flop"], wl["sf"]),
                     "peak_source": "me_probe_fp64 (FP64 FMA, measured in this run)",
                     "hbm": {"achieved": ts_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ts_gbs / hbm_peak,
                             "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650"}},
        "clocks": clk,
        "ranks": rank_view,
        "check": {"acceptance_rate": acc_rate, "pooled_var_x0": float(ps["cov_real"][0, 0]) if n_r else None,
                  "invariance": {"sha256_state_of_global_chains_0_255_after_one_pass": digest,
                                 "how": "state block [words, 256] of rank 0 after reset() + one pass; the same at every N"}},
        "ess": {"g_steps": g_steps, "ess_per_sec": value / g_steps if g_steps else None,
                "how": "statistical inefficiency per step (pymbar's definition, worst coordinate, median of 1024 "
                       "chains, 6000 consecutive steps after adaptation), device kernel me_statistical_inefficiency"},
        "workloads": sub,
    }
    # ---- CPU baseline on this box's host cores (bounded sample)
    if not args.no_cpu:
        ref_root = find_reference()
        kind, what = _cpu_kind(ref_root)
        steps, busy, wall, procs = cpu_baseline(args.workload, seconds=args.cpu_seconds, ref_root=ref_root)
        line["cpu_baseline"] = {
            "value": steps / busy, "unit": "chain-steps/s", "cores": procs, "kind": kind,
            "sample": "%d processes x %.0f s of the same schedule, one chain each (OMP_NUM_THREADS=1); %s"
                      % (procs, args.cpu_seconds, what),
            "c_oracle_1core": c_oracle_rate(args.workload),
            "g_steps": cpu_baseline.last_g,
            "ess_per_sec": (steps / busy) / cpu_baseline.last_g if cpu_baseline.last_g == cpu_baseline.last_g else None,
        }
    print(json.dumps(line))
    ctx.close()
    return 0


def run_c4(args):
    """--workload c4 as the headline line (BASELINE config 4)."""
    ctx = Ctx()
    peaks = _peaks() or {}
    with ClockSampler(ctx.local_rank) as clocks:
        rec = c4_pass(ctx, peaks, steps=args.steps, warmup=args.warmup, measures=(args.measures or 100),
                      dump=args.dump_outputs if ctx.rank == 0 else None)
    if ctx.rank != 0:
        ctx.close()
        return 0
    line = {
        "metric": "ensemble chain-steps/sec", "value": rec["value"], "unit": "chain-steps/s", "n_gpus": ctx.world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": rec["ms_per_pass"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": rec["dtype"], "data": "synthetic",
        "config": {"workload": C4_NAME, "chains_per_gpu": rec["chains_per_gpu"],
                   "measures_per_bench_step": rec["measures_per_pass"], "measure_every": rec["measure_every"]},
        "gpu_launches": rec["gpu_launches"], "roofline": rec["roofline"], "clocks": clocks.summary(),
        "check": {"acceptance_rate": rec["acceptance_rate"]},
        "step_kernel_only_chain_steps_per_s": rec["step_kernel_only_chain_steps_per_s"],
    }
    if not args.no_cpu:
        ref_root = find_reference()
        kind, what = _cpu_kind(ref_root)
        steps, busy, wall, procs = cpu_baseline("c4", seconds=args.cpu_seconds, ref_root=ref_root)
        line["cpu_baseline"] = {"value": steps / busy, "unit": "chain-steps/s", "cores": procs, "kind": kind,
                                "sample": "%d processes x %.0f s, one chain each with the reference's per-chain covariance "
                                          "(ME:274-302); %s" % (procs, args.cpu_seconds, what)}
    print(json.dumps(line))
    ctx.close()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS) + ["c4"])
    ap.add_argument("--measures", type=int, default=0, help="override measures per bench step (debug)")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-workloads", action="store_true", help="skip the c1/c3/c4/c5 sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float64, under 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3                                   # timing rule: W >= 3
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "c4":
        return run_c4(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())

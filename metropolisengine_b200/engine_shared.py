"""Shared-covariance ensemble engine for large parameter spaces (BASELINE config 4: cylinder-style field with 1 real
amplitude + n_c complex Fourier coefficients, n_c = 8, 16, 32 or 64), driving the warp-specialised tcgen05 kernel of
csrc/me_k4_device.cuh.

Same public surface as ``MetropolisEngine`` (reference metropolisengine/metropolis_engine.py: ``step_all`` ME:241-259,
``measure`` ME:342-356, ``real_mean`` / ``complex_mean`` / ``covariance_matrix_*`` / ``observables_mean`` /
``save_time_series`` / ``df``), with one difference that north_star asks for: the proposal covariance of the complex
block is *pooled over the ensemble* and shared by all chains.  It is the running covariance of every (chain, measure)
sample so far plus the reference's ``sigma^2/n`` regulariser (ME:418,425), used from the 50th measure on (ME:389,396);
across GPUs its moments are summed with one NCCL all-reduce per measure (the path's only collective).

Work per measure (all stream-ordered, no host sync): per-chain means / observable means / time-series row
(me_k4_measure); pooled moments as a symmetric rank-k update (me_k4_moments); covariance + 64x64 complex Cholesky + BF16
re-packing of the factor into the UMMA operand layout (me_k4_refactor).  The factor refresh is a one-CTA kernel, so by
default it runs on a SIDE stream beside the next block of steps (the step kernel leaves one SM free): the steps after
measure b use the factor of measure b-1.  The lag is deterministic and only shapes the (symmetric) proposal;
``async_refresh=False`` gives the strictly sequential schedule.
"""
import ctypes
import math

import numpy as np
import torch

from . import _lib
from . import parallel
from .engine import adaptation_constants, _ptr

N_C = 64          # default number of complex parameters (BASELINE config 4)


class SharedEnergy:
    """User energy functor of the shared-covariance path (the reference's plugin surface, ME:20, 110-120).  ``source``
    is CUDA C++ defining the per-mode contributions to two sums and the total (include/me_b200.h, me_k4_set_energy_source)::

        __device__ void   me_k4_mode(double q, double re, double im, const double* k, double& s0, double& s1);  // q = j - n_c/2
        __device__ double me_k4_total(double a, double s0, double s1, const double* k, int n_c);
        __device__ bool   me_k4_reject(double a, const double* k);          // only when has_reject=True

    i.e. energies E = total(a, sum_j f0_j(c_j), sum_j f1_j(c_j)); compiled by NVRTC into the same tcgen05 step kernel."""

    def __init__(self, source, consts=(), has_reject=False):
        self.source, self.consts, self.has_reject = source, tuple(float(c) for c in consts), bool(has_reject)


class SharedCovarianceEngine:
    def mbar(self, *args, **kwargs):
        """MBAR passes run on the per-chain engine's fused shapes only (``MetropolisEngine.mbar``)."""
        raise NotImplementedError("MBAR is not available for shared-covariance engines")

    def __init__(self, energy_consts=(10.0, -1.0, 0.05, 1.0), reject_condition=True, initial_real_params=None,
                 initial_complex_params=None, sampling_width=0.05, covariance_matrix_real=None,
                 covariance_matrix_complex=None, params_names=None, target_acceptance=.3, temp=0, *, n_chains=128,
                 seed=0, device=None, record=True, distributed=False, ts_chunk_rows=64, async_refresh=True,
                 energy=None, n_complex=None):
        """``energy_consts`` = (kappa, alpha, gamma, beta) of the built-in cylinder-style energy (SURVEY.md §8d C4);
        ``reject_condition=True`` enables its hard wall ``|a| >= 1`` (legacy metropolis_engine.py:103,139).
        ``energy``: a ``SharedEnergy`` (user CUDA functor) instead of the built-in one.  The number of complex parameters
        (8, 16, 32 or 64) is taken from ``initial_complex_params`` (or ``n_complex``; default 64)."""
        if not torch.cuda.is_available():
            raise RuntimeError("SharedCovarianceEngine needs a CUDA device: the hot path is CUDA-only (no CPU fallback)")
        if temp is None or not temp >= 0:
            raise AssertionError("temp must be >= 0")                                        # ME:92
        self._lib = _lib.load()
        self.launch_count = 0
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        xr = np.zeros(1) if initial_real_params is None else np.asarray(initial_real_params, dtype=np.float64)
        nc = int(n_complex) if n_complex is not None else (N_C if initial_complex_params is None
                                                           else np.asarray(initial_complex_params).shape[-1])
        xc = (np.zeros(nc, dtype=np.complex128) if initial_complex_params is None
              else np.asarray(initial_complex_params, dtype=np.complex128))
        if xr.shape[-1] != 1 or xc.shape[-1] != nc or nc not in (8, 16, 32, 64):
            raise ValueError("the shared-covariance path serves 1 real + 8 / 16 / 32 / 64 complex parameters")
        self._nc = nc
        lay = _lib.MeK4Layout()
        self._lib.me_k4_layout_for(nc, ctypes.byref(lay))
        self._lay = lay
        self.num_real_params, self.num_complex_params = 1, nc
        self.n_chains_total = int(n_chains)
        self._rank, self._world = (parallel.world() if distributed else (0, 1))
        lo, hi = parallel.shard_range(self.n_chains_total, self._rank, self._world)
        self.chain_offset, self.n_chains = lo, hi - lo
        self._distributed = bool(distributed) and self._world > 1
        self._comm = None            # library-side communicator (me_comm) of the moment all-reduce, created on first use
        self.temp, self.target_acceptance = temp, target_acceptance
        self.alpha, self.m, self.ratio = adaptation_constants(1, nc, target_acceptance)
        self.params_names = list(params_names) if params_names else ["param_" + str(i) for i in range(1 + nc)]
        self.observables_names = ["abs_param_" + str(i) for i in range(1 + nc)] + ["param_0_squared"]
        self.seed = int(seed)
        self.df = None
        cfg = _lib.MeK4Config(1, nc, self.n_chains, self.chain_offset, float(temp), float(target_acceptance),
                              self.ratio, self.seed, self.device.index, int(bool(reject_condition)),
                              (ctypes.c_double * 4)(*[float(c) for c in energy_consts]))
        h = ctypes.c_void_p()
        rc = self._lib.me_k4_create(ctypes.byref(cfg), ctypes.byref(h))
        if rc != 0:
            msg = self._lib.me_k4_last_error(None).decode()
            raise ValueError(msg) if rc == _lib.ME_ERR_INVALID else _lib.MeError(msg)
        self._h = h
        if energy is not None:
            if not isinstance(energy, SharedEnergy):
                raise TypeError("energy must be a SharedEnergy (CUDA functor of the shared-covariance path)")
            consts = (ctypes.c_double * max(len(energy.consts), 1))(*energy.consts)
            self._check(self._lib.me_k4_set_energy_source(self._h, energy.source.encode(), consts, len(energy.consts),
                                                          int(energy.has_reject)))
        dev, f64 = self.device, torch.float64
        self.state = torch.zeros((lay.WORDS, self.n_chains), dtype=f64, device=dev)
        # factor / s_a are triple-buffered: one pair is read by the step kernel, one holds the finished refresh that the
        # next launch adopts, one is being written by the refresh in flight
        self._factors = [torch.zeros((2 * nc // 8, 2 * nc, 8), dtype=torch.bfloat16, device=dev) for _ in range(3)]
        self._s_as = [torch.ones(1, dtype=f64, device=dev) for _ in range(3)]
        self._cur = 0
        self._factor, self._s_a = self._factors[0], self._s_as[0]
        self._async = bool(async_refresh)
        self._side = torch.cuda.Stream(device=dev) if self._async else None
        self._in_flight = None          # (event, buffer index) of the refresh launched at the last measure
        self._ready = None              # ... of the one before: adopted by the next step launch
        self._refresh_count = 0
        self._last_accept = torch.zeros(self.n_chains, dtype=torch.uint8, device=dev)
        self._check(self._lib.me_k4_bind(self._h, _ptr(self.state), _ptr(self._factor), _ptr(self._last_accept)))
        # shared covariances (ME:63-70): identity unless given
        self._cov_c = (torch.eye(nc, dtype=torch.complex128, device=dev) if covariance_matrix_complex is None
                       else torch.as_tensor(np.asarray(covariance_matrix_complex, dtype=np.complex128),
                                            device=dev).contiguous())
        self._cov_a = torch.ones(1, dtype=f64, device=dev) if covariance_matrix_real is None else \
            torch.as_tensor(np.asarray(covariance_matrix_real, dtype=np.float64).reshape(1), device=dev)
        self._install_factor()
        # pooled running moments about a fixed shift (the initial ensemble mean)
        x0 = np.concatenate([xr.reshape(-1)[:1] if xr.ndim == 1 else [xr[:, 0].mean()],
                             (xc if xc.ndim == 1 else xc.mean(0)).real, (xc if xc.ndim == 1 else xc.mean(0)).imag])
        self._shift = torch.as_tensor(np.ascontiguousarray(x0), dtype=f64, device=dev)
        n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
        self._scratch = torch.zeros((n_sm + 1) * lay.MOM_SCRATCH_PER_SM, dtype=f64, device=dev)
        self._incs = [torch.zeros(lay.MOM_WORDS, dtype=torch.complex128, device=dev) for _ in range(2)]
        self._inc_full = self._incs[0]          # increment of the latest measure
        self._measure_count = 0
        self._mom = torch.zeros(4 + nc + nc * nc, dtype=torch.complex128, device=dev)   # count, -, sum a, sum a^2, sum c, sum c c^H
        self._snaps = [torch.zeros(lay.MOM_WORDS + 2, dtype=torch.complex128, device=dev) for _ in range(2)]
        self._snap_events = [None, None]
        if self._async:
            self._check(self._lib.me_k4_set_reserved_sms(self._h, 1))
        self._inc = torch.zeros(2, dtype=torch.complex128, device=dev)
        self._psd_status = torch.zeros(1, dtype=torch.int32, device=dev)
        if self._distributed:              # collective set-up (every rank constructs its engine)
            self._comm = parallel.library_comm(self._lib, dev.index) or False
        per_chain = xr.ndim == 2 or xc.ndim == 2
        if per_chain:
            full = np.zeros((lay.D, self.n_chains_total))
            full[0] = xr[:, 0] if xr.ndim == 2 else xr[0]
            full[1:1 + nc] = xc.real.T if xc.ndim == 2 else xc.real[:, None]
            full[1 + nc:] = xc.imag.T if xc.ndim == 2 else xc.imag[:, None]
            x0_dev = torch.tensor(np.ascontiguousarray(full[:, lo:hi]), dtype=f64, device=dev)
        else:
            x0_dev = torch.tensor(x0, dtype=f64, device=dev)
        self._sampling_width0 = float(sampling_width)
        self._launch(self._lib.me_k4_init(self._h, _ptr(x0_dev), 0 if per_chain else 1, self._sampling_width0,
                                          self._stream()))
        self.record = bool(record)
        self._ts_chunks, self._ts_chunk_rows = [], int(ts_chunk_rows)

    @classmethod
    def from_reference_arguments(cls, energy_functions, reject_condition=None, initial_real_params=None,
                                 initial_complex_params=None, sampling_width=0.05, covariance_matrix_real=None,
                                 covariance_matrix_complex=None, params_names=None, target_acceptance=.3, temp=0,
                                 complex_sample_method="multivariate-gaussian", **kw):
        """``MetropolisEngine(..., adapt="pooled")``: the reference's constructor arguments (ME:17) mapped onto this
        engine.  The energy must be the cylinder-style device functor (``("cylinder", kappa, alpha, gamma, beta)`` or
        ``BuiltinEnergy("cylinder", ...)``); its hard wall is switched on by ``BuiltinEnergy(..., reject=True)``."""
        from .engine import BuiltinEnergy
        e = energy_functions
        if isinstance(e, str):
            e = BuiltinEnergy(e)
        elif isinstance(e, tuple) and e and isinstance(e[0], str):
            e = BuiltinEnergy(e[0], *e[1:])
        if reject_condition is not None:
            raise NotImplementedError("adapt='pooled': put the hard wall in the functor (BuiltinEnergy(reject=True) / "
                                      "SharedEnergy(has_reject=True))")
        for k in ("strict", "callable_layout", "graph_callable", "ts_chunk_bytes", "_shard"):
            kw.pop(k, None)
        if isinstance(e, SharedEnergy):
            return cls(energy=e, reject_condition=e.has_reject, initial_real_params=initial_real_params,
                       initial_complex_params=initial_complex_params, sampling_width=sampling_width,
                       covariance_matrix_real=covariance_matrix_real, covariance_matrix_complex=covariance_matrix_complex,
                       params_names=params_names, target_acceptance=target_acceptance, temp=temp, **kw)
        if not isinstance(e, BuiltinEnergy) or e.name != "cylinder":
            raise NotImplementedError("adapt='pooled' (shared proposal covariance on the tensor cores) serves the "
                                      "cylinder-style device functor or a SharedEnergy; other energies use "
                                      "adapt='per_chain'")
        consts = e.consts if len(e.consts) == 4 else (10.0, -1.0, 0.05, 1.0)
        return cls(energy_consts=consts, reject_condition=e.reject, initial_real_params=initial_real_params,
                   initial_complex_params=initial_complex_params, sampling_width=sampling_width,
                   covariance_matrix_real=covariance_matrix_real, covariance_matrix_complex=covariance_matrix_complex,
                   params_names=params_names, target_acceptance=target_acceptance, temp=temp, **kw)

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, rc):
        if rc != 0:
            msg = self._lib.me_k4_last_error(self._h).decode()
            raise ValueError(msg) if rc == _lib.ME_ERR_INVALID else _lib.MeError(msg)

    def _launch(self, rc):
        self._check(rc)
        self.launch_count += 1

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None:
            self._lib.me_k4_destroy(h)
            self._h = None

    def _install_factor(self):
        """C_c = G G^H -> real embedding of conj(G)/sqrt2 in interleaved (Re, Im) coordinates -> BF16 in the UMMA
        canonical K-major layout [k-chunk][n][8]; s_a = sqrt(C_a).  Stream-ordered, no host sync."""
        G = torch.linalg.cholesky_ex(self._cov_c)[0]
        gr, gi = G.real / math.sqrt(2.0), G.imag / math.sqrt(2.0)
        n2 = 2 * self._nc
        B = torch.zeros((n2, n2), dtype=torch.float64, device=self.device)
        B[0::2, 0::2] = gr
        B[0::2, 1::2] = gi
        B[1::2, 0::2] = -gi
        B[1::2, 1::2] = gr
        self._B = B
        for f, sa in zip(self._factors, self._s_as):
            f.copy_(B.view(n2, n2 // 8, 8).permute(1, 0, 2).to(torch.bfloat16))
            sa.copy_(torch.sqrt(self._cov_a))

    @property
    def measure_step_counter(self):
        n, s = ctypes.c_int64(), ctypes.c_uint64()
        self._lib.me_k4_get_counters(self._h, ctypes.byref(n), ctypes.byref(s))
        return n.value

    @property
    def steps_done(self):
        n, s = ctypes.c_int64(), ctypes.c_uint64()
        self._lib.me_k4_get_counters(self._h, ctypes.byref(n), ctypes.byref(s))
        return s.value

    # ------------------------------------------------------------------ hot path
    def _adopt_refresh(self):
        """Switch the step kernel to the most recent factor whose refresh was launched at least one measure ago."""
        if self._ready is not None:
            ev, idx = self._ready
            torch.cuda.current_stream(self.device).wait_event(ev)      # finished long ago: no stall
            self._cur = idx
            self._factor, self._s_a = self._factors[idx], self._s_as[idx]
            self._check(self._lib.me_k4_set_factor(self._h, _ptr(self._factor)))
            self._ready = None

    def synchronize_refresh(self):
        """Wait for the factor refresh in flight and make it the current one (reads of the shared covariance, tests)."""
        if self._in_flight is not None:
            self._ready, self._in_flight = self._in_flight, None
        self._adopt_refresh()
        if self._side is not None:
            self._side.synchronize()

    def step(self, k=1, _dbg=None):
        """``k`` x step_all() in one launch.  ``_dbg``: (normals [2 n_c, chains] f32, increments [2 n_c, chains] f32[,
        scalar draws [2, chains] f64]) taps of the first step of the launch (tests, oracle injection)."""
        dz = dd = ds = None
        if _dbg is not None:
            dz, dd = _dbg[0], _dbg[1]
            ds = _dbg[2] if len(_dbg) > 2 else None
        self._adopt_refresh()
        self._launch(self._lib.me_k4_step(self._h, int(k), _ptr(self._s_a), _ptr(dz), _ptr(dd), _ptr(ds), self._stream()))
        if self._in_flight is not None:           # the refresh launched at the last measure becomes adoptable
            self._ready, self._in_flight = self._in_flight, None

    def step_all(self):
        self.step(1)
        return self._last_accept.bool()

    def _ts_slot(self):
        if not self._ts_chunks or self._ts_chunks[-1][1] == self._ts_chunks[-1][0].shape[0]:
            t = torch.empty((self._ts_chunk_rows, self._lay.TS_COLS, self.n_chains), dtype=torch.float64,
                            device=self.device)
            self._ts_chunks.append([t, 0])
        t, used = self._ts_chunks[-1]
        self._ts_chunks[-1][1] = used + 1
        return t, used

    def measure(self):
        """means / observable means / time-series row per chain, then the pooled covariance update that every
        chain's next proposals share."""
        if self.record:
            t, row = self._ts_slot()
            self._launch(self._lib.me_k4_measure(self._h, _ptr(t), row, self._stream()))
        else:
            self._launch(self._lib.me_k4_measure(self._h, None, 0, self._stream()))
        inc, snap, parity, fused = self._moment_buffers()
        self._launch(self._lib.me_k4_moments(self._h, _ptr(self._shift), _ptr(self._scratch), self._scratch.numel(),
                                             _ptr(inc), _ptr(self._mom) if fused else None,
                                             _ptr(snap) if fused else None, self._stream()))
        self.launch_count += 2
        self._after_moments(inc, snap, parity, fused)

    def step_measure(self, k):
        """``k`` x step_all() then measure() as ONE launch of the step kernel (+ the two small reductions of the pooled
        moments): the measurement and this CTA's share of the pooled moments are taken by the epilogue warps while the
        chain states are still in shared memory, the second moments on the tensor cores (include/me_b200.h,
        me_k4_step_measure).  step(k); measure() is the same schedule with all-FP64 moments."""
        self._adopt_refresh()
        t, row = self._ts_slot() if self.record else (None, 0)
        inc, snap, parity, fused = self._moment_buffers()
        self._launch(self._lib.me_k4_step_measure(self._h, int(k), _ptr(self._s_a), _ptr(t), row, _ptr(self._shift),
                                                  _ptr(self._scratch), self._scratch.numel(), _ptr(inc),
                                                  _ptr(self._mom) if fused else None, _ptr(snap) if fused else None,
                                                  self._stream()))
        self.launch_count += 2
        if self._in_flight is not None:           # the refresh launched at the last measure becomes adoptable
            self._ready, self._in_flight = self._in_flight, None
        self._after_moments(inc, snap, parity, fused)

    def _moment_buffers(self):
        parity = self._measure_count % 2
        self._measure_count += 1
        inc, snap = self._incs[parity], self._snaps[parity]
        self._inc_full = inc
        main = torch.cuda.current_stream(self.device)
        if self._snap_events[parity] is not None:      # side-stream work of two measures ago that used these buffers
            main.wait_event(self._snap_events[parity])
            self._snap_events[parity] = None
        fused = not self._distributed            # single GPU: the moments kernel advances mom and writes the snapshot
        return inc, snap, parity, fused

    def _after_moments(self, inc, snap, parity, fused):
        n = self.measure_step_counter
        main = torch.cuda.current_stream(self.device)
        refresh = n > 50                                                                      # ME:389,396
        if fused and not refresh:
            return
        mw = self._lay.MOM_WORDS

        def tail(stream, idx):
            """all-reduce + accumulation (multi-GPU) and the factor refresh, all stream-ordered on `stream`"""
            if not fused:
                # the path's only collective: inside the library (one-shot sum over the NVLink peer windows, else NCCL)
                if self._comm is None:
                    self._comm = parallel.library_comm(_lib.load(), self.device.index) or False
                if self._comm:
                    if _lib.load().me_comm_allreduce(self._comm, _ptr(inc), 2 * inc.numel(), self._stream()) != 0:
                        raise _lib.MeError("me_comm_allreduce: " + _lib.load().me_comm_last_error().decode())
                else:
                    parallel.allreduce_sum_(torch.view_as_real(inc))
                self._launch(self._lib.me_k4_accumulate_moments(self._h, _ptr(inc), _ptr(self._mom), _ptr(snap),
                                                                ctypes.c_void_p(stream.cuda_stream)))
            if refresh:
                self._launch(self._lib.me_k4_refactor(self._h, _ptr(snap), _ptr(snap[mw:]), n, _ptr(self._cov_c),
                                                      _ptr(self._cov_a), _ptr(self._factors[idx]),
                                                      _ptr(self._s_as[idx]), _ptr(self._psd_status),
                                                      ctypes.c_void_p(stream.cuda_stream)))

        if not self._async:
            tail(main, self._cur)
            return
        # side stream, behind this measure: the collective, the accumulation and the one-CTA refresh run beside the next
        # block of steps; the refresh writes a buffer that is neither read by the step kernel nor waiting to be adopted
        idx = None
        if refresh:
            if self._in_flight is not None:       # two measures without a step in between: the older refresh (finished
                self._ready, self._in_flight = self._in_flight, None     # before this one starts) becomes adoptable
            busy = {self._cur} | ({self._ready[1]} if self._ready is not None else set())
            idx = min(i for i in range(3) if i not in busy)
        self._side.wait_stream(main)
        with torch.cuda.stream(self._side):
            tail(self._side, idx)
            ev = torch.cuda.Event()
            ev.record(self._side)
        self._snap_events[parity] = ev
        if refresh:
            self._in_flight = (ev, idx)

    def run(self, n_measures, steps_per_measure, fused_measure=True):
        """``n_measures`` x [``steps_per_measure`` x step_all(), measure()].  By default every block is one step_measure()
        launch; ``fused_measure=False`` keeps step() and measure() as separate kernels with all-FP64 pooled moments."""
        for _ in range(int(n_measures)):
            if fused_measure and steps_per_measure >= 1:
                self.step_measure(int(steps_per_measure))
            else:
                self.step(int(steps_per_measure))
                self.measure()

    # ------------------------------------------------------------------ reads (reference attribute names)
    def _pooled(self, t):
        s = t.sum(dim=-1)
        if self._distributed:
            parallel.allreduce_sum_(s)
        return (s / self.n_chains_total).cpu().numpy()

    @property
    def real_params_per_chain(self):
        return self.state[self._lay.X:self._lay.X + 1].t()

    @property
    def complex_params_per_chain(self):
        x = self._lay.X
        nc = self._nc
        return torch.complex(self.state[x + 1:x + 1 + nc], self.state[x + 1 + nc:x + 1 + 2 * nc]).t()

    @property
    def sampling_width_per_chain(self):
        return self.state[self._lay.SIG]

    @property
    def energy_per_chain(self):
        return self.state[self._lay.E]

    @property
    def accept_count_per_chain(self):
        return self.state[self._lay.NACC]

    @property
    def real_mean(self):
        return self._pooled(self.state[self._lay.MEAN:self._lay.MEAN + 1])

    @property
    def complex_mean(self):
        m = self._lay.MEAN
        nc = self._nc
        return self._pooled(torch.complex(self.state[m + 1:m + 1 + nc], self.state[m + 1 + nc:m + 1 + 2 * nc]))

    @property
    def observables_mean(self):
        return self._pooled(self.state[self._lay.OBSM:self._lay.OBSM + 2 + self._nc])

    @property
    def covariance_matrix_real(self):
        if self._side is not None:
            self._side.synchronize()
        return self._cov_a.reshape(1, 1).cpu().numpy()

    @property
    def covariance_matrix_complex(self):
        if self._side is not None:
            self._side.synchronize()
        return self._cov_c.cpu().numpy()

    @property
    def sampling_width(self):
        return float(self._pooled(self.state[self._lay.SIG:self._lay.SIG + 1])[0])

    real_group_sampling_width = sampling_width
    complex_group_sampling_width = sampling_width

    @property
    def energy_total(self):
        return float(self._pooled(self.state[self._lay.E:self._lay.E + 1])[0])

    @property
    def acceptance_rate(self):
        return float(self._pooled(self.state[self._lay.NACC:self._lay.NACC + 1])[0]) / max(self.steps_done, 1)

    def time_series(self):
        parts = [t[:used] for t, used in self._ts_chunks if used]
        if not parts:
            return torch.empty((0, self._lay.TS_COLS, self.n_chains), dtype=torch.float64, device=self.device)
        return parts[0] if len(parts) == 1 else torch.cat(parts, dim=0)

    def save_time_series(self, chain=0):
        """``self.df`` for one chain, reference column order (ME:466-478)."""
        import pandas
        rows = self.time_series()[:, :, chain].cpu().numpy()
        d, nc = self._lay.D, self._nc
        a, c = rows[:, 0], rows[:, 1:1 + nc] + 1j * rows[:, 1 + nc:d]
        cols = {self.observables_names[0]: np.abs(a)}
        for j in range(nc):
            cols[self.observables_names[1 + j]] = np.abs(c[:, j])
        cols[self.observables_names[1 + nc]] = a * a
        cols["total_energy"] = rows[:, d]
        cols[self.params_names[0]] = a
        cols["real_group_sampling_width"] = rows[:, d + 1]
        for j in range(nc):
            cols[self.params_names[1 + j]] = c[:, j]
        cols["complex_group_sampling_width"] = rows[:, d + 1]
        self.df = pandas.DataFrame.from_dict(cols)
        return self.df

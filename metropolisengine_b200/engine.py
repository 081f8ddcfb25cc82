"""Host-side mirror of the reference's one public class, driving the CUDA hot path through the C ABI.

``MetropolisEngine`` keeps the reference's constructor signature, method names and read attributes
(/root/reference/metropolisengine/metropolis_engine.py, "ME"; README.md:23-58) and adds keyword-only ensemble
controls.  A 1-chain engine behaves like the reference (numpy values, ``step_all()`` returns a bool); an
``n_chains > 1`` engine runs that many independent chains on the GPU and reports pooled values, with
``*_per_chain`` tensors beside them.

Energy plugin forms (the reference's plugin surface, ME:20, ME:110-120):
  * ``BuiltinEnergy`` / a name such as ``"xy_well"``     -> ahead-of-time fused kernels
  * ``CudaEnergy(source)``                               -> device functor compiled with NVRTC, fused
  * a python callable over torch tensors, or a dict of them (ME:111-115) -> unfused propose / callable / accept

PyTorch is used for device memory, streams and torch.distributed only; all arithmetic of the path runs in
libme_b200.so.  There is no CPU fallback.
"""
import ctypes
import math

import numpy as np
import torch

from . import _lib
from . import parallel


class BuiltinEnergy:
    """A built-in device energy functor (csrc/me_energies.cuh): ``x2``, ``xy_well(const)``,
    ``mixed_well(k, alpha, beta)``, ``cylinder(kappa, alpha, gamma, beta)`` (the latter with its hard wall
    ``|a| >= 1`` when ``reject=True``)."""

    def __init__(self, name, *consts, reject=False):
        if name not in _lib.ENERGY_IDS:
            raise ValueError("unknown built-in energy %r (have %s)" % (name, sorted(_lib.ENERGY_IDS)))
        self.name, self.consts, self.reject = name, tuple(float(c) for c in consts), bool(reject)


class CudaEnergy:
    """User device functor.  ``source`` is CUDA C++ defining::

        __device__ double me_user_energy(const double* x, const double* c_re, const double* c_im, const double* k);
        __device__ bool   me_user_reject(...same...);      // only when has_reject=True

    ``x`` holds the real parameters, ``c_re`` / ``c_im`` the complex ones, ``k`` the ``consts``; the macros
    ``ME_NR`` / ``ME_NC`` give the shape.  Compiled for sm_100a by NVRTC and fused into the step kernel."""

    def __init__(self, source, consts=(), has_reject=False):
        self.source, self.consts, self.has_reject = source, tuple(float(c) for c in consts), bool(has_reject)


def adaptation_constants(n_real, n_complex, target_acceptance):
    """alpha, m, ratio exactly as the reference evaluates them (ME:101-107; note ``/ 2 * alpha``)."""
    try:
        from scipy.stats import norm
        alpha = -1 * norm.ppf(target_acceptance / 2)
    except ImportError:                                    # pragma: no cover
        from statistics import NormalDist
        alpha = -1 * NormalDist().inv_cdf(target_acceptance / 2)
    m = n_real + n_complex
    ratio = ((1 - (1 / m)) * math.sqrt(2 * math.pi) * math.exp(alpha ** 2 / 2) / 2 * alpha
             + 1 / (m * target_acceptance * (1 - target_acceptance)))
    return float(alpha), m, float(ratio)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


class MetropolisEngine:
    """Adaptive random-walk Metropolis over real and complex parameters, many chains per GPU.

    Positional/keyword arguments up to ``complex_sample_method`` are the reference's (ME:17).  Keyword-only
    additions:

    n_chains          chains in the whole job (default 1 = reference behaviour)
    seed              Philox key; chain i of the job always uses sub-stream i
    device            torch device (default: current CUDA device)
    strict            reference operation order without FMA contraction; enables ``run_injected``
    record            keep a time-series row per chain at every ``measure()`` (default True)
    callable_layout   layout of the tensors handed to a python energy callable: ``"chains_first"``
                      ([chains, n_params], default) or ``"params_first"`` ([n_params, chains], so reference-style
                      bodies such as ``real_params[0]**2`` vectorise unchanged)
    distributed       shard ``n_chains`` over the ranks of the default torch.distributed group
    graph_callable    python energy callables only: capture the ``steps_per_measure`` steps between two measures
                      (propose -> callable -> accept, each) in a CUDA graph on first use and replay it in ``run()``;
                      the callable must then be capture-safe (static shapes, no host synchronisation)
    replica_exchange  with ``temp`` a sequence of R temperatures (a ladder: global chain g runs at ``temp[g % R]``):
                      0 = a temperature sweep without swaps; k > 0 = parallel tempering, a replica-exchange round of
                      neighbour rungs (deterministic even/odd pairing) at every k-th measure.  Pooled attributes and
                      ``pooled_statistics()`` of a ladder engine gain a leading rung axis of length R.
    rung_consts       [R, K] array: a Hamiltonian ladder.  Rung r (global chain g is rung g % R) runs the energy functor
                      with the constants ``rung_consts[r]`` instead of the energy's own, at ``temp`` (a number: every rung)
                      or ``temp[r]`` (a sequence of length R).  K must equal the number of constants the energy was given.
                      With ``replica_exchange=k > 0`` neighbour rungs a < b swap configurations with probability
                      min(1, exp(-D)), D = (E_a(x_b) - E_a(x_a)) / T_a + (E_b(x_a) - E_b(x_b)) / T_b, and a chain that
                      takes a configuration takes its own rung's energy of it; 0 = a sweep over the constants in one
                      launch.  Everything else is as for temperature ladders.
    """

    def __new__(cls, *args, adapt="per_chain", **kw):
        """One front door (SURVEY §5 config row): ``adapt="pooled"`` builds the shared-covariance engine (the proposal
        covariance of the complex block pooled over the ensemble, L.Z on the tensor cores) from the same arguments."""
        if adapt == "pooled" and cls is MetropolisEngine:
            if np.ndim(kw.get("temp", args[9] if len(args) > 9 else 0)) > 0 or kw.get("rung_consts") is not None:
                raise NotImplementedError("temperature and Hamiltonian ladders run with adapt='per_chain' only")
            from .engine_shared import SharedCovarianceEngine
            return SharedCovarianceEngine.from_reference_arguments(*args, **kw)
        if adapt not in ("per_chain", "pooled"):
            raise ValueError("adapt must be 'per_chain' (the reference's algorithm) or 'pooled'")
        return super().__new__(cls)

    def __init__(self, energy_functions, reject_condition=None, initial_real_params=None,
                 initial_complex_params=None, sampling_width=0.05, covariance_matrix_real=None,
                 covariance_matrix_complex=None, params_names=None, target_acceptance=.3, temp=0,
                 complex_sample_method="multivariate-gaussian", *, n_chains=1, seed=0, device=None, strict=False,
                 record=True, callable_layout="chains_first", distributed=False, ts_chunk_bytes=1 << 30,
                 graph_callable=False, adapt="per_chain", replica_exchange=0, rung_consts=None, _shard=None):
        if initial_real_params is None and initial_complex_params is None:
            raise ValueError("must give a list containing at least one value for initial real or complex "
                             "parameters")                                                   # ME:37-39
        if complex_sample_method not in ("multivariate-gaussian", "magnitude-phase"):
            # the reference prints a notice and falls back (ME:131-133); nothing is printed here (SURVEY App. B-12)
            complex_sample_method = "multivariate-gaussian"
        self.complex_sample_method = complex_sample_method
        self._ladder = None             # temperatures [R] of a ladder engine
        self._swap_every = int(replica_exchange)
        if self._swap_every < 0:
            raise ValueError("replica_exchange must be >= 0")
        if np.ndim(temp) == 1:
            temps = np.asarray(temp, dtype=np.float64)
            if temps.size == 0:
                raise ValueError("temp as a sequence needs at least one temperature")
            if temps.size > 1:
                self._ladder = temps
            temp = float(temps[0])
        elif np.ndim(temp) > 1:
            raise ValueError("temp is a number or a 1-D sequence of temperatures")
        self._rung_consts = None        # [R, K] functor constants of a Hamiltonian ladder's rungs
        if rung_consts is not None:
            rc = np.array(rung_consts, dtype=np.float64)
            if rc.ndim != 2 or rc.shape[0] < 2 or rc.shape[1] < 1:
                raise ValueError("rung_consts is an [R, K] array with R >= 2 rungs and K >= 1 constants")
            if not np.all(np.isfinite(rc)):
                raise ValueError("rung_consts must be finite")
            if self._ladder is None:
                self._ladder = np.full(rc.shape[0], temp, dtype=np.float64)
            elif self._ladder.size != rc.shape[0]:
                raise ValueError("temp has %d temperatures for %d rungs of rung_consts" % (self._ladder.size, rc.shape[0]))
            self._rung_consts = rc
        if self._swap_every and self._ladder is None:
            raise ValueError("replica_exchange needs temp as a sequence of at least 2 temperatures")
        if temp is None or not temp >= 0:
            raise AssertionError("temp must be >= 0")                                        # ME:92
        self._width_pair = None
        if isinstance(sampling_width, (list, tuple)):                                        # ME:93-95
            if len(sampling_width) != 2:
                raise ValueError("sampling_width as a list is [sigma_real, sigma_complex]")
            self._width_pair = (float(sampling_width[0]), float(sampling_width[1]))
            # the reference leaves self.sampling_width undefined in this form and its mixed step_all() then fails at
            # ME:431; here a mixed step_all() continues from the real group's width (SURVEY App. B-4)
            sampling_width = self._width_pair[0]
        if not torch.cuda.is_available():
            raise RuntimeError("MetropolisEngine needs a CUDA device: the hot path is CUDA-only (no CPU fallback)")
        self._lib = _lib.load()
        self.launch_count = 0
        self._graph_callable = bool(graph_callable)
        self._graphs = {}               # steps per measure -> captured torch.cuda.CUDAGraph
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())

        # ---- parameter space (ME:40-60)
        xr = None if initial_real_params is None else np.asarray(initial_real_params, dtype=np.float64)
        xc = None if initial_complex_params is None else np.asarray(initial_complex_params, dtype=np.complex128)
        self.num_real_params = 0 if xr is None else xr.shape[-1]
        self.num_complex_params = 0 if xc is None else xc.shape[-1]
        self.param_space_dims = self.num_real_params + self.num_complex_params
        if self.param_space_dims == 0:
            raise ValueError("empty parameter space")
        nr, nc = self.num_real_params, self.num_complex_params
        self._kind = "mixed" if (nr and nc) else ("real" if nr else "complex")
        self._lay = _lib.layout(nr, nc)
        self._d = self._lay.D

        # ---- chains and sharding
        self.n_chains_total = int(n_chains)
        self._group = None
        self._rank, self._world = (parallel.world() if distributed else (0, 1))
        R = 1 if self._ladder is None else self._ladder.size
        if self.n_chains_total % R:
            raise ValueError("n_chains (%d) must be a multiple of the ladder's %d rungs" % (self.n_chains_total, R))
        lo, hi = parallel.shard_range(self.n_chains_total, self._rank, self._world, granule=R)
        if _shard is not None:          # explicit global chain range [lo, hi) (tests, custom launchers)
            lo, hi = int(_shard[0]), int(_shard[1])
            if lo % R or hi % R:
                raise ValueError("a ladder engine's shard must hold whole ladders of %d chains" % R)
        self.chain_offset, self.n_chains = lo, hi - lo
        self._distributed = bool(distributed) and self._world > 1

        per_chain_init = (xr is not None and xr.ndim == 2) or (xc is not None and xc.ndim == 2)
        x0 = np.zeros((self._d, self.n_chains_total if per_chain_init else 1))
        if xr is not None:
            x0[:nr] = xr.T if xr.ndim == 2 else xr[:, None]
        if xc is not None:
            x0[nr:nr + nc] = (xc.real.T if xc.ndim == 2 else xc.real[:, None])
            x0[nr + nc:] = (xc.imag.T if xc.ndim == 2 else xc.imag[:, None])
        if per_chain_init and x0.shape[1] != self.n_chains_total:
            raise ValueError("per-chain initial parameters must have n_chains rows")
        self._shift_host = x0.mean(axis=1)

        # ---- names (ME:82-87)
        self.params_names = list(params_names) if params_names else ["param_" + str(i) for i in range(nr + nc)]
        self.observables_names = ["abs_param_" + str(i) for i in range(nr + nc)]
        self.observables_names.extend(["param_" + str(i) + "_squared" for i in range(nr)])

        # ---- adaptation constants (ME:91-107)
        self.temp = temp if self._ladder is None else self._ladder.copy()
        self.target_acceptance = target_acceptance
        self.alpha, self.m, self.ratio = adaptation_constants(nr, nc, target_acceptance)
        self._sampling_width0 = float(sampling_width)
        self.strict = bool(strict)
        self.seed = int(seed)
        self.df = None                                                                       # ME:108

        # ---- native handle
        cfg = _lib.MeConfig(nr, nc, self.n_chains, self.chain_offset, float(temp), float(target_acceptance),
                            self.ratio, self.seed, self.device.index, int(self.strict))
        h = ctypes.c_void_p()
        _lib.check(None, self._lib.me_create(ctypes.byref(cfg), ctypes.byref(h)))
        self._h = h
        grid, block = ctypes.c_int32(), ctypes.c_int32()
        dev, f64 = self.device, torch.float64
        self._walker = self._swap_acc = None
        pw = self._lay.POOL_WORDS
        if self._ladder is not None:
            self._check_ladder_supported(energy_functions, reject_condition, complex_sample_method)
            self._walker = torch.arange(lo, hi, dtype=torch.int32, device=dev)
            self._swap_acc = torch.zeros(self.n_chains, dtype=torch.int32, device=dev)     # read as uint32 by the library
            temps = (ctypes.c_double * R)(*self._ladder.tolist())
            if self._rung_consts is None:
                self._check(self._lib.me_set_ladder(self._h, temps, R, self._swap_every, _ptr(self._walker),
                                                    _ptr(self._swap_acc)))
            else:
                K = self._rung_consts.shape[1]
                n_energy = len(self._device_energy(energy_functions).consts)
                if n_energy != K:
                    raise ValueError("rung_consts has %d constants per rung, the energy takes %d" % (K, n_energy))
                table = (ctypes.c_double * (R * K))(*self._rung_consts.ravel().tolist())
                self._check(self._lib.me_set_hamiltonian_ladder(self._h, temps, table, K, R, self._swap_every,
                                                                _ptr(self._walker), _ptr(self._swap_acc)))
            pw = pw * R if R <= 32 and R & (R - 1) == 0 else 0      # per-rung rows; see me_set_ladder
        self._lib.me_launch_dims(self._h, ctypes.byref(grid), ctypes.byref(block))
        self._grid, self._block = grid.value, block.value

        # ---- device buffers (owned here, borrowed by the library)
        self.state = torch.zeros((self._lay.WORDS, self.n_chains), dtype=f64, device=dev)
        self._pool = torch.zeros((self._grid, pw), dtype=f64, device=dev) if pw > 0 else None
        self._shift = torch.tensor(self._shift_host, dtype=f64, device=dev)
        self._last_accept = torch.zeros(self.n_chains, dtype=torch.uint8, device=dev)
        self._pool_out = torch.zeros(max(pw, 1), dtype=f64, device=dev)
        # pooled moments live on the device: [POOL_WORDS sums | sample count], summed over ranks inside the library
        # (me_allreduce_stats); the host reads them once, when statistics are asked for
        self._pool_inc = torch.zeros(pw + 1, dtype=f64, device=dev)
        self._pool_tot = torch.zeros(pw + 1, dtype=f64, device=dev)
        self._pool_pending = 0          # local (chain, measure) samples accumulated since the last reduction
        self._comm = None
        self._ctr_on = False
        self._generic = self._d > 32          # large shapes: runtime-shape kernels, unfused step (me_generic.cu)
        self._scratch = torch.zeros((self._d, self.n_chains), dtype=f64, device=dev) if self._generic else None
        self._prop = torch.zeros((self._d, self.n_chains), dtype=f64, device=dev) if self._generic else None
        bufs = _lib.MeBuffers(_ptr(self.state), _ptr(self._pool), _ptr(self._shift), _ptr(self._last_accept),
                              _ptr(self._scratch), _ptr(self._prop))
        self._check(self._lib.me_bind(self._h, ctypes.byref(bufs)))

        # ---- energy plugin (ME:110-120) and hard-wall predicate (ME:126-127, 142-146)
        self._callable = None
        self._terms = None
        self.reject_condition = None
        self._group_mode = 0
        self._callable_layout = callable_layout
        if callable_layout not in ("chains_first", "params_first"):
            raise ValueError("callable_layout must be 'chains_first' or 'params_first'")
        self._install_energy(energy_functions)
        self._check_reject_supported(reject_condition)
        self.reject_condition = reject_condition

        # ---- state initialisation (ME:63-81, 123-125)
        if per_chain_init:
            x0_dev = torch.tensor(np.ascontiguousarray(x0[:, lo:hi]), dtype=f64, device=dev)
        else:
            x0_dev = torch.tensor(np.ascontiguousarray(x0[:, 0]), dtype=f64, device=dev)
        cov_r = cov_c_re = cov_c_im = None
        if covariance_matrix_real is not None and nr:
            cov_r = torch.tensor(np.ascontiguousarray(covariance_matrix_real, dtype=np.float64), device=dev)
            assert cov_r.shape == (nr, nr)
        if covariance_matrix_complex is not None and nc:
            cc = np.asarray(covariance_matrix_complex, dtype=np.complex128)
            assert cc.shape == (nc, nc)
            cov_c_re = torch.tensor(np.ascontiguousarray(cc.real), device=dev)
            cov_c_im = torch.tensor(np.ascontiguousarray(cc.imag), device=dev)
        e0 = None
        if self._callable is not None:
            full = x0_dev if per_chain_init else x0_dev[:, None].expand(self._d, self.n_chains).contiguous()
            e0 = self._eval_callable(full)
        self._launch(self._lib.me_init(self._h, _ptr(x0_dev), 0 if per_chain_init else 1, self._sampling_width0,
                                      _ptr(cov_r), _ptr(cov_c_re), _ptr(cov_c_im), _ptr(e0), self._stream()))
        self._apply_width_pair()
        self._energy0 = self.state[self._lay.E].clone()
        self._term_energy0 = None
        if self._terms is not None:
            full = self.state[:self._d]
            self._term_energy0 = {t: self._eval_term(fn, full).clone() for t, fn in self._terms["all"].items()}
        self._group_mode = 0
        self.step_counter = 1                                                               # ME:72
        self.complex_group_step_counter = 1
        self.real_group_step_counter = 1

        # ---- time series (the lists of ME:31-35)
        self.record = bool(record)
        self._ts_chunks = []          # list of [tensor (rows, TS_COLS, n_chains), used_rows]
        self._ts_rows = 0
        self._ts_chunk_rows = max(1, int(ts_chunk_bytes) // (self._lay.TS_COLS * self.n_chains * 8))
        self._term_series = {} if self._terms is not None else None

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, rc):
        _lib.check(self._h, rc)

    def _launch(self, rc):
        """Bookkeeping for calls that launch one of the library's kernels."""
        _lib.check(self._h, rc)
        self.launch_count += 1

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and getattr(self, "_lib", None) is not None:
            self._lib.me_destroy(h)
            self._h = None

    def _apply_width_pair(self):
        """sampling_width=[sigma_real, sigma_complex] (ME:93-95): the two group widths start apart."""
        if self._width_pair is not None:
            self.state[self._lay.SIG].fill_(self._width_pair[0])
            self.state[self._lay.SIG + 1].fill_(self._width_pair[1])

    @staticmethod
    def _device_energy(energy):
        """A built-in name or (name, consts...) tuple as its BuiltinEnergy; anything else unchanged."""
        if isinstance(energy, str):
            return BuiltinEnergy(energy)
        if isinstance(energy, tuple) and energy and isinstance(energy[0], str):
            return BuiltinEnergy(energy[0], *energy[1:])
        return energy

    def _install_energy(self, energy):
        energy = self._device_energy(energy)
        if isinstance(energy, BuiltinEnergy):
            consts = (ctypes.c_double * max(len(energy.consts), 1))(*energy.consts)
            self._check(self._lib.me_set_energy_builtin(self._h, _lib.ENERGY_IDS[energy.name], consts,
                                                        len(energy.consts), int(energy.reject)))
            self.energy_term_names = ["total"]
        elif isinstance(energy, CudaEnergy):
            consts = (ctypes.c_double * max(len(energy.consts), 1))(*energy.consts)
            self._check(self._lib.me_set_energy_source(self._h, energy.source.encode(), consts, len(energy.consts),
                                                       int(energy.has_reject)))
            self.energy_term_names = ["total"]
        elif isinstance(energy, dict):                       # dict of terms (ME:111-115)
            names = set()
            for group in energy.values():
                names = names.union(group)
            self.energy_term_names = names
            self._terms = energy
            self._callable = lambda r, c: sum(fn(r, c) for fn in energy["all"].values())
            self._check(self._lib.me_set_energy_external(self._h))
        elif callable(energy):
            self.energy_term_names = ["total"]
            self._callable = energy
            self._check(self._lib.me_set_energy_external(self._h))
        else:
            raise TypeError("energy_functions must be a built-in name, BuiltinEnergy, CudaEnergy, a callable or a "
                            "dict of callables")
        self._energy_spec = energy

    def set_energy_function(self, energy_function):                                        # ME:136-140
        if self._rung_consts is not None:
            raise NotImplementedError("a Hamiltonian ladder's rung_consts belong to its energy functor; build a new engine "
                                      "to change the functor")
        if self._ladder is not None:
            self._check_ladder_supported(energy_function, self.reject_condition, self.complex_sample_method)
        self._callable = self._terms = None
        self._install_energy(energy_function)

    def set_reject_condition(self, reject_fct):                                            # ME:142-146
        if self._ladder is not None and reject_fct is not None:
            raise NotImplementedError("temperature ladders take the hard wall inside the device functor, not a python "
                                      "reject_condition")
        self._check_reject_supported(reject_fct)
        self.reject_condition = reject_fct

    def _check_ladder_supported(self, energy, reject_condition, complex_sample_method):
        """Temperature ladders run in the fused step kernel only (its PT instantiation)."""
        if self._d > 32:
            raise NotImplementedError("temperature ladders need n_real + 2 n_complex <= 32 (fused shapes)")
        if not isinstance(energy, (BuiltinEnergy, CudaEnergy, str)) and not (
                isinstance(energy, tuple) and energy and isinstance(energy[0], str)):
            raise NotImplementedError("temperature ladders need a device energy functor (BuiltinEnergy / CudaEnergy)")
        if reject_condition is not None:
            raise NotImplementedError("temperature ladders take the hard wall inside the device functor, not a python "
                                      "reject_condition")
        if complex_sample_method == "magnitude-phase":
            raise NotImplementedError("temperature ladders do not run magnitude-phase complex moves")

    def _check_reject_supported(self, reject_fct):
        """A python predicate (ME:142-146) is evaluated on the proposal block between the proposal and the decision,
        so an engine that has one steps unfused: me_propose -> device functor (me_energy_builtin) or python energy ->
        predicate -> me_accept.  The fast form of a hard wall is inside the functor (``BuiltinEnergy(...,
        reject=True)`` / ``CudaEnergy(..., has_reject=True)``), which keeps the step fused."""
        if reject_fct is not None and not callable(reject_fct):
            raise TypeError("reject_condition must be callable: (real_params, complex_params) -> bool per chain")

    def _split(self, block):
        """[D, chains] block -> (real, complex) tensors in the callable's layout."""
        nr, nc = self.num_real_params, self.num_complex_params
        r = block[:nr]
        c = torch.complex(block[nr:nr + nc], block[nr + nc:nr + 2 * nc]) if nc else block[:0].to(torch.complex128)
        if self._callable_layout == "chains_first":
            return r.t(), c.t()
        return r, c

    def _eval_term(self, fn, block):
        r, c = self._split(block)
        e = fn(r, c)
        if not torch.is_tensor(e):
            e = torch.as_tensor(e, device=self.device)
        if e.is_complex():
            e = e.real                                         # reference energies may carry a zero imaginary part (App. B-9)
        e = e.to(torch.float64)
        if e.dim() == 0:
            e = e.expand(self.n_chains)
        if e.shape != (self.n_chains,):
            raise ValueError("energy callable must return one value per chain, shape (%d,), got %s; check "
                             "callable_layout=%r" % (self.n_chains, tuple(e.shape), self._callable_layout))
        return e.contiguous()

    def _eval_callable(self, block):
        return self._eval_term(self._callable, block)

    # ------------------------------------------------------------------ time-series storage
    def _ts_segments(self, n_rows):
        """Reserve n_rows rows; returns (chunk tensor, first row in chunk, rows) per launch."""
        out = []
        for c in self._ts_chunks:
            if n_rows <= 0:
                break
            t, used = c
            take = min(n_rows, t.shape[0] - used)
            if take > 0:
                out.append((t, used, take))
                c[1] = used + take
                self._ts_rows += take
                n_rows -= take
        while n_rows > 0:
            t = torch.empty((self._ts_chunk_rows, self._lay.TS_COLS, self.n_chains), dtype=torch.float64,
                            device=self.device)
            take = min(n_rows, t.shape[0])
            self._ts_chunks.append([t, take])
            out.append((t, 0, take))
            self._ts_rows += take
            n_rows -= take
        return out

    def reserve_rows(self, n_rows):
        """Pre-allocate time-series storage for n_rows further measures (keeps cudaMalloc out of the run)."""
        have = sum(t.shape[0] - used for t, used in self._ts_chunks)
        while have < n_rows:
            rows = min(self._ts_chunk_rows, n_rows - have) if not self._ts_chunks else self._ts_chunk_rows
            rows = max(rows, 1)
            t = torch.empty((rows, self._lay.TS_COLS, self.n_chains), dtype=torch.float64, device=self.device)
            self._ts_chunks.append([t, 0])
            have += rows

    def clear_time_series(self, keep_storage=True):
        """Forget recorded rows (optionally keeping the allocated storage for reuse)."""
        if keep_storage:
            for c in self._ts_chunks:
                c[1] = 0
        else:
            self._ts_chunks = []
        self._ts_rows = 0
        if self._term_series is not None:
            self._term_series = {}

    def reset(self, initial_real_params=None, initial_complex_params=None, sampling_width=None):
        """Re-initialise every chain (ME:40-125) from host or device arrays without rebuilding the engine:
        parameters [n_chains, n] (or [n] broadcast), means, identity covariances, widths, counters."""
        nr, nc, d = self.num_real_params, self.num_complex_params, self._d
        x0 = torch.empty((d, self.n_chains), dtype=torch.float64, device=self.device)
        if nr:
            r = torch.as_tensor(initial_real_params, dtype=torch.float64)
            r = r.to(self.device, non_blocking=True)
            x0[:nr] = r.t() if r.dim() == 2 else r[:, None]
        if nc:
            c = torch.as_tensor(initial_complex_params, dtype=torch.complex128)
            c = c.to(self.device, non_blocking=True)
            x0[nr:nr + nc] = c.real.t() if c.dim() == 2 else c.real[:, None]
            x0[nr + nc:] = c.imag.t() if c.dim() == 2 else c.imag[:, None]
        e0 = self._eval_callable(x0) if self._callable is not None else None
        if isinstance(sampling_width, (list, tuple)):
            self._width_pair = (float(sampling_width[0]), float(sampling_width[1]))
            sampling_width = self._width_pair[0]
        elif sampling_width is not None:
            self._width_pair = None
        sw = self._sampling_width0 if sampling_width is None else float(sampling_width)
        self._launch(self._lib.me_init(self._h, _ptr(x0), 0, sw, None, None, None, _ptr(e0), self._stream()))
        self._apply_width_pair()
        self._energy0 = self.state[self._lay.E].clone()
        if self._ladder is not None:
            self._walker.copy_(torch.arange(self.chain_offset, self.chain_offset + self.n_chains, dtype=torch.int32))
            self._swap_acc.zero_()
        self.reset_pooled_statistics()
        self.clear_time_series()
        self.step_counter = 1

    # ------------------------------------------------------------------ the hot path
    def run(self, n_measures, steps_per_measure):
        """``n_measures x (steps_per_measure x step_all() + measure())`` — the README/demo loop
        (README.md:39-44, demo/toymodel_xypotentialwell.py:39-44) in as few launches as possible."""
        n_measures, steps_per_measure = int(n_measures), int(steps_per_measure)
        if n_measures <= 0:
            return
        if self._unfused():
            graphed = (self._graph_callable and self._callable is not None and not self._generic
                       and steps_per_measure > 0)
            for _ in range(n_measures):
                if graphed:
                    self._replay_steps(steps_per_measure)
                else:
                    for _ in range(steps_per_measure):
                        self._step_external()
                self.measure()
            return
        if self.record:
            for t, row0, rows in self._ts_segments(n_measures):
                self._launch(self._lib.me_run(self._h, rows, steps_per_measure, 1, _ptr(t), row0, self._stream()))
        else:
            self._launch(self._lib.me_run(self._h, n_measures, steps_per_measure, 1, None, 0, self._stream()))
        self._pool_pending += n_measures * self.n_chains
        self.step_counter += n_measures * steps_per_measure if self._kind == "complex" else 0

    def run_graphed(self, n_measures, steps_per_measure, launches=1):
        """``run()`` followed by the pooled-moment reduction and its all-reduce across ranks, as ONE CUDA-graph launch
        (fused device-functor engines, ``record=False``): for ensembles whose launch lasts only a fraction of a
        millisecond the per-launch host work otherwise bounds the job.  The first call runs eagerly (it makes every
        allocation), the second captures, later ones replay; the Philox step index and the measure counter come from
        the device copy of the counters, so a replay continues the chains exactly like an eager call
        (``test_graph_replay_of_fused_runs_is_bit_identical``).

        ``launches > 1`` puts that many consecutive ``[run -> reduction -> all-reduce]`` rounds into the one graph and
        moves each round's collective (``me_accumulate_stats``: NCCL all-reduce + accumulation into the device-resident
        totals) to a side stream, where it overlaps the NEXT round's stepping launch (SURVEY §8e); only the fixed-order
        reduction of the per-CTA rows (``me_reduce_stats``) stays between two stepping launches.  Two increment buffers
        alternate.  The totals are the same sums in the same order as with ``launches`` separate calls."""
        n_measures, steps_per_measure, launches = int(n_measures), int(steps_per_measure), int(launches)
        if self._unfused() or self._generic or self.record:
            raise RuntimeError("run_graphed serves fused device-functor engines (D <= 32) with record=False")
        if launches < 1:
            raise ValueError("launches must be >= 1")
        key = ("fused", n_measures, steps_per_measure, launches)
        seen = self._graphs.get(key)
        if seen is None:                        # first use: eager, so that no allocation happens under capture
            for _ in range(launches):
                self.run(n_measures, steps_per_measure)
                self._flush_pool()
            if launches > 1 and getattr(self, "_pool_inc2", None) is None:
                self._pool_inc2 = torch.zeros_like(self._pool_inc)
                self._side_stream = torch.cuda.Stream(device=self.device)
            self._graphs[key] = "warm"
            return
        n, s0 = ctypes.c_int64(), ctypes.c_uint64()
        self._lib.me_get_counters(self._h, ctypes.byref(n), ctypes.byref(s0))
        if not self._ctr_on:
            self._check(self._lib.me_device_counters(self._h, 1, self._stream()))
            self._ctr_on = True
        if seen == "warm":
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            pending = self._pool_pending
            samples = n_measures * self.n_chains
            with torch.cuda.graph(g):
                if launches == 1:
                    self._launch(self._lib.me_run(self._h, n_measures, steps_per_measure, 1, None, 0, self._stream()))
                    self._launch(self._lib.me_allreduce_stats(self._h, self._library_comm(), _ptr(self._pool_inc),
                                                              _ptr(self._pool_tot), samples, self._stream()))
                else:
                    main, side = torch.cuda.current_stream(self.device), self._side_stream
                    incs, free = (self._pool_inc, self._pool_inc2), [None, None]
                    for i in range(launches):
                        self._launch(self._lib.me_run(self._h, n_measures, steps_per_measure, 1, None, 0, self._stream()))
                        k = i & 1
                        if free[k] is not None:
                            main.wait_event(free[k])            # the collective two rounds ago is done with this buffer
                        self._launch(self._lib.me_reduce_stats(self._h, _ptr(incs[k]), samples, self._stream()))
                        ready = torch.cuda.Event()
                        ready.record(main)
                        side.wait_event(ready)
                        with torch.cuda.stream(side):
                            self._launch(self._lib.me_accumulate_stats(self._h, self._library_comm(), _ptr(incs[k]),
                                                                       _ptr(self._pool_tot), self._stream()))
                        free[k] = torch.cuda.Event()
                        free[k].record(side)
                    main.wait_stream(side)
            self._check(self._lib.me_set_counters(self._h, n.value, s0.value))     # capture moved the host counters
            self._pool_pending = pending
            self._graphs[key] = seen = g
        if self._pool_pending:
            self._flush_pool()                  # samples of earlier eager runs go in before the graph's own
        seen.replay()
        self.launch_count += 3 * launches
        self._check(self._lib.me_set_counters(self._h, n.value + launches * n_measures,
                                              s0.value + launches * n_measures * steps_per_measure))
        self.step_counter += launches * n_measures * steps_per_measure if self._kind == "complex" else 0

    def step(self, k=1):
        """``k`` calls of ``step_all()`` in one launch (no measure)."""
        k = int(k)
        if self._unfused():
            for _ in range(k):
                self._step_external()
            return
        self._launch(self._lib.me_run(self._h, 1, k, 0, None, 0, self._stream()))
        self.step_counter += k if self._kind == "complex" else 0

    def step_all(self):
        """One Metropolis step of every chain over all parameters (ME:241-259; for all-real / all-complex engines
        the reference rebinds this to the group step, ME:46,56).  Returns the accept decision: a python bool for a
        1-chain engine (as the reference), a bool tensor [n_chains] on the device otherwise."""
        self.step(1)
        if self.n_chains_total == 1:
            return bool(self._last_accept.item())
        return self._last_accept.bool()

    # ---- group-wise stepping (SURVEY §8 row f1; ME:209-239, 440-456)
    def _set_group(self, group):
        if group and self._ladder is not None:
            raise NotImplementedError("temperature ladders step all parameters at once (step_all / step / run)")
        if group != self._group_mode:
            self._check(self._lib.me_set_group(self._h, group))
            self._group_mode = group

    def _group_step(self, group, k=1):
        self._set_group(group)
        try:
            self.step(k)
        finally:
            self._set_group(0)
        if group in (2, 3) and self._kind == "mixed":
            self.step_counter += int(k)                                                     # ME:450
        if group == 4 and self._kind == "complex":
            self.step_counter -= int(k)             # the phase redraw does not go through ME:449-456
        if self.n_chains_total == 1:
            return bool(self._last_accept.item())
        return self._last_accept.bool()

    def step_real_group(self, k=1):
        """Propose and decide the real block only, with its own width (ME:225-239, 440-446).  For all-real engines
        this is ``step_all`` (ME:56)."""
        if not self.num_real_params:
            raise ValueError("engine has no real parameters")
        return self._group_step(1 if self._kind == "mixed" else 0, k)

    def step_complex_group(self, k=1):
        """Propose and decide the complex block only, with its own width (ME:209-223, 449-456).  With
        ``complex_sample_method="magnitude-phase"`` the reference rebinds this method (ME:129-130) to a Gaussian
        move of the moduli followed by a uniform redraw of the phases (ME:168-176) and returns None; so does this.
        ``step_all`` keeps the multivariate-Gaussian proposal in either case, as in the reference (ME:46, ME:246)."""
        if not self.num_complex_params:
            raise ValueError("engine has no complex parameters")
        if self.complex_sample_method == "magnitude-phase":
            for _ in range(int(k)):
                self.step_complex_group_magnitude()
                self.step_complex_group_phase()
            return None
        return self._group_step(2 if self._kind == "mixed" else 0, k)

    def _require_magnitude_phase_kernels(self):
        if not self.num_complex_params:
            raise ValueError("engine has no complex parameters")

    def step_complex_group_magnitude(self, k=1):
        """Gaussian move of every modulus at fixed phase, own Metropolis test, adapts the complex width (ME:178-192;
        draw ME:304-310, including the reference's use of sigma^2 C_jj as the standard deviation)."""
        self._require_magnitude_phase_kernels()
        return self._group_step(3, k)

    def step_complex_group_phase(self, k=1):
        """Uniform redraw of every phase at fixed modulus, own Metropolis test, adapts nothing (ME:194-207, 312-317)."""
        self._require_magnitude_phase_kernels()
        return self._group_step(4, k)

    def run_injected_group(self, group, delta, u, k):
        """Parity mode for group steps: ``k`` injected steps of one group (no measure).  For groups 3 / 4 (magnitude /
        phase moves) the complex block of ``delta`` holds the proposed values themselves, not increments."""
        self._set_group(group if (self._kind == "mixed" or group >= 3) else 0)
        try:
            self.run_injected(delta, u, 1, k, do_measure=False)
        finally:
            self._set_group(0)
        if group in (2, 3) and self._kind == "mixed":
            self.step_counter += int(k)

    def _unfused(self):
        """True when a step is propose -> energy -> accept (separate launches) instead of one kernel: python energies,
        any engine carrying a python reject_condition, and large shapes doing magnitude / phase moves.  Large shapes
        (D > 32) with a device functor run whole schedules in one launch of the runtime-shape kernel (gk_run)."""
        return (self._callable is not None or self.reject_condition is not None
                or (self._generic and self._group_mode >= 3))

    def _step_external(self, inj_delta=None, inj_u=None):
        prop = torch.empty((self._d, self.n_chains), dtype=torch.float64, device=self.device)
        self._launch(self._lib.me_propose(self._h, _ptr(prop), _ptr(inj_delta), self._stream()))
        rej = None
        if self._callable is None:              # device functor (large shape, or a python predicate): energy + wall
            e_new = torch.empty(self.n_chains, dtype=torch.float64, device=self.device)
            rej = torch.empty(self.n_chains, dtype=torch.uint8, device=self.device)
            self._launch(self._lib.me_energy_builtin(self._h, _ptr(prop), _ptr(e_new), _ptr(rej), self._stream()))
        if self.reject_condition is not None:                                               # ME:227, ME:247
            r, c = self._split(prop)
            mask = torch.as_tensor(self.reject_condition(r, c), device=self.device)
            mask = (mask.to(torch.uint8).expand(self.n_chains).contiguous() if mask.dim() == 0
                    else mask.to(torch.uint8).contiguous())
            rej = mask if rej is None else torch.maximum(rej, mask)
        if self._callable is not None:
            e_new = self._eval_callable(prop)
        self._launch(self._lib.me_accept(self._h, _ptr(prop), _ptr(e_new), _ptr(rej), _ptr(inj_u), self._stream()))
        self.step_counter += 1 if self._kind == "complex" else 0

    def _replay_steps(self, k):
        """``k`` unfused steps as one CUDA-graph launch.  Kernel parameters are frozen at capture, so the step index
        and the measure counter live in a device copy (``me_device_counters``) that the accept kernel advances; the
        handle's own counters are moved by hand after each replay."""
        n, s0 = ctypes.c_int64(), ctypes.c_uint64()
        self._lib.me_get_counters(self._h, ctypes.byref(n), ctypes.byref(s0))
        g = self._graphs.get(k)
        if g is None:
            self._check(self._lib.me_device_counters(self._h, 1, self._stream()))
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for _ in range(k):
                    self._step_external()                    # recorded, not executed
            self._graphs[k] = g
            self._check(self._lib.me_set_counters(self._h, n.value, s0.value))      # capture moved the host counters
            self.step_counter -= k if self._kind == "complex" else 0
        self._check(self._lib.me_device_counters(self._h, 1, self._stream()))         # device copy <- (step, n_measure)
        g.replay()
        self.launch_count += 1
        self._check(self._lib.me_set_counters(self._h, n.value, s0.value + k))
        self._check(self._lib.me_device_counters(self._h, 0, self._stream()))
        self.step_counter += k if self._kind == "complex" else 0

    def measure(self):
        """Running means, covariance recursion, observable means and one time-series row (ME:342-427)."""
        if self.record:
            (t, row0, rows), = self._ts_segments(1)
            self._launch(self._lib.me_run(self._h, 1, 0, 1, _ptr(t), row0, self._stream()))
        else:
            self._launch(self._lib.me_run(self._h, 1, 0, 1, None, 0, self._stream()))
        self._pool_pending += self.n_chains
        if self._term_series is not None and self.record:
            full = self.state[:self._d]
            for tname, fn in self._terms["all"].items():
                self._term_series.setdefault(tname, []).append(self._eval_term(fn, full).clone())

    def run_injected(self, delta, u, n_measures, steps_per_measure, do_measure=True):
        """Parity mode (strict engines): drive the schedule with recorded draws (SURVEY §8c level L-A).
        ``delta``: [steps, D] or [steps, D, n_chains] increments in the order [real, Re c, Im c];
        ``u``: [steps] or [steps, n_chains] accept uniforms, NaN where none was drawn."""
        if self._ladder is not None:
            raise NotImplementedError("temperature ladders run on Philox draws only (no draw injection)")
        S = int(n_measures) * int(steps_per_measure)
        delta = torch.as_tensor(np.asarray(delta, dtype=np.float64), device=self.device)
        u = torch.as_tensor(np.asarray(u, dtype=np.float64), device=self.device)
        if delta.dim() == 2:
            delta = delta[:, :, None].expand(S, self._d, self.n_chains)
        if u.dim() == 1:
            u = u[:, None].expand(S, self.n_chains)
        delta, u = delta.contiguous(), u.contiguous()
        assert delta.shape == (S, self._d, self.n_chains) and u.shape == (S, self.n_chains)
        if self._unfused() or self._generic:      # runtime shapes inject one step at a time (me_propose / me_accept)
            s = 0
            for _ in range(int(n_measures)):
                for _ in range(int(steps_per_measure)):
                    self._step_external(delta[s], u[s])
                    s += 1
                if do_measure:
                    self.measure()
            return
        ts, row0 = None, 0
        if self.record and do_measure:
            segs = self._ts_segments(int(n_measures))
            if len(segs) != 1:
                raise RuntimeError("run_injected spans time-series chunks; use a smaller schedule")
            ts, row0, _ = segs[0]
        self._launch(self._lib.me_run_injected(self._h, int(n_measures), int(steps_per_measure), int(bool(do_measure)),
                                              _ptr(delta), _ptr(u), _ptr(ts), row0, self._stream()))
        if do_measure:
            self._pool_pending += int(n_measures) * self.n_chains
        self.step_counter += S if self._kind == "complex" else 0

    # ------------------------------------------------------------------ counters
    @property
    def measure_step_counter(self):                                                        # ME:73
        n, s = ctypes.c_int64(), ctypes.c_uint64()
        self._lib.me_get_counters(self._h, ctypes.byref(n), ctypes.byref(s))
        return n.value

    @property
    def steps_done(self):
        n, s = ctypes.c_int64(), ctypes.c_uint64()
        self._lib.me_get_counters(self._h, ctypes.byref(n), ctypes.byref(s))
        return s.value

    # ------------------------------------------------------------------ per-chain device views
    def _rows(self, off, n):
        return self.state[off:off + n]

    @property
    def real_params_per_chain(self):
        return self._rows(self._lay.X, self.num_real_params).t()

    @property
    def complex_params_per_chain(self):
        nr, nc = self.num_real_params, self.num_complex_params
        return torch.complex(self._rows(nr, nc), self._rows(nr + nc, nc)).t()

    @property
    def energy_per_chain(self):
        return self.state[self._lay.E]

    @property
    def real_group_sampling_width_per_chain(self):
        return self.state[self._lay.SIG]

    @property
    def complex_group_sampling_width_per_chain(self):
        return self.state[self._lay.SIG + 1]

    @property
    def sampling_width_per_chain(self):
        return self.state[self._lay.SIG + (1 if self._kind == "complex" else 0)]

    @property
    def real_mean_per_chain(self):
        return self._rows(self._lay.MEAN, self.num_real_params).t()

    @property
    def complex_mean_per_chain(self):
        nr, nc = self.num_real_params, self.num_complex_params
        m = self._lay.MEAN
        return torch.complex(self._rows(m + nr, nc), self._rows(m + nr + nc, nc)).t()

    @property
    def observables_mean_per_chain(self):
        return self._rows(self._lay.OBSM, 2 * self.num_real_params + self.num_complex_params).t()

    def _unpack_sym(self, off):
        nr = self.num_real_params
        out = torch.zeros((self.n_chains, nr, nr), dtype=torch.float64, device=self.device)
        for i in range(nr):
            for j in range(i + 1):
                v = self.state[off + i * (i + 1) // 2 + j]
                out[:, i, j] = v
                out[:, j, i] = v
        return out

    def _unpack_herm(self, off, lower_only=False):
        nc = self.num_complex_params
        out = torch.zeros((self.n_chains, nc, nc), dtype=torch.complex128, device=self.device)
        dg = nc * (nc - 1)
        for i in range(nc):
            out[:, i, i] = self.state[off + dg + i].to(torch.complex128)
            for j in range(i):
                p = 2 * (i * (i - 1) // 2 + j)
                v = torch.complex(self.state[off + p], self.state[off + p + 1])
                out[:, i, j] = v
                if not lower_only:
                    out[:, j, i] = v.conj()
        return out

    @property
    def covariance_matrix_real_per_chain(self):
        return self._unpack_sym(self._lay.COVR)

    @property
    def covariance_matrix_complex_per_chain(self):
        return self._unpack_herm(self._lay.COVC)

    @property
    def accept_count_per_chain(self):
        return self.state[self._lay.NACC]

    @property
    def status_per_chain(self):
        return self.state[self._lay.STATUS].to(torch.int32)

    def check_status(self):
        """Raise the exception the reference would have raised for a device-side fault (SURVEY §5)."""
        st = self.status_per_chain
        bad = int(st.max().item()) if st.numel() else 0
        if bad & _lib.STATUS_NOT_PSD:
            raise ValueError("covariance is not symmetric positive-semidefinite.")           # numpy's message, ME:270
        if bad & _lib.STATUS_SIGMA_NONPOS:
            raise AssertionError("sampling_width > 0 violated")                              # ME:438
        if bad & _lib.STATUS_ENERGY_NAN:
            raise FloatingPointError("energy functor returned NaN")

    # ------------------------------------------------------------------ pooled reads (reference attribute names)
    def _pooled(self, t):
        """Mean over all chains of the job of a per-chain tensor [n_chains, ...] -> numpy.  Ladder engines: mean over
        the ladders, per rung -> [R, ...] (a shard holds whole ladders, so local chain i is rung i % R)."""
        if self._ladder is not None:
            R = self._ladder.size
            s = t.reshape((self.n_chains // R, R) + tuple(t.shape[1:])).sum(dim=0)
            count = self.n_chains_total // R
        else:
            s, count = t.sum(dim=0), self.n_chains_total
        if self._distributed:
            parallel.allreduce_sum_(s, self._group)
        return (s / count).cpu().numpy()

    def _pooled_scalar(self, t):
        """``_pooled`` of a per-chain scalar [n_chains]: a float, or numpy [R] for a ladder engine."""
        v = self._pooled(t[:, None])[..., 0]
        return float(v) if self._ladder is None else v

    def _single(self):
        return self.n_chains_total == 1

    @property
    def real_params(self):
        if self._single():
            return self.real_params_per_chain[0].cpu().numpy()
        return self.real_params_per_chain

    @property
    def complex_params(self):
        if self._single():
            return self.complex_params_per_chain[0].cpu().numpy()
        return self.complex_params_per_chain

    @property
    def real_mean(self):                                                                   # ME:77
        return self._pooled(self.real_mean_per_chain)

    @property
    def complex_mean(self):                                                                # ME:78
        return self._pooled(self.complex_mean_per_chain)

    @property
    def covariance_matrix_real(self):                                                      # ME:63-66
        return self._pooled(self.covariance_matrix_real_per_chain) if self.num_real_params else None

    @property
    def covariance_matrix_complex(self):                                                   # ME:67-70
        return self._pooled(self.covariance_matrix_complex_per_chain) if self.num_complex_params else None

    @property
    def observables_mean(self):                                                            # ME:80-81
        return self._pooled(self.observables_mean_per_chain)

    @property
    def observables(self):                                                                 # ME:458-463
        nr, nc = self.num_real_params, self.num_complex_params
        x = self.state[:self._d]
        obs = torch.cat([x[:nr].abs(), torch.hypot(x[nr:nr + nc], x[nr + nc:nr + 2 * nc]), x[:nr] * x[:nr]], dim=0)
        return self._pooled(obs.t())

    @property
    def real_group_sampling_width(self):                                                   # ME:98
        return self._pooled_scalar(self.real_group_sampling_width_per_chain)

    @property
    def complex_group_sampling_width(self):                                                # ME:99
        return self._pooled_scalar(self.complex_group_sampling_width_per_chain)

    @property
    def sampling_width(self):
        """ME:97.  Only the mixed ``step_all`` adapts this attribute; all-real / all-complex engines adapt their
        group width and leave it at its initial value (SURVEY App. B-1)."""
        if self._kind == "mixed":
            return self.real_group_sampling_width
        if self._width_pair is not None:
            raise AttributeError("sampling_width is undefined when the widths were given as [sigma_real, "
                                 "sigma_complex] (ME:93-95); read the group widths")
        return self._sampling_width0

    @property
    def energy_total(self):
        """ME:125.  Live for mixed engines (ME:255); all-real / all-complex engines leave it at its initial value
        and keep the live energy in ``energy`` (SURVEY App. B-1)."""
        src = self.state[self._lay.E] if self._kind == "mixed" else self._energy0
        return self._pooled_scalar(src)

    @property
    def energy(self):
        """ME:152-156: dict of energy terms.  Single-callable engines have the one key ``"total"`` holding the live
        energy; for dict-of-terms engines each term is re-evaluated on the current state."""
        if self._terms is None:
            return {"total": self._pooled_scalar(self.state[self._lay.E])}
        full = self.state[:self._d]
        return {t: self._pooled_scalar(self._eval_term(fn, full)) for t, fn in self._terms["all"].items()}

    @property
    def acceptance_rate(self):
        steps = self.steps_done
        if steps == 0:
            return float("nan")
        return self._pooled_scalar(self.accept_count_per_chain) / steps

    # ------------------------------------------------------------------ temperature ladders
    @property
    def temperatures(self):
        """The temperatures, numpy [R] (R = 1 for a scalar ``temp``)."""
        return self._ladder.copy() if self._ladder is not None else np.array([float(self.temp)])

    @property
    def rung_consts(self):
        """Functor constants of every rung of a Hamiltonian ladder, numpy [R, K] (None for other engines)."""
        return None if self._rung_consts is None else self._rung_consts.copy()

    @property
    def rung_per_chain(self):
        """Rung of every local chain, int64 [n_chains]: global chain g is rung g % R."""
        R = 1 if self._ladder is None else self._ladder.size
        return torch.arange(self.chain_offset, self.chain_offset + self.n_chains, device=self.device) % R

    @property
    def walker_per_chain(self):
        """Label of the walker (the global id of the chain it started in) whose configuration each chain holds."""
        if self._ladder is None:
            return torch.arange(self.chain_offset, self.chain_offset + self.n_chains, dtype=torch.int32,
                                device=self.device)
        return self._walker

    def _swap_attempts(self):
        """Replica-exchange rounds each neighbour pair (r, r + 1) took part in, per ladder, numpy [R - 1]: rounds
        k = n / swap_every over the measure counters n = 2 .. measure_step_counter, pair r in rounds k = r (mod 2)."""
        R, e = self._ladder.size, self._swap_every
        first, last = -(-2 // e), self.measure_step_counter // e
        out = np.zeros(R - 1, dtype=np.int64)
        for r in range(R - 1):
            k0 = first + ((r - first) % 2)                  # first round >= first with k = r (mod 2)
            out[r] = max(0, (last - k0) // 2 + 1) if last >= k0 else 0
        return out

    @property
    def swap_acceptance_rate(self):
        """Accepted over attempted swaps of every neighbour pair (r, r + 1), numpy [R - 1], pooled over ladders and
        ranks (NaN before the first round of a pair)."""
        if self._ladder is None or not self._swap_every:
            raise AttributeError("swap_acceptance_rate needs a ladder engine with replica_exchange > 0")
        R = self._ladder.size
        acc = self._swap_acc.to(torch.int64).reshape(self.n_chains // R, R).sum(dim=0).to(torch.float64)
        if self._distributed:
            parallel.allreduce_sum_(acc, self._group)
        att = self._swap_attempts() * (self.n_chains_total // R)
        with np.errstate(invalid="ignore", divide="ignore"):
            return acc.cpu().numpy()[:R - 1] / att

    # ------------------------------------------------------------------ clean pooled ensemble statistics
    def _library_comm(self):
        if self._distributed and self._comm is None:
            self._comm = parallel.library_comm(self._lib, self.device.index, self._group)
        return self._comm if self._distributed else None

    def _flush_pool(self):
        """Per-CTA accumulators -> fixed-order sum -> all-reduce across ranks (NCCL, inside the library) -> device
        totals.  Stream-ordered, no host synchronisation."""
        self._launch(self._lib.me_allreduce_stats(self._h, self._library_comm(), _ptr(self._pool_inc),
                                                  _ptr(self._pool_tot), int(self._pool_pending), self._stream()))
        self._pool_pending = 0

    def pooled_statistics(self):
        """Ensemble mean / covariance / observable means over every (chain, measure) sample of the whole job,
        from the in-kernel shifted moments; across ranks this is the path's one all-reduce (SURVEY §8e), issued inside
        the library (``me_allreduce_stats``).  The moments stay on the device; this call is their one read-back."""
        pw = self._lay.POOL_WORDS
        if pw == 0:
            raise NotImplementedError("parameter space too large for in-kernel pooled moments")
        if self._pool is None:
            raise NotImplementedError("pooled moments per rung need a ladder of 2, 4, 8, 16 or 32 rungs")
        if self._distributed and self._library_comm() is None:
            # no NCCL group (e.g. gloo on a CPU-only rendezvous): reduce locally, sum across ranks through torch
            self._launch(self._lib.me_allreduce_stats(self._h, None, _ptr(self._pool_inc), _ptr(self._pool_tot),
                                                      int(self._pool_pending), self._stream()))
            self._pool_pending = 0
            tot = parallel.allreduce_sum_(self._pool_tot.clone(), self._group).cpu().numpy()
        else:
            self._flush_pool()
            tot = self._pool_tot.cpu().numpy()
        if self._ladder is not None:          # rung-major rows of pw words; every rung has the same sample count
            R = self._ladder.size
            if tot[-1] / R < 2:
                raise RuntimeError("pooled statistics need at least two measured samples")
            per = [parallel.finalize_pooled(tot[r * pw:(r + 1) * pw], tot[-1] / R, self._shift_host,
                                            self.num_real_params, self.num_complex_params) for r in range(R)]
            return {k: np.stack([np.asarray(p[k]) for p in per]) for k in per[0]}
        if tot[-1] < 2:
            raise RuntimeError("pooled statistics need at least two measured samples")
        return parallel.finalize_pooled(tot[:pw], tot[-1], self._shift_host, self.num_real_params,
                                        self.num_complex_params)

    def reset_pooled_statistics(self):
        """Forget the pooled moments accumulated so far (e.g. after burn-in)."""
        if self._pool is not None:
            self._launch(self._lib.me_pool_reduce(self._h, _ptr(self._pool_out), 1, self._stream()))
        self._pool_tot.zero_()
        self._pool_pending = 0

    # ------------------------------------------------------------------ output (ME:466-479)
    def time_series(self):
        """All recorded rows as one tensor [rows, TS_COLS, n_chains] (columns: parameters in the order
        [real, Re c, Im c], live energy, sampling width — both group widths for mixed engines)."""
        parts = [t[:used] for t, used in self._ts_chunks if used]
        if not parts:
            return torch.empty((0, self._lay.TS_COLS, self.n_chains), dtype=torch.float64, device=self.device)
        return parts[0] if len(parts) == 1 else torch.cat(parts, dim=0)

    def save_time_series(self, chain=0):
        """Build ``self.df`` for one chain with the reference's columns and order (ME:466-478): observables,
        ``<term>_energy``, real parameters + ``real_group_sampling_width``, complex parameters +
        ``complex_group_sampling_width``.  Derived columns (abs, squares) are recomputed from the stored
        parameters.  Unlike the reference nothing is printed (SURVEY App. B-12)."""
        import pandas
        nr, nc, d = self.num_real_params, self.num_complex_params, self._d
        parts = [t[:used, :, chain] for t, used in self._ts_chunks if used]
        rows = (torch.cat(parts, dim=0) if parts else torch.empty((0, self._lay.TS_COLS), dtype=torch.float64)).cpu().numpy()
        x = rows[:, :nr]
        c = rows[:, nr:nr + nc] + 1j * rows[:, nr + nc:d]
        cols = {}
        for i in range(nr):
            cols[self.observables_names[i]] = np.abs(x[:, i])
        for j in range(nc):
            cols[self.observables_names[nr + j]] = np.abs(c[:, j])
        for i in range(nr):
            cols[self.observables_names[nr + nc + i]] = x[:, i] * x[:, i]
        if self._terms is None:
            cols["total_energy"] = rows[:, d]
        else:
            for tname in self._terms["all"]:
                ser = self._term_series.get(tname, [])
                cols[tname + "_energy"] = np.array([v[chain].item() for v in ser]) if ser else np.zeros(0)
        if nr:
            for i in range(nr):
                cols[self.params_names[i]] = x[:, i]
            cols["real_group_sampling_width"] = rows[:, d + 1]
        if nc:
            for j in range(nc):
                cols[self.params_names[nr + j]] = c[:, j]
            cols["complex_group_sampling_width"] = rows[:, d + 2] if self._kind == "mixed" else rows[:, d + 1]
        self.df = pandas.DataFrame.from_dict(cols)
        return self.df

    def to_csv(self, path, chain=0):
        """On-disk time series of one chain in the reference's format (SURVEY §8 row f2): the columns of
        ``save_time_series`` written with ``DataFrame.to_csv`` — complex parameters print as ``(a+bj)``, exactly
        like the reference's recorded ``exampledata.csv``; readable by its ``statistics.py:7-23``."""
        df = self.save_time_series(chain)
        df.to_csv(path)
        return path

    def save_npz(self, path):
        """Dense binary dump of every recorded row of every local chain (for 1e9-row ensembles where CSV is
        hopeless): ``rows[row, column, chain]`` with ``columns`` = parameters in the order [real, Re c, Im c],
        ``energy``, ``sampling_width``; plus names and the chain offset of this rank."""
        ts = self.time_series().cpu().numpy()
        nr, nc = self.num_real_params, self.num_complex_params
        cols = ([self.params_names[i] for i in range(nr)] + ["Re_" + self.params_names[nr + j] for j in range(nc)]
                + ["Im_" + self.params_names[nr + j] for j in range(nc)] + ["energy"]
                + (["real_group_sampling_width", "complex_group_sampling_width"] if self._kind == "mixed"
                   else ["sampling_width"]))
        np.savez_compressed(path, rows=ts, columns=np.array(cols), chain_offset=self.chain_offset,
                            observables_names=np.array(self.observables_names))
        return path

    def statistical_inefficiency(self, column=0, n_chains=1024, burn_in=0.2, max_lag=0):
        """Per-chain statistical inefficiency g (in units of measures) of one stored time-series column
        (``column`` indexes [parameters in the order real, Re c, Im c | energy | sigma]) for the first ``n_chains``
        local chains, discarding the first ``burn_in`` fraction of rows — the quantity the reference's
        ``save_equilibrium_stats`` gets from pymbar (ME:490, statistics.py:36-38).  ESS per chain = rows / g."""
        chunks = [(t, used) for t, used in self._ts_chunks if used]
        if len(chunks) != 1:
            raise RuntimeError("statistical_inefficiency needs the series in one storage chunk (raise ts_chunk_bytes)")
        t, used = chunks[0]
        n_sel = min(int(n_chains), self.n_chains)
        g = torch.empty(n_sel, dtype=torch.float64, device=self.device)
        rc = self._lib.me_statistical_inefficiency(_ptr(t), used, int(used * burn_in), self._lay.TS_COLS, self.n_chains,
                                                   int(column), 0, n_sel, int(max_lag), _ptr(g), self._stream())
        if rc != 0:
            raise ValueError("bad arguments to me_statistical_inefficiency")
        return g

    def _equilibration_kernel(self, block, col, n_sel, nskip, fast=True):
        """(t0, g, Neff_max) tensors [n_sel] for column ``col`` of a block [rows, cols, ld] on the device."""
        rows, cols, ld = block.shape
        n_cand = (rows - 1 + nskip - 1) // nskip
        scratch = torch.empty(2 * n_cand * n_sel, dtype=torch.float64, device=self.device)
        out = torch.empty((3, n_sel), dtype=torch.float64, device=self.device)
        rc = self._lib.me_detect_equilibration(_ptr(block), rows, cols, ld, int(col), 0, n_sel, int(nskip), int(bool(fast)),
                                               _ptr(scratch), scratch.numel(), _ptr(out[0]), _ptr(out[1]), _ptr(out[2]),
                                               self._stream())
        if rc != 0:
            raise ValueError("bad arguments to me_detect_equilibration (need at least 3 recorded rows)")
        return out[0].long(), out[1], out[2]

    def detect_equilibration(self, column=0, n_chains=1024, nskip=1, fast=True):
        """Per-chain start of the production region ``t0`` (in measures), statistical inefficiency ``g`` and
        ``Neff_max`` of one stored column for the first ``n_chains`` local chains: pymbar's ``detectEquilibration``
        (what the reference's ``save_equilibrium_stats`` evaluates per data-frame column, ME:490, statistics.py:25-48)
        as a device kernel — one thread per (chain, candidate t0).  ``nskip`` thins the candidates (pymbar's own
        parameter; use ~rows/100 for long series)."""
        chunks = [(t, used) for t, used in self._ts_chunks if used]
        if len(chunks) != 1:
            raise RuntimeError("detect_equilibration needs the series in one storage chunk (raise ts_chunk_bytes)")
        t, used = chunks[0]
        return self._equilibration_kernel(t[:used], column, min(int(n_chains), self.n_chains), nskip, fast)

    def save_equilibrium_stats(self, external_df=None, chain=0, nskip=1):
        """The reference's post-run summary for one chain (ME:481-504).  ``external_df``: a list of data frames of
        external observables recorded alongside the run (the cylinder app's field profiles); those whose first entry is
        a float or int join the equilibration analysis (ME:485-487), and every one of them is re-averaged from the
        global cut-off (ME:494-502: ``field_profile`` / ``field_abs_profile`` are the first two).  ``eq_means_error`` is
        the empty dict the reference's ``get_equilibrated_means`` returns (statistics.py:59,64: never filled).
        ``eq_points`` = {column: [t0, g, Neff_max]} for every non-constant data-frame column (complex ones split into
        ``_real`` / ``_imag``, statistics.py:25-48), ``global_eq_point`` = the largest t0 among the columns that are
        not sampling widths (ME:492), ``equilibrated_means`` = column means from that row on (statistics.py:53-64)
        plus ``"global_cutoff"``.  The series are analysed on the device (me_detect_equilibration)."""
        import pandas
        own = self.save_time_series(chain)
        df = own
        if external_df is not None:                                                          # ME:485-487
            keep = [own] + [e for e in external_df if isinstance(e.iloc[0, 0], (float, int, np.floating, np.integer))]
            df = pandas.concat(keep, axis=1)
        names, series = [], []
        for name in df.columns.values:
            col = df[name].to_numpy()
            if np.iscomplexobj(col):
                parts = ((name + "_real", col.real), (name + "_imag", col.imag))
            else:
                parts = ((name, col.astype(np.float64)),)
            if df[name].nunique() > 1:                                           # statistics.py:33 "ignore const series"
                for n_, v in parts:
                    names.append(n_)
                    series.append(v)
        self.eq_points = {}
        if series:
            # one block [rows, columns, 1]: every data-frame column is analysed by the same kernel
            block = torch.tensor(np.stack(series, axis=1)[:, :, None], dtype=torch.float64, device=self.device).contiguous()
            for k, n_ in enumerate(names):
                t0, g, neff = self._equilibration_kernel(block, k, 1, nskip)
                self.eq_points[n_] = [int(t0.item()), float(g.item()), float(neff.item())]
        cut = [t for key, (t, _g, _n) in self.eq_points.items() if "sampling_width" not in key]
        self.global_eq_point = max(cut) if cut else 0
        def means_from(frame):                                                              # statistics.py:53-64
            # (the reference averages every column and would raise on a string-valued external frame; those are skipped)
            return {name: np.average(frame.loc[self.global_eq_point:, name]) for name in frame.columns.values
                    if pandas.api.types.is_numeric_dtype(frame[name])}

        self.equilibrated_means, self.eq_means_error = means_from(own), {}                  # ME:494
        if external_df is not None:                                                          # ME:495-502
            profiles = [means_from(e) for e in external_df]
            self.field_profile = profiles[0] if len(profiles) > 0 else None
            self.field_abs_profile = profiles[1] if len(profiles) > 1 else None
        self.equilibrated_means["global_cutoff"] = self.global_eq_point
        return self.eq_points

    # ------------------------------------------------------------------ checkpoint / resume (SURVEY §5)
    def state_dict(self):
        n, s = ctypes.c_int64(), ctypes.c_uint64()
        self._lib.me_get_counters(self._h, ctypes.byref(n), ctypes.byref(s))
        return dict(state=self.state.clone(), n_measure=n.value, step=s.value, seed=self.seed,
                    chain_offset=self.chain_offset, pool=None if self._pool is None else self._pool.clone(),
                    pool_tot=self._pool_tot.clone(), pool_pending=self._pool_pending,
                    walker=None if self._walker is None else self._walker.clone(),
                    swap_acc=None if self._swap_acc is None else self._swap_acc.clone())

    def load_state_dict(self, sd):
        if sd["state"].shape != self.state.shape:
            raise ValueError("checkpoint shape %s does not match engine %s" % (tuple(sd["state"].shape),
                                                                             tuple(self.state.shape)))
        self.state.copy_(sd["state"])
        if self._pool is not None and sd.get("pool") is not None:
            self._pool.copy_(sd["pool"])
        self._pool_tot.copy_(sd["pool_tot"])
        self._pool_pending = int(sd["pool_pending"])
        if self._walker is not None:
            self._walker.copy_(sd["walker"])
            self._swap_acc.copy_(sd["swap_acc"])
        self._check(self._lib.me_set_counters(self._h, int(sd["n_measure"]), int(sd["step"])))
        if self._ctr_on:
            self._check(self._lib.me_device_counters(self._h, 1, self._stream()))

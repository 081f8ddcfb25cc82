"""ctypes binding of libme_b200.so (C ABI: include/me_b200.h).

There is no CPU fallback: if the library has not been built (``python -c "import __graft_entry__ as g; g.build()"``
or ``make -C metropolisengine_b200/csrc``) loading raises, and every engine operation needs a CUDA device.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ME_B200_LIB") or os.path.join(HERE, "lib", "libme_b200.so")   # override: kernel experiments

ME_ABI_VERSION = 10

ME_OK, ME_ERR_INVALID, ME_ERR_CUDA, ME_ERR_COMPILE, ME_ERR_UNSUPPORTED, ME_ERR_STATE = range(6)

ENERGY_IDS = {"x2": 0, "xy_well": 1, "mixed_well": 2, "cylinder": 3}
ENERGY_EXTERNAL = 99
ENERGY_USER = 100

STATUS_NOT_PSD, STATUS_SIGMA_NONPOS, STATUS_ENERGY_NAN = 1, 2, 4

_i32, _i64, _u64, _f64 = ctypes.c_int32, ctypes.c_int64, ctypes.c_uint64, ctypes.c_double
_vp, _cp = ctypes.c_void_p, ctypes.c_char_p


class MeConfig(ctypes.Structure):
    _fields_ = [("n_real", _i32), ("n_complex", _i32), ("n_chains", _i64), ("chain_offset", _i64),
                ("temp", _f64), ("target_acceptance", _f64), ("ratio", _f64), ("seed", _u64),
                ("device", _i32), ("strict", _i32)]


class MeLayout(ctypes.Structure):
    _fields_ = [(k, _i32) for k in ("X", "E", "SIG", "MEAN", "COVR", "COVC", "OBSM", "FACR", "FACC", "NACC",
                                    "STATUS", "WORDS", "D", "TS_COLS", "POOL_WORDS")]


class MeBuffers(ctypes.Structure):
    _fields_ = [("state", _vp), ("pool", _vp), ("shift", _vp), ("last_accept", _vp), ("scratch", _vp), ("prop", _vp)]


class MeK4Config(ctypes.Structure):
    _fields_ = [("n_real", _i32), ("n_complex", _i32), ("n_chains", _i64), ("chain_offset", _i64),
                ("temp", _f64), ("target_acceptance", _f64), ("ratio", _f64), ("seed", _u64),
                ("device", _i32), ("use_reject", _i32), ("consts", _f64 * 4)]


class MeK4Layout(ctypes.Structure):
    _fields_ = [(k, _i32) for k in ("X", "E", "SIG", "MEAN", "OBSM", "NACC", "STATUS", "WORDS", "D", "TS_COLS",
                                    "N_COMPLEX", "TILE", "FACTOR_BYTES", "MOM_WORDS", "MOM_SCRATCH_PER_SM", "SUM_GROUPS")]


# every symbol include/me_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "me_abi_version": (ctypes.c_int, []),
    "me_state_layout": (ctypes.c_int, [_i32, _i32, ctypes.POINTER(MeLayout)]),
    "me_create": (ctypes.c_int, [ctypes.POINTER(MeConfig), ctypes.POINTER(_vp)]),
    "me_destroy": (ctypes.c_int, [_vp]),
    "me_set_energy_builtin": (ctypes.c_int, [_vp, _i32, ctypes.POINTER(_f64), _i32, _i32]),
    "me_set_energy_source": (ctypes.c_int, [_vp, _cp, ctypes.POINTER(_f64), _i32, _i32]),
    "me_set_energy_external": (ctypes.c_int, [_vp]),
    "me_check_energy_source": (ctypes.c_int, [_cp, _i32, _i32, _i32, _i32, _cp, _i64]),
    "me_set_group": (ctypes.c_int, [_vp, _i32]),
    "me_set_ladder": (ctypes.c_int, [_vp, ctypes.POINTER(_f64), _i32, _i64, _vp, _vp]),
    "me_set_hamiltonian_ladder": (ctypes.c_int, [_vp, ctypes.POINTER(_f64), ctypes.POINTER(_f64), _i32, _i32, _i64, _vp,
                                                 _vp]),
    "me_launch_dims": (ctypes.c_int, [_vp, ctypes.POINTER(_i32), ctypes.POINTER(_i32)]),
    "me_bind": (ctypes.c_int, [_vp, ctypes.POINTER(MeBuffers)]),
    "me_init": (ctypes.c_int, [_vp, _vp, _i32, _f64, _vp, _vp, _vp, _vp, _vp]),
    "me_run": (ctypes.c_int, [_vp, _i64, _i64, _i32, _vp, _i64, _vp]),
    "me_run_injected": (ctypes.c_int, [_vp, _i64, _i64, _i32, _vp, _vp, _vp, _i64, _vp]),
    "me_propose": (ctypes.c_int, [_vp, _vp, _vp, _vp]),
    "me_accept": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "me_energy_builtin": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "me_pool_reduce": (ctypes.c_int, [_vp, _vp, _i32, _vp]),
    "me_comm_set_library": (ctypes.c_int, [_cp]),
    "me_comm_unique_id": (ctypes.c_int, [_vp]),
    "me_comm_create": (ctypes.c_int, [_vp, _i32, _i32, _i32, ctypes.POINTER(_vp)]),
    "me_comm_adopt": (ctypes.c_int, [_vp, _i32, _i32, _i32, ctypes.POINTER(_vp)]),
    "me_comm_destroy": (ctypes.c_int, [_vp]),
    "me_comm_last_error": (_cp, []),
    "me_allreduce_stats": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _vp]),
    "me_reduce_stats": (ctypes.c_int, [_vp, _vp, _i64, _vp]),
    "me_comm_peer_init": (ctypes.c_int, [_vp, _i64, _vp]),
    "me_comm_peer_connect": (ctypes.c_int, [_vp, _vp]),
    "me_comm_peer_enable": (ctypes.c_int, [_vp, ctypes.c_int32]),
    "me_comm_allreduce": (ctypes.c_int, [_vp, _vp, _i64, _vp]),
    "me_accumulate_stats": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "me_get_counters": (ctypes.c_int, [_vp, ctypes.POINTER(_i64), ctypes.POINTER(_u64)]),
    "me_set_counters": (ctypes.c_int, [_vp, _i64, _u64]),
    "me_k4_layout_get": (ctypes.c_int, [ctypes.POINTER(MeK4Layout)]),
    "me_k4_create": (ctypes.c_int, [ctypes.POINTER(MeK4Config), ctypes.POINTER(_vp)]),
    "me_k4_destroy": (ctypes.c_int, [_vp]),
    "me_k4_bind": (ctypes.c_int, [_vp, _vp, _vp, _vp]),
    "me_k4_init": (ctypes.c_int, [_vp, _vp, _i32, _f64, _vp]),
    "me_k4_layout_for": (ctypes.c_int, [_i32, ctypes.POINTER(MeK4Layout)]),
    "me_k4_set_energy_source": (ctypes.c_int, [_vp, _cp, ctypes.POINTER(_f64), _i32, _i32]),
    "me_k4_check_energy_source": (ctypes.c_int, [_cp, _i32, _i32, _cp, _i64]),
    "me_k4_step": (ctypes.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "me_k4_step_measure": (ctypes.c_int, [_vp, _i64, _vp, _vp, _i64, _vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    "me_k4_measure": (ctypes.c_int, [_vp, _vp, _i64, _vp]),
    "me_k4_moments": (ctypes.c_int, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    "me_k4_refactor": (ctypes.c_int, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "me_k4_accumulate_moments": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "me_k4_set_factor": (ctypes.c_int, [_vp, _vp]),
    "me_k4_set_reserved_sms": (ctypes.c_int, [_vp, _i32]),
    "me_k4_normal_table": (ctypes.c_int, [_vp, _i32]),
    "me_k4_get_counters": (ctypes.c_int, [_vp, ctypes.POINTER(_i64), ctypes.POINTER(_u64)]),
    "me_k4_last_error": (_cp, [_vp]),
    "me_probe_fp64": (ctypes.c_int, [_i32, _i64, _vp, _i64, _vp, ctypes.POINTER(_i64)]),
    "me_device_counters": (ctypes.c_int, [_vp, _i32, _vp]),
    "me_statistical_inefficiency": (ctypes.c_int, [_vp, _i64, _i64, _i32, _i64, _i32, _i64, _i64, _i64, _vp, _vp]),
    "me_detect_equilibration": (ctypes.c_int, [_vp, _i64, _i32, _i64, _i32, _i64, _i64, _i64, _i32, _vp, _i64, _vp, _vp,
                                               _vp, _vp]),
    "me_mbar_words": (ctypes.c_int, [_vp, _i32, _i32, ctypes.POINTER(_i64)]),
    "me_mbar_pass": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i64, _vp, _i64, _i32, _vp, _vp, _i32, _vp, _i32, _vp]),
    "me_mbar_hist_words": (ctypes.c_int, [_vp, _i32, _vp, ctypes.POINTER(_i64)]),
    "me_mbar_hist_pass": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i64, _vp, _i64, ctypes.c_double, _vp, _i32, _vp, _vp,
                                         _vp, _vp, _vp, _vp, _i32, _vp]),
    "me_mbar_cov_words": (ctypes.c_int, [_vp, _i32, _i32, _i32, ctypes.POINTER(_i64)]),
    "me_mbar_cov_pass": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i64, _vp, _i64, _i32, _vp, _vp, _i32, _i32, _vp, _vp,
                                        _i32, _vp]),
    "me_last_error": (_cp, [_vp]),
}

_lib = None


class MeError(RuntimeError):
    pass


def load():
    """Load libme_b200.so; raises if it has not been built (no fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("libme_b200.so is not built (%s missing): run __graft_entry__.build() or "
                          "`make -C metropolisengine_b200/csrc`; there is no CPU fallback" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)     # AttributeError here = ABI symbol missing
        fn.restype = res
        fn.argtypes = args
    got = lib.me_abi_version()
    if got != ME_ABI_VERSION:
        raise ImportError("libme_b200.so ABI version %d, binding expects %d: rebuild" % (got, ME_ABI_VERSION))
    _lib = lib
    return lib


def layout(n_real, n_complex):
    lay = MeLayout()
    rc = load().me_state_layout(n_real, n_complex, ctypes.byref(lay))
    if rc != ME_OK:
        raise ValueError("invalid parameter-space shape (%d real, %d complex)" % (n_real, n_complex))
    return lay


def check(handle, rc):
    """Map a C return code to the exception the reference would have raised."""
    if rc == ME_OK:
        return
    msg = load().me_last_error(handle)
    msg = msg.decode(errors="replace") if msg else "error %d" % rc
    if rc == ME_ERR_INVALID:
        raise ValueError(msg)
    raise MeError(msg)


def check_energy_source(source, n_real, n_complex, use_reject=False, strict=False):
    """Compile-only check of a CUDA energy functor (works without a GPU).  Returns (ok, log)."""
    buf = ctypes.create_string_buffer(1 << 16)
    rc = load().me_check_energy_source(source.encode() if source is not None else None, n_real, n_complex,
                                       int(use_reject), int(strict), buf, len(buf))
    return rc == ME_OK, buf.value.decode(errors="replace")

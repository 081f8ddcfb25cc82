"""ctypes front-end of the ladder oracle (oracle/me_oracle_ladder.c).  TEST INFRASTRUCTURE ONLY — the product package
never imports this module.  The rungs are initialised by the scalar oracle (``c_oracle.CChain``); the ladder library is
the scalar oracle compiled together with ``meo_run_ladder`` / ``meo_swap_uniform``."""
import ctypes
import os
import subprocess

import numpy as np

from oracle.c_oracle import CChain, _dp

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "me_oracle_ladder.c")
DEPS = (SRC, os.path.join(HERE, "me_oracle.c"))
LIB = os.path.join(HERE, "libme_oracle_ladder.so")


def build(force=False):
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(p) for p in DEPS):
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", LIB, SRC, "-lm"])
    return LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
        _lib.meo_swap_uniform.restype = ctypes.c_double
        _lib.meo_swap_uniform.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int64]
        _lib.meo_run_ladder.restype = ctypes.c_int
    return _lib


class CLadder:
    """One temperature ladder of the C oracle (``meo_run_ladder``): R chains with the global ids chain0 .. chain0 + R - 1,
    rung r at ``temps[r]``, replica-exchange rounds every ``swap_every`` measures (0 = none).  Keyword arguments as
    ``CChain``; ``x0`` is one start for every rung or an [R, d] array."""

    def __init__(self, n_r, n_c, energy, temps, swap_every=1, x0=None, chain0=0, **kw):
        self.temps = np.ascontiguousarray(temps, dtype=np.float64)
        R = self.R = len(self.temps)
        self.swap_every, self.chain0 = int(swap_every), int(chain0)
        x0 = np.broadcast_to(np.asarray(x0, dtype=np.float64), (R, n_r + 2 * n_c))
        self.chains = [CChain(n_r, n_c, energy, temp=float(self.temps[r]), x0=x0[r], **kw) for r in range(R)]
        self.cfg, self.off, self.d = self.chains[0].cfg, self.chains[0].off, self.chains[0].d
        self.states = np.ascontiguousarray(np.stack([ch.state for ch in self.chains]))
        self.n_measure = ctypes.c_int64(1)
        self.walker = np.arange(self.chain0, self.chain0 + R, dtype=np.int32)
        self.swap_acc = np.zeros(R, dtype=np.uint32)
        self.swap_att = np.zeros(R, dtype=np.uint32)

    def run(self, n_blocks, spm, do_measure=True, seed=0, step0=0):
        u32 = ctypes.POINTER(ctypes.c_uint32)
        rc = lib().meo_run_ladder(ctypes.byref(self.cfg), self.R, _dp(self.temps), _dp(self.states),
                                  ctypes.c_int64(self.swap_every), ctypes.c_int64(n_blocks), ctypes.c_int64(spm),
                                  int(do_measure), ctypes.byref(self.n_measure), ctypes.c_uint64(seed),
                                  ctypes.c_uint64(self.chain0), ctypes.c_uint64(step0),
                                  self.walker.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                                  self.swap_acc.ctypes.data_as(u32), self.swap_att.ctypes.data_as(u32))
        assert rc == 0

    @property
    def x(self):
        return self.states[:, self.off.X:self.off.X + self.d]


def swap_uniform(seed, chain, n):
    """The replica-exchange uniform of the pair whose lower rung is global chain ``chain`` at measure counter ``n``."""
    return lib().meo_swap_uniform(seed, chain, n)

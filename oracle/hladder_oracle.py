"""ctypes front-end of the Hamiltonian-ladder oracle (oracle/me_oracle_hladder.c).  TEST INFRASTRUCTURE ONLY — the product
package never imports this module.  The rungs are initialised by the scalar oracle (``c_oracle.CChain``), each with its own
constants; the library is the ladder oracle compiled together with ``meo_run_hladder``."""
import ctypes
import os
import subprocess

import numpy as np

from oracle.c_oracle import CChain, _dp

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "me_oracle_hladder.c")
DEPS = (SRC, os.path.join(HERE, "me_oracle_ladder.c"), os.path.join(HERE, "me_oracle.c"))
LIB = os.path.join(HERE, "libme_oracle_hladder.so")


def build(force=False):
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(p) for p in DEPS):
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", LIB, SRC, "-lm"])
    return LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
        _lib.meo_run_hladder.restype = ctypes.c_int
    return _lib


class CHLadder:
    """One Hamiltonian ladder of the C oracle (``meo_run_hladder``): R chains with the global ids chain0 .. chain0 + R - 1,
    rung r at ``temps[r]`` with the functor constants ``rung_consts[r]``, replica-exchange rounds every ``swap_every``
    measures (0 = none).  ``energy`` is a built-in name or a list of R python callables ``f(x)``, one per rung (each
    closing over its rung's constants: the oracle's callbacks see x only); ``reject`` likewise a list of R predicates or
    None.  Other keyword arguments as ``CChain``; ``x0`` is one start for every rung or an [R, d] array."""

    def __init__(self, n_r, n_c, energy, temps, rung_consts, swap_every=1, x0=None, chain0=0, reject=None, **kw):
        self.temps = np.ascontiguousarray(temps, dtype=np.float64)
        R = self.R = len(self.temps)
        self.rung_consts = np.asarray(rung_consts, dtype=np.float64)
        assert self.rung_consts.shape[0] == R
        self.swap_every, self.chain0 = int(swap_every), int(chain0)
        x0 = np.broadcast_to(np.asarray(x0, dtype=np.float64), (R, n_r + 2 * n_c))
        en = energy if isinstance(energy, (list, tuple)) else [energy] * R
        rej = reject if reject is not None else [None] * R
        self.chains = [CChain(n_r, n_c, en[r], consts=list(self.rung_consts[r]), temp=float(self.temps[r]), x0=x0[r],
                              reject=rej[r], **kw) for r in range(R)]
        self.off, self.d = self.chains[0].off, self.chains[0].d
        self.cfgs = (type(self.chains[0].cfg) * R)(*[ch.cfg for ch in self.chains])
        self.states = np.ascontiguousarray(np.stack([ch.state for ch in self.chains]))
        self.n_measure = ctypes.c_int64(1)
        self.walker = np.arange(self.chain0, self.chain0 + R, dtype=np.int32)
        self.swap_acc = np.zeros(R, dtype=np.uint32)
        self.swap_att = np.zeros(R, dtype=np.uint32)

    def run(self, n_blocks, spm, do_measure=True, seed=0, step0=0):
        u32 = ctypes.POINTER(ctypes.c_uint32)
        rc = lib().meo_run_hladder(self.cfgs, self.R, _dp(self.states), ctypes.c_int64(self.swap_every),
                                   ctypes.c_int64(n_blocks), ctypes.c_int64(spm), int(do_measure),
                                   ctypes.byref(self.n_measure), ctypes.c_uint64(seed), ctypes.c_uint64(self.chain0),
                                   ctypes.c_uint64(step0), self.walker.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                                   self.swap_acc.ctypes.data_as(u32), self.swap_att.ctypes.data_as(u32))
        assert rc == 0

    @property
    def x(self):
        return self.states[:, self.off.X:self.off.X + self.d]

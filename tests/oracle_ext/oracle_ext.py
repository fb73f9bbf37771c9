"""Python handle on the CPU oracle with the extension headers (tests/oracle_ext/librem2d_oracle_ext.so). TEST INFRASTRUCTURE
ONLY: the oracle of oracle/rem2d_oracle.c, unchanged, plus the episode statistics (include/rem2d_stats.h), joint-target stepping
and observations (include/rem2d_control.h) and the test-only sine outputs."""
import ctypes as C
import os
import subprocess

import numpy as np

from gym_rem2d_b200.capi import Engine

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "librem2d_oracle_ext.so")


def build():
    subprocess.check_call(["make", "-s", "-C", HERE])
    return LIB


class OracleExtEngine(Engine):
    def __init__(self, threads=1, **overrides):
        super().__init__(lib_path=build(), **overrides)
        self.lib.rem2d_oracle_set_threads.argtypes = [C.c_void_p, C.c_int]
        self.lib.rem2d_oracle_set_threads(self.h, int(threads))
        self.lib.rem2d_control_sine_outputs.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]

    def sine_outputs(self, T):
        """float64[T, n_joints]: the next T outputs of every joint's sine controller from the current state (nothing changes)."""
        nj = self.pop.n_bodies - self.pop.n_creatures
        out = np.zeros((T, nj), np.float64)
        self._check(self.lib.rem2d_control_sine_outputs(self.h, int(T), out.ctypes.data), "rem2d_control_sine_outputs")
        return out

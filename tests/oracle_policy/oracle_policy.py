"""Python handle on the CPU oracle with the extension headers and the per-joint feedback policy
(tests/oracle_policy/librem2d_oracle_policy.so). TEST INFRASTRUCTURE ONLY: everything of tests/oracle_ext plus rem2d_set_policy
(include/rem2d_policy.h)."""
import ctypes as C
import os
import subprocess
import sys

from gym_rem2d_b200.capi import Engine

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "oracle_ext"))
from oracle_ext import OracleExtEngine  # noqa: E402

LIB = os.path.join(HERE, "librem2d_oracle_policy.so")


def build():
    subprocess.check_call(["make", "-s", "-C", HERE])
    return LIB


class OraclePolicyEngine(OracleExtEngine):
    def __init__(self, threads=1, **overrides):
        Engine.__init__(self, lib_path=build(), **overrides)
        self.lib.rem2d_oracle_set_threads.argtypes = [C.c_void_p, C.c_int]
        self.lib.rem2d_oracle_set_threads(self.h, int(threads))
        self.lib.rem2d_control_sine_outputs.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]

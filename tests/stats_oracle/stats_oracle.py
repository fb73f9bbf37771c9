"""Python handle on the CPU oracle with the episode statistics (tests/stats_oracle/librem2d_oracle_stats.so). TEST
INFRASTRUCTURE ONLY: the oracle of oracle/rem2d_oracle.c, unchanged, plus rem2d_set_stats / rem2d_read_stats
(include/rem2d_stats.h)."""
import ctypes as C
import os
import subprocess

from gym_rem2d_b200.capi import Engine

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "librem2d_oracle_stats.so")


def build():
    subprocess.check_call(["make", "-s", "-C", HERE])
    return LIB


class StatsOracleEngine(Engine):
    def __init__(self, threads=1, **overrides):
        super().__init__(lib_path=build(), **overrides)
        self.lib.rem2d_oracle_set_threads.argtypes = [C.c_void_p, C.c_int]
        self.lib.rem2d_oracle_set_threads(self.h, int(threads))

"""ctypes handle on the probe harness of single device-code functions (tests/probe/rem2d_probe.cu). TEST INFRASTRUCTURE ONLY.

Three builds of the same source: "emu" (g++ on the CPU through the emulation shim), "cuda" (nvcc -fmad=false, what the CUDA
library runs) and "fma" (nvcc -fmad=true, what Engine(precision="fast") runs). All arrays are float32 / int32, one row per case.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIBS = {"emu": "librem2d_probe_emu.so", "cuda": "librem2d_probe_cuda.so", "fma": "librem2d_probe_cuda_fma.so"}

_libs = {}


def build(kind="emu"):
    subprocess.check_call(["make", "-s", "-C", HERE, LIBS[kind]])
    return os.path.join(HERE, LIBS[kind])


def lib(kind="emu"):
    if kind not in _libs:
        L = C.CDLL(build(kind))
        p = C.c_void_p
        L.probe_rot_set.argtypes = [C.c_int, p, p, p]
        L.probe_contact_update.argtypes = [p, C.c_int, C.c_int] + [p] * 11
        L.probe_distance.argtypes = [C.c_int] + [p] * 12
        L.probe_toi.argtypes = [C.c_int] + [p] * 7
        for f in (L.probe_rot_set, L.probe_contact_update, L.probe_distance, L.probe_toi, L.probe_fmad):
            f.restype = C.c_int
        _libs[kind] = L
    return _libs[kind]


def _f(a, shape=None):
    a = np.ascontiguousarray(a, np.float32)
    return a if shape is None else a.reshape(shape)


def _i(a, shape=None):
    a = np.ascontiguousarray(a, np.int32)
    return a if shape is None else a.reshape(shape)


def _call(fn, *args):
    rc = fn(*[a.ctypes.data if isinstance(a, np.ndarray) else a for a in args])
    if rc != 0:
        raise RuntimeError("%s failed: %d" % (fn.__name__, rc))


def rot_set(a, kind="emu"):
    """(s, c) = rot_set(a) of every angle."""
    a = _f(a)
    s, c = np.empty_like(a), np.empty_like(a)
    _call(lib(kind).probe_rot_set, len(a), a, s, c)
    return s, c


def contact_update(edges, edge, circle, hx, hy, x, y, angle, old_i=None, old_imp=None, kind="emu"):
    """Sim::contact_update of one pool contact (body 0, edge[i] of the table `edges` [n_edges, 4]) per case.
    Returns dict: count, type, touching, ids [n, 2], normal, local_point, points [n, 2, 2], impulses [n, 4], q [n, 2] (s, c)."""
    edges = _f(edges, (-1, 4))
    n = len(edge)
    old_i = _i(np.zeros((n, 3)) if old_i is None else old_i, (n, 3))
    old_imp = _f(np.zeros((n, 4)) if old_imp is None else old_imp, (n, 4))
    oi, of = np.zeros((n, 5), np.int32), np.zeros((n, 14), np.float32)
    _call(lib(kind).probe_contact_update, edges, len(edges), n, _i(edge), _i(circle), _f(hx), _f(hy), _f(x), _f(y), _f(angle),
          old_i, old_imp, oi, of)
    return dict(count=oi[:, 0], type=oi[:, 1], touching=oi[:, 2], ids=oi[:, 3:5], normal=of[:, 0:2], local_point=of[:, 2:4],
                points=of[:, 4:8].reshape(n, 2, 2), impulses=of[:, 8:12], q=of[:, 12:14])


def distance(ev, circle, hx, hy, x, y, angle, cache=None, metric=None, kind="emu"):
    """Sim::gjk between edge ev[i] = (v1, v2) and the core of body 0 at (x, y, angle). cache: [n, 7] (count, ia[3], ib[3]),
    count 0 = cold start. Returns (distance, cache out, metric out)."""
    n = len(circle)
    cache = _i(np.zeros((n, 7)) if cache is None else cache, (n, 7))
    metric = _f(np.zeros(n) if metric is None else metric)
    d, co, mo = np.zeros(n, np.float32), np.zeros((n, 7), np.int32), np.zeros(n, np.float32)
    _call(lib(kind).probe_distance, n, _f(ev, (n, 4)), _i(circle), _f(hx), _f(hy), _f(x), _f(y), _f(angle), cache, metric, d, co, mo)
    return d, co, mo


def toi(ev, circle, hx, hy, sweep, kind="emu"):
    """Sim::time_of_impact of body 0 along sweep[i] = (c0.x, c0.y, a0, c.x, c.y, a, alpha0) against edge ev[i].
    Returns (touching, t)."""
    n = len(circle)
    touching, t = np.zeros(n, np.int32), np.zeros(n, np.float32)
    _call(lib(kind).probe_toi, n, _f(ev, (n, 4)), _i(circle), _f(hx), _f(hy), _f(sweep, (n, 7)), touching, t)
    return touching.astype(bool), t

"""The C-ABI library loads without a GPU and exports every symbol include/rem2d.h declares; the product
path refuses to run without its native library / a CUDA device (no CPU fallback)."""
import ctypes
import os
import re

import pytest

from gym_rem2d_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "rem2d.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(rem2d_[a-z0-9_]+)\s*\(", src)))


@pytest.mark.parametrize("lib", [capi.CUDA_LIB, capi.CUDA_LIB_FAST, os.path.join(ROOT, "oracle", "librem2d_oracle.so")])
def test_library_exports_every_declared_symbol(lib):
    if not os.path.exists(lib):
        import __graft_entry__ as g
        g.build()
    h = ctypes.CDLL(lib)
    syms = declared_symbols()
    assert len(syms) >= 18
    for s in syms:
        assert hasattr(h, s), "%s does not export %s" % (os.path.basename(lib), s)
    h.rem2d_backend.restype = ctypes.c_char_p
    assert h.rem2d_abi_version() == 1
    assert h.rem2d_backend() in (b"cuda-sm_100a", b"oracle-c")


def test_default_config_matches_reference_constants():
    lib = capi.load_library(capi.CUDA_LIB)
    cfg = capi.Config()
    lib.rem2d_default_config(ctypes.byref(cfg))
    assert abs(cfg.dt - 1 / 50) < 1e-9 and cfg.velocity_iterations == 180 and cfg.position_iterations == 60
    assert cfg.gravity_y == -10.0 and cfg.p_gain == 1.9 and cfg.wod_speed == 0.04
    assert cfg.evaluation_steps == 10000 and cfg.env_length == 100.0 and cfg.continuous == 1 and cfg.terminate == 1


def test_missing_library_fails_loudly(tmp_path):
    with pytest.raises(capi.Rem2dError, match="no CPU fallback"):
        capi.load_library(str(tmp_path / "nope.so"))


def test_no_gpu_means_error_not_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(capi.Rem2dError, match="no CUDA device|CUDA"):
        capi.Engine(device=0)


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "gym_rem2d_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert "import oracle" not in text and "from oracle" not in text and "librem2d_oracle" not in text, f


def test_documented_options_are_the_implemented_ones():
    """DESIGN.md's option list, the names rem2d_set_option of the CUDA library parses (read from its source) and the names the
    oracle's stub accepts are the same set; unknown names, and the names of removed execution strategies, are an error."""
    import ctypes
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    doc = open(os.path.join(root, "DESIGN.md")).read()
    block = doc[doc.index("Options (`rem2d_set_option`"):]
    block = block[:block.index("Defaults are")]
    documented = set(re.findall(r"`([a-z_0-9<>]+)`", block)) - {"rem2d_set_option"}
    src = open(os.path.join(root, "gym_rem2d_b200", "csrc", "rem2d_cuda.cu")).read()
    body = src[src.index("static bool set_option("):src.index("static void options_from_env(")]
    implemented = set(re.findall(r'n == "([a-z_0-9]+)"', body)) | {"class_gs_<k>"}
    assert documented == implemented, (documented ^ implemented)
    from oracle.oracle import OracleEngine
    e = OracleEngine()
    for name in sorted(implemented):
        e.set_option(name.replace("<k>", "3"), 1.0)
    removed = ("phased", "second_group_shift", "park_late_ticks", "park_lead", "priority_mode", "min_class", "small_weight",
               "wide_weight")
    for name in ("no_such_option",) + removed:
        assert name not in implemented, name
        with pytest.raises(Exception):
            e.set_option(name, 1.0)

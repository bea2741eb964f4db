"""CPU-only: the C-ABI library loads, exports every symbol include/sdrg.h declares, fails loudly
without a GPU, and its host-side design code lands on the reference's own coefficients."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT, golden_names, load_golden
from libsdr_b200 import _lib
from libsdr_b200.nodes import IQBaseBand, Config, ConfigError


def header_symbols():
    src = open(os.path.join(ROOT, "include", "sdrg.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(sdrg_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported_and_bound():
    lib = _lib.load()
    syms = header_symbols()
    assert len(syms) > 30
    for s in syms:
        assert hasattr(lib, s), "libsdrg.so does not export %s" % s
        assert s in _lib.SIGNATURES, "python binding lacks %s" % s
    assert lib.sdrg_abi_version() == 2


def _make(g):
    bb = IQBaseBand(str(g["scalar"]), float(g["Fc"]), float(g["Ff"]), float(g["width"]), int(g["order"]),
                    int(g["sub_sample_arg"]), float(g["oFs"]))
    if int(g["setcf"]):
        bb.setCenterFrequency(float(g["Fc"]))
        bb.setFilterFrequency(float(g["Ff"]))
    return bb


@pytest.mark.parametrize("name", golden_names("bb_"))
def test_host_design_matches_reference(name):
    g = load_golden(name)
    bb = _make(g)
    out = bb.design_only(sample_rate=float(g["Fs"]), buffer_size=int(g["buffer_size"]))
    inf = bb.info()
    assert inf.order == int(g["ref_order"])
    assert inf.sub_sample == int(g["ref_sub_sample"])
    assert inf.lut_inc == int(g["ref_lut_inc"])
    assert inf.negative_shift == int(g["ref_neg"])
    k, lut = bb.design()
    np.testing.assert_array_equal(k, g["ref_kernel"])
    np.testing.assert_array_equal(lut, g["ref_lut"])
    # published output config (baseband.hh:192-193)
    bs, ss = int(g["buffer_size"]), int(g["ref_sub_sample"])
    assert out.buffer_size == bs // ss + (1 if bs % ss else 0)
    assert out.sample_rate == float(int(g["Fs"]) // ss)
    assert out.type == {"s16": _lib.T_CS16, "s8": _lib.T_CS8}[str(g["scalar"])]


@pytest.mark.parametrize("name", golden_names("rbb_"))
def test_real_baseband_host_design_matches_reference(name):
    from libsdr_b200.nodes import BaseBand
    g = load_golden(name)
    bb = BaseBand(float(g["Fc"]), float(g["Ff"]), float(g["width"]), int(g["order"]), int(g["sub_sample"]))
    out = bb.design_only(sample_rate=float(g["Fs"]), buffer_size=int(g["buffer_size"]))
    inf = bb.info()
    assert inf.lut_inc == int(g["ref_lut_inc"]) and inf.negative_shift == int(g["ref_neg"])
    np.testing.assert_array_equal(bb.design()[0], g["ref_kernel"])
    bs, ss = int(g["buffer_size"]), int(g["sub_sample"])
    assert out.buffer_size == bs // ss + (1 if bs % ss else 0)
    assert out.sample_rate == float(g["Fs"]) / ss                 # a double here (baseband.hh:396-397)
    assert out.type == _lib.T_CS16
    with pytest.raises(ConfigError):                              # complex input is a type error (baseband.hh:363-369)
        bb.design_only(Config(_lib.T_CS16, 48e3, 1024, 1))


def test_config_error_on_type_mismatch_and_silent_on_incomplete():
    bb = IQBaseBand("s16", 100e3, 100e3, 12.5e3, 15, 1, 48000.0)
    with pytest.raises(ConfigError):
        bb.design_only(Config(_lib.T_CF32, 2.4e6, 4096, 1))
    # incomplete configs are ignored (baseband.hh:118)
    out = bb.design_only(Config(_lib.T_CS16, 0.0, 4096, 1))
    assert out.type == _lib.T_UNDEFINED
    out = bb.design_only(Config(_lib.T_UNDEFINED, 2.4e6, 4096, 1))
    assert out.type == _lib.T_UNDEFINED


def test_no_cpu_fallback():
    """Without a CUDA device the compute entry points must fail, not silently compute."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    bb = IQBaseBand("s16", 100e3, 100e3, 12.5e3, 15, 1, 48000.0)
    with pytest.raises(RuntimeError):
        bb.config(sample_rate=2.4e6, buffer_size=4096)
    with pytest.raises(RuntimeError):
        bb.process(np.zeros((16, 2), dtype=np.int16))


def test_product_never_touches_oracle():
    """No file of the product (package, headers) may reference the oracle."""
    bad = []
    for base in ("libsdr_b200", "include"):
        for dp, _, fs in os.walk(os.path.join(ROOT, base)):
            for f in fs:
                if f.endswith((".py", ".cu", ".cuh", ".cc", ".h", ".hh")):
                    txt = open(os.path.join(dp, f), errors="replace").read()
                    if re.search(r"oracle[/.]|sdr_oracle|liboracle|import oracle", txt):
                        bad.append(os.path.join(dp, f))
    assert not bad, bad


def test_shipped_library_has_no_result_changing_switches():
    """The default build must not honour any environment variable of its own: no SDRG_* name in the .so (the
    static CUDA runtime still reads its CUDA_* variables), the probe / ablation / TMA kernels are not linked,
    and float path 3 is refused."""
    import subprocess
    lib = _lib.load()
    assert lib.sdrg_build_has_experiments() == 0
    so = _lib.LIB_PATH
    names = subprocess.run(["strings", so], capture_output=True, text=True, check=True).stdout
    assert "SDRG_FOLD" not in names and "SDRG_FFT_R16" not in names
    assert "SDRG_" not in names.replace("SDRG_ERR", "").replace("SDRG_T_", "").replace("SDRG_EXPERIMENTS", "")
    syms = subprocess.run(["nm", "-C", so], capture_output=True, text=True, check=True).stdout
    assert "launch_fold_probe" not in syms and "launch_fold_tma" not in syms
    h = C.c_void_p()
    _lib.call("sdrg_iqbb_create", _lib.T_F32, 1e5, 1e5, 1e4, 16, 64, 0.0, C.byref(h))
    with pytest.raises(_lib.ConfigError):
        _lib.call("sdrg_iqbb_set_float_path", h, 3)
    lib.sdrg_iqbb_destroy(h)


def test_one_build_without_environment_switches():
    """The library is built one way only: no C/C++/CUDA source reads the environment, and nothing in the package or
    the header names a second (experiments) build."""
    offenders = []
    for base in ("libsdr_b200", "include"):
        for dp, dirs, fs in os.walk(os.path.join(ROOT, base)):
            dirs[:] = [d for d in dirs if d != "__pycache__"]
            for f in fs:
                path = os.path.join(dp, f)
                rel = os.path.relpath(path, ROOT)
                text = open(path, encoding="utf-8", errors="replace").read()
                native = f.endswith((".cu", ".cuh", ".cc", ".cpp", ".c", ".h", ".hh")) and \
                    (base == "include" or rel.startswith(os.path.join("libsdr_b200", "csrc")))
                if native and "getenv" in text:
                    offenders.append((rel, "getenv"))
                if "SDRG_EXPERIMENTS" in text:
                    offenders.append((rel, "SDRG_EXPERIMENTS"))
    assert not offenders, offenders

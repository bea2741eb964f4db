"""Pins the oracle against the REFERENCE ITSELF on random node parameters.  Complements the committed goldens
(tests/golden/*.npz) with configurations nobody hand-picked.  Every case checks its outputs against the
reference's recorded outputs on the same seeded input (tests/recorded.py); when oracle/_ref/ref_harness (the
unmodified libsdr classes compiled by oracle/Makefile) is built, it also runs the reference and compares
directly.  CPU only."""
import os
import subprocess

import numpy as np
import pytest

import recorded
from conftest import ROOT
from oracle import oracle as orc

HARNESS = os.path.join(ROOT, "oracle", "_ref", "ref_harness")
LIVE = os.path.exists(HARNESS)


def _params(g):
    Fs = float(g.choice([48e3, 1e6, 2.4e6, 20e6, 100e6]))
    order = int(g.integers(1, 41))
    ss = int(g.choice([1, 2, 3, 7, 8, 31, 32, 50, 64, 65, 125, 300]))
    Fc = float(g.choice([0.0, 1.0, -1.0]) * g.uniform(0, 0.45) * Fs)
    Ff = Fc if g.random() < 0.5 else float(g.uniform(-0.4, 0.4) * Fs)
    width = float(g.uniform(0.001, 0.4) * Fs)
    return Fs, Fc, Ff, width, order, ss


@pytest.mark.parametrize("seed", range(16))
@pytest.mark.parametrize("scalar", ["s16", "s8"])
def test_iqbaseband_and_demods_vs_live_reference(scalar, seed, tmp_path):
    g = np.random.default_rng(31000 + 100 * (scalar == "s8") + seed)
    Fs, Fc, Ff, width, order, ss = _params(g)
    oFs = 0.0 if seed % 2 else Fs / ss                  # both ways of choosing the sub-sampling (baseband.hh:156-160)
    setcf = seed % 3 == 0
    dt = np.int16 if scalar == "s16" else np.int8
    amp = np.iinfo(dt).max if seed % 4 == 0 else np.iinfo(dt).max // 8      # full scale: wrap regime
    n, bs = 12000, 4096
    x = g.integers(-amp, amp + 1, size=(n, 2)).astype(dt)
    sc = orc.S16 if scalar == "s16" else orc.S8
    o = orc.IQBaseBand(sc, Fc, Ff, width, order, ss, oFs)
    if setcf:
        o.set_center_frequency(Fc); o.set_filter_frequency(Ff)
    o.config(Fs, bs)
    ofm = orc.FMDemod(sc)
    bb, fm, am, usb, counts = [], [], [], [], []
    for k in range(0, n, bs):
        y = o.process(x[k:k + bs]); counts.append(y.shape[0])
        if y.shape[0]:
            bb.append(y); fm.append(ofm.process(y, inplace=True)); am.append(orc.amdemod(y, sc)); usb.append(orc.usbdemod(y, sc))
    out = {"counts": np.array(counts, dtype=np.uint32)}
    if bb:
        out.update(bb=np.concatenate(bb), fm=np.concatenate(fm), am=np.concatenate(am), usb=np.concatenate(usb))
    recorded.check("iqbb_%s_%d" % (scalar, seed), **out)
    if LIVE:
        inp = tmp_path / "x.bin"; x.tofile(inp)
        pre = str(tmp_path / "out")
        subprocess.run([HARNESS, "bb", scalar, str(inp), str(bs), repr(Fs), repr(Fc), repr(Ff), repr(width), str(order), str(ss),
                        repr(oFs), str(int(setcf)), pre], check=True)
        np.testing.assert_array_equal(out["counts"], np.fromfile(pre + ".counts", dtype=np.uint32))
        if bb:
            np.testing.assert_array_equal(out["bb"], np.fromfile(pre + ".bb", dtype=dt).reshape(-1, 2))
            np.testing.assert_array_equal(out["fm"], np.fromfile(pre + ".fm", dtype=np.int16))
            np.testing.assert_array_equal(out["am"], np.fromfile(pre + ".am", dtype=dt))
            np.testing.assert_array_equal(out["usb"], np.fromfile(pre + ".usb", dtype=dt))


@pytest.mark.parametrize("seed", range(12))
def test_real_baseband_vs_live_reference(seed, tmp_path):
    g = np.random.default_rng(32000 + seed)
    Fs, Fc, Ff, width, order, ss = _params(g)
    n, bs = 9000, 2048
    x = g.integers(-32768, 32768, size=n).astype(np.int16)
    o = orc.BaseBand(Fc, Ff, width, order, ss); o.config(Fs, bs)
    outs = [o.process(x[k:k + bs]) for k in range(0, n, bs)]
    counts, bb = np.array([y.shape[0] for y in outs], dtype=np.uint32), np.concatenate(outs)
    recorded.check("rbb_%d" % seed, counts=counts, bb=bb)
    if LIVE:
        inp = tmp_path / "x.bin"; x.tofile(inp)
        pre = str(tmp_path / "out")
        subprocess.run([HARNESS, "rbb", str(inp), str(bs), repr(Fs), repr(Fc), repr(Ff), repr(width), str(order), str(ss), pre], check=True)
        np.testing.assert_array_equal(counts, np.fromfile(pre + ".counts", dtype=np.uint32))
        np.testing.assert_array_equal(bb, np.fromfile(pre + ".bb", dtype=np.int16).reshape(-1, 2))


@pytest.mark.parametrize("seed", range(12))
def test_real_baseband_int8_vs_live_reference(seed, tmp_path):
    """BaseBand<int8_t>: 16-bit wraps in the FIR sum, the window sum and complex<int16_t>::operator/= ."""
    g = np.random.default_rng(36000 + seed)
    Fs, Fc, Ff, width, order, ss = _params(g)
    if (ss * ss) % 65536 == 0:
        ss += 1                                   # the reference divides by zero there
    n, bs = 9000, 2048
    amp = 127 if seed % 3 == 0 else 40
    x = g.integers(-amp, amp + 1, size=n).astype(np.int8)
    o = orc.BaseBand(Fc, Ff, width, order, ss, scalar=orc.S8); o.config(Fs, bs)
    outs = [o.process(x[k:k + bs]) for k in range(0, n, bs)]
    counts, bb = np.array([y.shape[0] for y in outs], dtype=np.uint32), np.concatenate(outs)
    recorded.check("rbb8_%d" % seed, counts=counts, bb=bb)
    if LIVE:
        inp = tmp_path / "x.bin"; x.tofile(inp)
        pre = str(tmp_path / "out")
        subprocess.run([HARNESS, "rbb8", str(inp), str(bs), repr(Fs), repr(Fc), repr(Ff), repr(width), str(order), str(ss), pre], check=True)
        np.testing.assert_array_equal(counts, np.fromfile(pre + ".counts", dtype=np.uint32))
        np.testing.assert_array_equal(bb, np.fromfile(pre + ".bb", dtype=np.int8).reshape(-1, 2))


@pytest.mark.parametrize("seed", range(8))
def test_ola_filter_vs_live_reference(seed, tmp_path):
    """FilterSink + FilterSource of the reference (with the double-precision FFT stand-in) on random bands."""
    g = np.random.default_rng(33000 + seed)
    block = int(g.choice([16, 64, 128, 512, 1024]))
    Fs = float(g.choice([1e6, 20e6]))
    f1, f2 = sorted(g.uniform(-0.45, 0.45, size=2) * Fs)
    nblk = 5
    x = (g.standard_normal(block * nblk) + 1j * g.standard_normal(block * nblk)).astype(np.complex64)
    f = orc.FilterOLA(block, float(f1), float(f2), Fs)
    taps, out = orc.filter_taps(block, float(f1), float(f2), Fs), f.process(x)
    recorded.check("ola_%d" % seed, taps=taps, kern=f.kern, out=out)
    if LIVE:
        inp = tmp_path / "x.bin"; x.tofile(inp)
        pre = str(tmp_path / "out")
        subprocess.run([HARNESS, "ola", str(inp), str(block), repr(Fs), repr(float(f1)), repr(float(f2)), pre], check=True)
        np.testing.assert_array_equal(taps, np.fromfile(pre + ".taps", dtype=np.complex64))
        np.testing.assert_array_equal(f.kern, np.fromfile(pre + ".kern", dtype=np.complex64))
        np.testing.assert_array_equal(out, np.fromfile(pre + ".out", dtype=np.complex64))


@pytest.mark.parametrize("fmt,dt", [("cu8", np.uint8), ("cs8", np.int8)])
def test_autocast_vs_live_reference(fmt, dt, tmp_path):
    g = np.random.default_rng(34000 + (fmt == "cs8"))
    x = g.integers(np.iinfo(dt).min, np.iinfo(dt).max + 1, size=(7001, 2)).astype(dt)
    out = orc.autocast_cs16(x)
    recorded.check("cast_" + fmt, cs16=out)
    if LIVE:
        inp = tmp_path / "x.bin"; x.tofile(inp)
        pre = str(tmp_path / "out")
        subprocess.run([HARNESS, "cast", fmt, str(inp), "1000", pre], check=True)
        np.testing.assert_array_equal(out, np.fromfile(pre + ".cs16", dtype=np.int16).reshape(-1, 2))


@pytest.mark.parametrize("Fs", [8000.0, 22050.0, 48000.0, 96000.0, 250e3])
def test_fmdeemph_vs_live_reference(Fs, tmp_path):
    g = np.random.default_rng(int(Fs))
    x = g.integers(-32768, 32768, size=5003).astype(np.int16)
    d = orc.FMDeemph(Fs)
    out = np.concatenate([d.process(x[o:o + 777]) for o in range(0, x.shape[0], 777)])
    recorded.check("deemph_%d" % int(Fs), out=out)
    if LIVE:
        inp = tmp_path / "x.bin"; x.tofile(inp)
        pre = str(tmp_path / "out")
        subprocess.run([HARNESS, "deemph", str(inp), "777", repr(Fs), pre], check=True)
        np.testing.assert_array_equal(out, np.fromfile(pre + ".out", dtype=np.int16))


@pytest.mark.parametrize("seed", range(16))
@pytest.mark.parametrize("scalar", ["s16", "s8"])
def test_product_host_design_vs_live_reference(scalar, seed, tmp_path):
    """The product's config-time design (csrc/design.cc through sdrg_iqbb_design, no GPU needed) reproduces the
    reference's own taps, LUT, increment and sub-sampling on random parameters."""
    from libsdr_b200.nodes import IQBaseBand
    g = np.random.default_rng(35000 + 100 * (scalar == "s8") + seed)
    Fs, Fc, Ff, width, order, ss = _params(g)
    oFs = 0.0 if seed % 2 else Fs / ss
    dt = np.int16 if scalar == "s16" else np.int8
    bb = IQBaseBand(scalar, Fc, Ff, width, order, ss, oFs)
    bb.design_only(sample_rate=Fs, buffer_size=64)
    inf = bb.info()
    params = np.array([inf.order, inf.sub_sample, inf.lut_inc, inf.negative_shift], dtype=np.int64)
    k, lut = bb.design()
    recorded.check("design_%s_%d" % (scalar, seed), params=params, kernel=k, lut=lut)
    if LIVE:
        x = np.zeros((64, 2), dtype=dt)
        inp = tmp_path / "x.bin"; x.tofile(inp)
        pre = str(tmp_path / "out")
        subprocess.run([HARNESS, "bb", scalar, str(inp), "64", repr(Fs), repr(Fc), repr(Ff), repr(width), str(order), str(ss),
                        repr(oFs), "0", pre], check=True)
        raw = np.fromfile(pre + ".params", dtype=np.uint8)
        hdr = raw[:32].view(np.int64); L = int(hdr[0])
        ref_kernel = raw[32:32 + 8 * L].view(np.int32).reshape(L, 2)
        ref_lut = raw[32 + 8 * L:32 + 8 * L + 8 * 128].view(np.int32).reshape(128, 2)
        assert tuple(int(v) for v in params) == (L, int(hdr[1]), int(hdr[2]), int(hdr[3]))
        np.testing.assert_array_equal(k, ref_kernel)
        np.testing.assert_array_equal(lut, ref_lut)

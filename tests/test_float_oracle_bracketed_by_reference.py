"""Brackets the FLOAT oracle by the reference.

IQBaseBand<float> does not compile and FMDemod<float> does not link in the reference, so the float path's
semantics are defined by oracle/sdr_oracle.c ("parity unpinned").  This test turns "defined" into "bounded by
the reference": the same int16-valued samples go through the reference's IQBaseBand<int16_t> (+ FMDemod) and
through the float oracle, and the two must agree to within the integer path's own truncation errors, stage by
stage.  The integer side is the int16 oracle, pinned bit-exact to the reference by test_oracle_vs_golden.py and
test_oracle_vs_live_reference.py; its outputs here are checked against recorded digests (tests/recorded.py) and,
when oracle/_ref/ref_harness (the reference's build) is present, against the reference itself:

  taps     k_i = trunc(2^14 a_i)        float uses a_i           |dk| < 2^-14 per component  (baseband.hh:260)
  FIR      y = (sum k x) >> 14          floor per component      <= 1
  LUT      l_j = trunc(2^16 e^{-i..})   float uses e^{-i..}      |dl| < 2^-16 per component  (freqshift.hh:31-35)
  NCO      z = (l y) >> 16              floor                    <= 1
  boxcar   out = trunc(S ss / ss^2)     float: S / ss            <= 1                         (baseband.hh:212-217)

With A = max |component of x| the per-component bound used below is computed from the ACTUAL tap / LUT
truncation errors of the configuration (not the worst case 2^-14 per tap):
  e_fir = A * sum_i(|dkr_i| + |dki_i|) + 1
  e_nco = (|l| sum) e_fir + max_j(|dlr_j| + |dli_j|) * Ymax + 1,  Ymax = A * sum_i(|ar_i| + |ai_i|)
  |out_ref - out_float| <= e_nco + 1            (e_fir + 1 when the mixer is bypassed, inc == 0)
FM (math.hh:31-40): phi = fast_atan2/2 in units of pi/16384 per LSB; for samples with |re|,|im| well above the
base-band bound the rational approximation has slope <= 8192 / (|re| + |im|) per unit of input error.
CPU only."""
import os
import subprocess

import numpy as np
import pytest

import recorded
from conftest import ROOT
from libsdr_b200 import synth
from oracle import oracle as orc

HARNESS = os.path.join(ROOT, "oracle", "_ref", "ref_harness")

#        name            Fs      Fc       Ff       width   order  ss  oFs      amplitude
CASES = [("c1",          2.4e6,  100e3,   100e3,   12.5e3, 15,    1,  48000.0, 8192),
         ("neg_shift",   2.4e6,  -100e3,  -100e3,  12.5e3, 21,    1,  48000.0, 12000),
         ("inc0",        2.4e6,  0.0,     0.0,     25e3,   16,    50, 0.0,     8192),     # mixer bypassed (freqshift.hh:61)
         ("c2_shape",    20e6,   100e3,   100e3,   12.5e3, 64,    1,  48000.0, 6000),     # the headline float geometry (64 taps, ss 416)
         ("ss7_frac",    1e6,    33333.3, 30000.0, 40e3,   33,    7,  0.0,     3000),
         ("wide_Ff_off", 2.4e6,  300e3,   250e3,   100e3,  40,    25, 0.0,     10000),
         ("ss1",         2.4e6,  -450e3,  -450e3,  200e3,  9,     1,  0.0,     5000)]


def _signal(n, Fs, Fc, amp, seed):
    # a carrier near the channel centre with FM-like phase wobble, an adjacent interferer, noise
    comps = [(amp * 0.6, Fc + 0.002 * Fs * 0.5, 0.3), (amp * 0.25, Fc - 0.0015 * Fs, 1.1), (amp * 0.1, Fc + 0.12 * Fs, 2.0)]
    return synth.iq_int(n, Fs, comps, max(1, amp // 100), seed, np.int16)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_float_oracle_within_truncation_bound_of_reference_int16(case, tmp_path):
    name, Fs, Fc, Ff, width, order, ss, oFs, amp = case
    n, bs = 60000, 20000
    x = _signal(n, Fs, Fc, amp, 77 + order)
    A = float(np.abs(x.astype(np.int64)).max())

    # the integer chain, buffer by buffer
    oi = orc.IQBaseBand(orc.S16, Fc, Ff, width, order, ss, oFs); oi.config(Fs, bs)
    oifm = orc.FMDemod(orc.S16)
    i_bb, i_fm, counts = [], [], []
    for k in range(0, n, bs):
        y = oi.process(x[k:k + bs]); counts.append(y.shape[0])
        if y.shape[0]:
            i_bb.append(y); i_fm.append(oifm.process(y, inplace=True))
    counts, i_bb, i_fm = np.array(counts, dtype=np.uint32), np.concatenate(i_bb), np.concatenate(i_fm)
    recorded.check("bracket_" + name, counts=counts, bb=i_bb, fm=i_fm)
    if os.path.exists(HARNESS):
        inp = tmp_path / "x.bin"; x.tofile(inp)
        pre = str(tmp_path / "out")
        subprocess.run([HARNESS, "bb", "s16", str(inp), str(bs), repr(Fs), repr(Fc), repr(Ff), repr(width), str(order), str(ss),
                        repr(oFs), "0", pre], check=True)
        np.testing.assert_array_equal(counts, np.fromfile(pre + ".counts", dtype=np.uint32))
        np.testing.assert_array_equal(i_bb, np.fromfile(pre + ".bb", dtype=np.int16).reshape(-1, 2))
        np.testing.assert_array_equal(i_fm, np.fromfile(pre + ".fm", dtype=np.int16))
    ref_bb, ref_fm = i_bb.astype(np.float64), i_fm.astype(np.float64)

    # the float oracle on the same sample VALUES
    of = orc.IQBaseBand(orc.F32, Fc, Ff, width, order, ss, oFs); of.config(Fs, bs)
    ofm = orc.FMDemod(orc.F32)
    f_bb, f_fm, first, f_counts = [], [], [], []
    off = 0
    for k in range(0, n, bs):
        y = of.process(x[k:k + bs].astype(np.float32))
        f_counts.append(y.shape[0])
        if y.shape[0]:
            f_bb.append(y.astype(np.float64)); f_fm.append(ofm.process(y, inplace=True).astype(np.float64)); first.append(off)
        off += y.shape[0]
    f_bb, f_fm = np.concatenate(f_bb), np.concatenate(f_fm)
    assert [int(c) for c in counts] == f_counts                  # same window grid, buffer by buffer
    assert f_bb.shape == ref_bb.shape and ref_bb.shape[0] > 100

    # the bound, from the configuration's own truncation errors
    a = of.kernel_f64()                                          # alpha_i / norm, double
    k = oi.kernel_i32().astype(np.float64) / 16384.0
    dk = np.abs(a.real - k[:, 0]) + np.abs(a.imag - k[:, 1])
    assert np.all(np.abs(a.real - k[:, 0]) < 2.0 ** -14) and np.all(np.abs(a.imag - k[:, 1]) < 2.0 ** -14)     # same taps up to truncation
    e_fir = A * float(dk.sum()) + 1.0
    if oi.lut_inc == 0:
        bound = e_fir + 1.0
    else:
        lut = oi.lut_i32().astype(np.float64) / 65536.0
        j = np.arange(128)
        ex = np.exp(-2j * np.pi * j / 128)
        dl = np.abs(ex.real - lut[:, 0]) + np.abs(ex.imag - lut[:, 1])
        assert np.all(np.abs(ex.real - lut[:, 0]) < 2.0 ** -16 + 1e-12) and np.all(np.abs(ex.imag - lut[:, 1]) < 2.0 ** -16 + 1e-12)
        ymax = A * float((np.abs(a.real) + np.abs(a.imag)).sum())
        lsum = float((np.abs(lut[:, 0]) + np.abs(lut[:, 1])).max())
        bound = lsum * e_fir + float(dl.max()) * ymax + 1.0 + 1.0
    d = np.abs(ref_bb - f_bb)
    assert d.max() <= bound, (name, d.max(), bound)
    # ... and the bound is tight enough to mean something: a small fraction of the signal
    rms = np.sqrt(np.mean(ref_bb ** 2))
    assert bound < 0.02 * A and np.sqrt(np.mean(d ** 2)) < 0.01 * rms, (name, bound, A, rms)

    # FM on non-degenerate samples: both components far from the sign/quadrant decisions of fast_atan2
    scale = 16384.0 / np.pi                                      # int16 LSB per radian of the float definition
    re, im = np.abs(ref_bb[:, 0]), np.abs(ref_bb[:, 1])
    ok = (re > 8 * bound) & (im > 8 * bound)
    okp = ok & np.roll(ok, 1)                                    # out[i] = phi[i-1] - phi[i]: both samples must qualify
    okp[first] = False                                           # element 0 of every buffer is not FM (demod.hh:245)
    okp[0] = False
    assert okp.sum() > 50, (name, okp.sum())
    mag = re + im
    slope = 8192.0 * bound / mag + 1.0                           # per-sample phi error, int16 LSB (|d ang| <= 8192 e / (|a|+|b|), /2, trunc)
    tol = slope + np.roll(slope, 1) + 1.0
    dfm = np.abs(ref_fm - f_fm * scale)
    dfm = np.minimum(dfm, np.abs(dfm - 32768.0))                 # int16 wrap of (last - phi) at +-pi
    assert np.all(dfm[okp] <= tol[okp]), (name, float((dfm[okp] - tol[okp]).max()))
    if os.environ.get("SDRG_TEST_VERBOSE"):
        print("%-12s bb: max|d| %.2f <= bound %.2f (A %.0f, rms %.0f, rms d %.2f); fm: %d samples, max|d| %.1f LSB, max tol %.1f"
              % (name, d.max(), bound, A, rms, np.sqrt(np.mean(d ** 2)), okp.sum(), dfm[okp].max(), tol[okp].max()))

"""GPU parity of the float channel bank, ChannelBank("f32") and ShardedChannelBank("f32").

Channel c must equal an oracle IQBaseBand<float>(Fc[c], Ff[c], width, order, ss, oFs) fed the same buffers and
followed by FMDemod / AMDemod / USBDemod<float> connected out of place, to 1e-5 relative RMS, checked per
channel and per output kind (a whole-array RMS over thousands of channels would hide one wrong channel).
Every checked channel carries a carrier that its NCO moves into the pass band, so that its relative error is
well conditioned.  FM outputs are pre-filled with NaN: element 0 of every buffer must stay NaN, no other
element may be NaN.

Kernels and where their edge logic acts (bank_kernels.cu):
  bank_fold_f32_kernel  one launch per call.  32 channels per CTA (counts 1, 31, 33, 37 leave the last group
                        partly empty), 2048 samples per warp staged 256 at a time (one-sample calls, calls shorter
                        than a window and lengths that are no multiple of 256 or 2048 cut chunks, warp spans
                        and windows anywhere), window tails
                        computed from the taps at every window end (orders 1 ... 256; order 256 at ss 256 makes
                        every sample of a window a tail sample and reaches into the history).  There is no
                        fold / direct selection: the fold is the only path (DESIGN §4.7b).
  bank_finalize_kernel<SDRG_T_F32>  one launch per requested demodulator, or one for the base band alone.
Every call asserts this launch count through sdrg_kernel_launch_count.  Window sums are float atomics, so no
case assumes bitwise repeatability.
"""
import numpy as np
import pytest

from conftest import rel_rms
from libsdr_b200 import _lib, synth
from libsdr_b200.nodes import (DEMOD_FM, ChannelBank, ConfigError, IQBaseBand, RxChain, ShardedChannelBank, T_CS16,
                               Config)
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

TOL = 1e-5
ALL = ("bb", "fm", "am", "usb")


def expected_launches(want):
    return 1 + max(1, sum(k in want for k in ("fm", "am", "usb")))


def nan_outputs(bank, n_out, want, stride=None, device=None):
    stride = max(n_out, 1) if stride is None else stride
    shapes = {"bb": (bank.channels, stride, 2), "fm": (bank.channels, stride), "am": (bank.channels, stride),
              "usb": (bank.channels, stride)}
    if device is None:
        return {k: np.full(shapes[k], np.nan, dtype=np.float32) for k in want}
    import torch
    return {k: torch.full(shapes[k], float("nan"), dtype=torch.float32, device=device) for k in want}


def run_bank(bank, x, calls, want=ALL, device=None, stride_pad=0):
    """calls: [(start, end, buffer_size)].  Returns ({kind: (C, n) float arrays}, fm buffer-first indices)."""
    outs = {k: [] for k in want}
    first, off = [], 0
    for s, e, bs in calls:
        n_out = bank.outputs_for(e - s)
        res = nan_outputs(bank, n_out, want, max(n_out, 1) + stride_pad, device)
        xs = x[s:e]
        n0 = _lib.kernel_launch_count()
        r = bank.process(xs, bs, want=want, out=res)
        assert _lib.kernel_launch_count() - n0 == expected_launches(want)
        for k in want:
            full = res[k].cpu().numpy() if device is not None else res[k]
            got = full[:, :n_out]
            assert r[k].shape[1] == n_out
            if stride_pad:
                assert np.all(np.isnan(full[:, n_out:])), "gap columns written (%s)" % k
            outs[k].append(got)
        for b in range(s, e, bs):       # outputs completed by each buffer of the call
            m = bank_outputs_between(bank, s, b, b + bs)
            if m:
                first.append(off)
            off += m
    return {k: np.concatenate(v, axis=1) for k, v in outs.items()}, np.array(first, dtype=np.int64)


def bank_outputs_between(bank, call_start, lo, hi):
    """outputs completed by samples [lo, hi) (global), from the window grid: window 0 holds ss+1 samples"""
    ss = bank.ss

    def done(c):
        return (c - 1) // ss if c else 0
    return done(hi) - done(lo)


def oracle_channel(Fc, Ff, width, order, ss, oFs, Fs, x, calls):
    o = orc.IQBaseBand(orc.F32, Fc, Ff, width, order, ss, oFs)
    o.config(Fs, calls[0][2])
    fm = orc.FMDemod(orc.F32)
    bb, f, first, off = [], [], [], 0
    for s, e, bs in calls:
        for b in range(s, e, bs):
            y = o.process(x[b:b + bs])
            bb.append(y)
            if y.shape[0]:
                f.append(fm.process(y, inplace=False)); first.append(off)
            off += y.shape[0]
    bb = np.concatenate(bb)
    f = np.concatenate(f) if f else np.zeros(0, np.float32)
    return dict(bb=bb, fm=f, am=orc.amdemod(bb, orc.F32), usb=orc.usbdemod(bb, orc.F32)), np.array(first, dtype=np.int64)


def cplx(a):
    return a.astype(np.float64).view(np.complex128).reshape(-1)


def check_channel(got, first, ref, ref_first, c, want=ALL):
    np.testing.assert_array_equal(first, ref_first)
    for k in want:
        g, o = got[k][c], ref[k]
        assert g.shape == o.shape, (k, c, g.shape, o.shape)
        if k == "fm":
            mask = np.ones(o.shape[0], dtype=bool); mask[ref_first] = False
            assert np.all(np.isnan(g[~mask])), "fm ch %d: element 0 of a buffer was written" % c
            assert not np.any(np.isnan(g[mask])), "fm ch %d: NaN left" % c
            g, o = g[mask], o[mask]
        else:
            assert not np.any(np.isnan(g)), "%s ch %d: NaN left" % (k, c)
        if k == "bb":
            g, o = cplx(g), cplx(o)
        if o.shape[0]:
            e = rel_rms(g, o)
            assert e < TOL, "%s ch %d: rel rms %.3g" % (k, c, e)


def make_bank(cls, Fc, Ff, width, order, ss, oFs, Fs, bs, **kw):
    bank = cls("f32", Fc, Ff, width, order, ss, oFs, **kw)
    bank.config(sample_rate=Fs, buffer_size=bs)
    bank.ss = max(1, int(Fs // oFs)) if oFs > 0 else ss
    return bank


def bank_vs_oracle(Fc, Ff, width, order, ss, oFs, Fs, x, calls, channels=None, device=None, want=ALL, stride_pad=0):
    bank = make_bank(ChannelBank, Fc, Ff, width, order, ss, oFs, Fs, calls[0][2])
    xin = x
    if device is not None:
        import torch
        xin = torch.from_numpy(x).to(device)
    got, first = run_bank(bank, xin, calls, want, device, stride_pad)
    for c in (range(len(Fc)) if channels is None else channels):
        ref, ref_first = oracle_channel(Fc[c], Fc[c] if Ff is None else Ff[c], width, order, ss, oFs, Fs, x, calls)
        check_channel(got, first, ref, ref_first, c, want)
    return bank, got, first


def carriers_for(Fc, Fs, delta):
    """one tone per channel that its NCO moves to `delta` Hz (|Fc| = Fs is no shift at all)"""
    f = [((fc if abs(fc) < Fs else 0.0) + delta) for fc in Fc]
    return [(0.4 / np.sqrt(len(f)), fk, 0.37 * k) for k, fk in enumerate(f)]


# ---- 1. mixed shifts, all four outputs ---------------------------------------------------------------------

def test_mixed_shifts_three_calls():
    Fs, bs = 2.4e6, 16384
    Fc = np.array([100e3, -100e3, 0.0, 333e3, -777.5e3, 1.19e6, 50.25e3, -2.4e6])
    Ff = np.array([100e3, -100e3, 0.0, 300e3, -700e3, 1.0e6, 50e3, 0.0])
    x = synth.iq_f32(6 * bs, Fs, carriers_for(Fc, Fs, 1.1e3), 0.01, 21)
    bank_vs_oracle(Fc, Ff, 25e3, 21, 300, 0.0, Fs, x, [(0, 2 * bs, bs), (2 * bs, 3 * bs, bs), (3 * bs, 6 * bs, bs)])


# ---- 2. ragged calls at ss 2083 -------------------------------------------------------------------------------

def test_ragged_calls_ss2083():
    Fs = 100e6
    Fc = (np.arange(6) - 3) * (Fs / 256)
    x = synth.iq_f32(200000, Fs, carriers_for(Fc, Fs, 2e3), 0.01, 22)
    cuts = [0, 1, 2083, 2084, 50000, 123457, 200000]
    calls = [(s, e, e - s) for s, e in zip(cuts[:-1], cuts[1:])]
    bank, _, _ = bank_vs_oracle(Fc, None, 25e3, 15, 1, 48000.0, Fs, x, calls)
    assert bank.ss == 2083


# ---- 3. C4 geometry in float: 256 channels, device tensors ----------------------------------------------------

def c_input(cfg, n, spot):
    carriers = sorted({(k + d) % cfg["channels"] for k in spot for d in (-1, 0, 1)})
    return synth.bank_input(n, cfg, carriers=carriers).astype(np.float32) / 64.0


def test_c4_geometry_256_channels():
    cfg = synth.C4
    Fs, bs = cfg["Fs"], 1 << 18
    spot = (0, 1, 127, 128, 129, 255)
    Fc = synth.bank_frequencies(cfg["channels"], Fs)
    x = c_input(cfg, 2 * bs, spot)
    bank, _, _ = bank_vs_oracle(Fc, None, cfg["width"], cfg["order"], cfg["sub_sample"], cfg["oFs"], Fs, x,
                                [(0, 2 * bs, bs)], channels=spot, device="cuda")
    for c in spot:
        inf, k = bank.channel_info(c)
        node = IQBaseBand("f32", Fc[c], Fc[c], cfg["width"], cfg["order"], cfg["sub_sample"], cfg["oFs"])
        node.config(sample_rate=Fs, buffer_size=bs)
        nk, _ = node.design()
        assert k.dtype == np.float32
        np.testing.assert_array_equal(k, nk)
        assert inf.lut_inc == node.info().lut_inc and inf.sub_sample == 2083
    assert bank.channel_info(128)[0].lut_inc == 0


# ---- 4. C5 geometry in float: 2048 channels ---------------------------------------------------------------------

C5_SPOT = (0, 1, 1023, 1024, 1025, 2047, 389, 1707)


def test_c5_geometry_2048_channels():
    cfg = synth.C5
    Fs, bs = cfg["Fs"], 1 << 18
    Fc = synth.bank_frequencies(cfg["channels"], Fs)
    x = c_input(cfg, 2 * bs, C5_SPOT)
    bank_vs_oracle(Fc, None, cfg["width"], cfg["order"], cfg["sub_sample"], cfg["oFs"], Fs, x, [(0, 2 * bs, bs)],
                   channels=C5_SPOT, device="cuda", want=("fm", "am"))


# ---- kernel edges: orders, channel counts, sample counts ---------------------------------------------------------

ORDER_CASES = [(1, 300), (2, 300), (15, 300), (16, 256), (32, 300), (33, 257), (64, 300), (128, 300), (256, 300), (256, 256)]


@pytest.mark.parametrize("order,ss", ORDER_CASES, ids=["L%d-ss%d" % c for c in ORDER_CASES])
def test_orders(order, ss):
    """calls of 1 sample, shorter than a window, and not multiples of the 256-sample chunk or 2048-sample warp
    span; at order 256 and ss 256 every sample of a window is a tail sample"""
    Fs = 2.4e6
    Fc = np.array([150e3, -420e3, 0.0, 37.5e3, -1.1e6])
    x = synth.iq_f32(60001, Fs, carriers_for(Fc, Fs, 1.3e3), 0.01, 23)
    cuts = [0, 1, 2, ss - 1, ss + 2, 2049, 16385 + ss, 40000, 60001]
    calls = [(s, e, e - s) for s, e in zip(cuts[:-1], cuts[1:])]
    bank_vs_oracle(Fc, None, 80e3, order, ss, 0.0, Fs, x, calls)


@pytest.mark.parametrize("channels", [1, 31, 33, 37])
def test_channel_counts(channels):
    Fs = 2.4e6
    Fc = np.round(np.linspace(-1.15e6, 1.15e6, channels) / 100.0) * 100.0 if channels > 1 else np.array([-211e3])
    x = synth.iq_f32(3 * 20000 + 777, Fs, carriers_for(Fc, Fs, 1.5e3), 0.005, 24)
    calls = [(0, 40000, 20000), (40000, 40777, 777), (40777, 60777, 20000)]
    bank_vs_oracle(Fc, None, 30e3, 17, 320, 0.0, Fs, x, calls, device="cuda")


def test_short_calls_and_one_sample():
    """single-sample calls, a call shorter than a window, a call that ends exactly at a window end"""
    Fs, ss = 2.4e6, 400
    Fc = np.array([200e3, -65e3, 0.0])
    x = synth.iq_f32(5000, Fs, carriers_for(Fc, Fs, 1e3), 0.01, 25)
    cuts = [0, 1, 2, 3, 250, 401, 801, 802, 2100, 5000]
    bank_vs_oracle(Fc, None, 40e3, 33, ss, 0.0, Fs, x, [(s, e, e - s) for s, e in zip(cuts[:-1], cuts[1:])])


def test_base_band_only_and_single_demodulator():
    """want subsets: one finalize launch for the base band alone, one per demodulator otherwise"""
    Fs, bs = 2.4e6, 9000
    Fc = np.array([120e3, -333e3])
    x = synth.iq_f32(3 * bs, Fs, carriers_for(Fc, Fs, 900.0), 0.01, 26)
    for want in (("bb",), ("usb",), ("bb", "am")):
        bank_vs_oracle(Fc, None, 25e3, 15, 300, 0.0, Fs, x, [(0, 3 * bs, bs)], want=want)


def test_out_stride_gap_stays_nan():
    Fs, bs = 2.4e6, 12000
    Fc = np.array([100e3, -250e3, 0.0, 600e3])
    x = synth.iq_f32(2 * bs, Fs, carriers_for(Fc, Fs, 1e3), 0.01, 27)
    bank_vs_oracle(Fc, None, 25e3, 15, 300, 0.0, Fs, x, [(0, bs, bs), (bs, 2 * bs, bs)], device="cuda", stride_pad=13)


# ---- cross-check against separate float nodes (no oracle) ---------------------------------------------------------

def test_bank_equals_separate_float_chains():
    import torch
    Fs, bs = 100e6, 1 << 16
    C = 12
    Fc = (np.arange(C) - C // 2) * (Fs / 64) + 1234.0
    x = synth.iq_f32(4 * bs, Fs, carriers_for(Fc, Fs, 2.5e3), 0.01, 28)
    xd = torch.from_numpy(x).cuda()
    bank = make_bank(ChannelBank, Fc, None, 25e3, 15, 1, 48000.0, Fs, bs)
    got, first = run_bank(bank, xd, [(0, 4 * bs, bs)], ("bb", "fm"), "cuda")
    for c in range(C):
        node = IQBaseBand("f32", Fc[c], Fc[c], 25e3, 15, 1, 48000.0)
        node.config(sample_rate=Fs, buffer_size=bs)
        yb, ya, counts = RxChain(node, DEMOD_FM).process(xd, bs)
        torch.cuda.synchronize()
        yb, ya = yb.cpu().numpy(), ya.cpu().numpy()
        nfirst = np.concatenate([[0], np.cumsum(counts)[:-1]])[counts > 0]
        np.testing.assert_array_equal(first, nfirst)
        assert rel_rms(cplx(got["bb"][c]), cplx(yb)) < TOL, c
        mask = np.ones(ya.shape[0], dtype=bool); mask[nfirst] = False
        assert rel_rms(got["fm"][c][mask], ya[mask]) < TOL, c


# ---- sharded bank ---------------------------------------------------------------------------------------------------

def sharded_devices():
    import torch
    devs = [[0, 0, 0]]
    if torch.cuda.device_count() > 1:
        devs.append(list(range(torch.cuda.device_count())))
    return devs


@pytest.mark.parametrize("pointers", ["device", "host"])
def test_sharded_float_bank(pointers):
    import torch
    Fs, bs = 2.4e6, 15000
    Fc = np.round(np.linspace(-1.1e6, 1.1e6, 40) / 100.0) * 100.0
    x = synth.iq_f32(4 * bs, Fs, carriers_for(Fc, Fs, 1.2e3), 0.005, 29)
    calls = [(0, bs, bs), (bs, 3 * bs, bs), (3 * bs, 4 * bs, bs)]
    device = "cuda" if pointers == "device" else None
    xin = torch.from_numpy(x).cuda() if device else x
    single = make_bank(ChannelBank, Fc, None, 25e3, 15, 300, 0.0, Fs, bs)
    ref, ref_first = run_bank(single, xin, calls, ALL, device)
    for devs in sharded_devices():
        sb = make_bank(ShardedChannelBank, Fc, None, 25e3, 15, 300, 0.0, Fs, bs, devices=devs)
        outs = {k: [] for k in ALL}
        for s, e, b in calls:
            n_out = sb.outputs_for(e - s)
            res = nan_outputs(sb, n_out, ALL, None, device)
            sb.process(xin[s:e], b, want=ALL, out=res)
            for k in ALL:
                outs[k].append(res[k].cpu().numpy() if device else res[k])
        got = {k: np.concatenate(v, axis=1) for k, v in outs.items()}
        for c in range(len(Fc)):
            mask = np.ones(got["fm"].shape[1], dtype=bool); mask[ref_first] = False
            assert np.all(np.isnan(got["fm"][c][~mask]))
            for k in ALL:
                g, o = got[k][c], ref[k][c]
                if k == "fm":
                    g, o = g[mask], o[mask]
                if k == "bb":
                    g, o = cplx(g), cplx(o)
                assert not np.any(np.isnan(g))
                assert rel_rms(g, o) < TOL, (devs, k, c)
        # and both against the oracle on two channels
        for c in (3, 31):
            r, rf = oracle_channel(Fc[c], Fc[c], 25e3, 15, 300, 0.0, Fs, x, calls)
            check_channel(got, ref_first, r, rf, c)


# ---- errors -----------------------------------------------------------------------------------------------------------

def test_errors():
    import torch
    bank = ChannelBank("f32", np.array([1e5]), None, 25e3, 15, 255, 0.0)
    with pytest.raises(ConfigError, match="IQBaseBand"):
        bank.config(sample_rate=2.4e6, buffer_size=4096)
    bank = ChannelBank("f32", np.array([1e5]), None, 25e3, 15, 300, 0.0)
    with pytest.raises(ConfigError, match="complex float"):
        bank.config(Config(T_CS16, 2.4e6, 4096, 1))
    with pytest.raises(RuntimeError, match="order"):
        ChannelBank("f32", np.array([1e5]), None, 25e3, 257, 300, 0.0)
    bank.config(sample_rate=2.4e6, buffer_size=4096)
    x = torch.zeros((4096, 2), dtype=torch.float32, device="cuda")
    n_out = bank.outputs_for(4096)
    short = {"bb": torch.zeros((1, n_out - 1, 2), dtype=torch.float32, device="cuda")}
    with pytest.raises(RuntimeError, match="out_stride"):
        bank.process(x, 4096, want=("bb",), out=short)

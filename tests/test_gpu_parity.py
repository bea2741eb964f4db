"""GPU parity tests: the CUDA path (through the C ABI, libsdr_b200/libsdrg.so) against
 (1) the golden vectors produced by the reference itself, and
 (2) the oracle on seeded inputs at sizes it finishes in seconds, and
 (3) size-independent properties at BASELINE.json's full sizes.
Integer paths: bit-exact.  Float paths: <= 1e-5 relative RMS (north_star's tolerance)."""
import numpy as np
import pytest

from conftest import golden_names, load_golden, rel_rms
from libsdr_b200 import _lib, synth
from libsdr_b200.nodes import (IQBaseBand, FMDemod, AMDemod, USBDemod, RxChain, Config, ConfigError,
                               DEMOD_FM, DEMOD_AM, DEMOD_USB, DEMOD_NONE)
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

FLOAT_TOL = 1e-5
OSC = {"s16": orc.S16, "s8": orc.S8, "f32": orc.F32}


def gpu_bb(g_or_cfg, Fs=None, bs=None, float_path=0):
    c = g_or_cfg
    bb = IQBaseBand(str(c["scalar"]), float(c["Fc"]), float(c["Ff"]), float(c["width"]), int(c["order"]),
                    int(c["sub_sample_arg"] if "sub_sample_arg" in c else c["sub_sample"]), float(c["oFs"]))
    if "setcf" in c and int(c["setcf"]):
        bb.setCenterFrequency(float(c["Fc"]))
        bb.setFilterFrequency(float(c["Ff"]))
    if float_path:
        bb.setFloatPath(float_path)
    bb.config(sample_rate=float(c["Fs"]) if Fs is None else Fs, buffer_size=int(c["buffer_size"]) if bs is None else bs)
    return bb


def orc_bb(c, bs=None):
    bb = orc.IQBaseBand(OSC[str(c["scalar"])], float(c["Fc"]), float(c["Ff"]), float(c["width"]), int(c["order"]),
                        int(c["sub_sample_arg"] if "sub_sample_arg" in c else c["sub_sample"]), float(c["oFs"]))
    if "setcf" in c and int(c["setcf"]):
        bb.set_center_frequency(float(c["Fc"]))
        bb.set_filter_frequency(float(c["Ff"]))
    bb.config(float(c["Fs"]), int(c["buffer_size"]) if bs is None else bs)
    return bb


# ---- (1) golden vectors from the reference ------------------------------------------------------

@pytest.mark.parametrize("name", golden_names("bb_"))
def test_golden_per_buffer_nodes(name):
    """Node-by-node, buffer-by-buffer, like the reference harness drove the reference."""
    g = load_golden(name)
    sc = str(g["scalar"])
    bb, fm, am, usb = gpu_bb(g), FMDemod(sc), AMDemod(sc), USBDemod(sc)
    cfg = bb.out_config
    assert fm.config(cfg).type == _lib.T_S16
    x, bs = g["x"], int(g["buffer_size"])
    bbs, fms, ams, usbs, counts = [], [], [], [], []
    for off in range(0, x.shape[0], bs):
        y = bb.process(x[off:off + bs])
        counts.append(y.shape[0]); bbs.append(y)
        if y.shape[0]:
            fms.append(fm.process(y, in_place=True))
        ams.append(am.process(y)); usbs.append(usb.process(y))
    np.testing.assert_array_equal(np.array(counts, dtype=np.uint32), g["counts"])
    np.testing.assert_array_equal(np.concatenate(bbs), g["bb"])
    np.testing.assert_array_equal(np.concatenate(fms), g["fm"])
    np.testing.assert_array_equal(np.concatenate(ams), g["am"])
    np.testing.assert_array_equal(np.concatenate(usbs), g["usb"])


@pytest.mark.parametrize("name", golden_names("bb_"))
@pytest.mark.parametrize("demod,key", [(DEMOD_FM, "fm"), (DEMOD_AM, "am"), (DEMOD_USB, "usb")])
def test_golden_fused_chain(name, demod, key):
    """All whole buffers in ONE launch pair (sdrg_rxchain_process), then the ragged tail."""
    g = load_golden(name)
    bb = gpu_bb(g)
    chain = RxChain(bb, demod)
    x, bs = g["x"], int(g["buffer_size"])
    nfull = x.shape[0] // bs
    y1, a1, c1 = chain.process(x[:nfull * bs], bs)
    parts_bb, parts_a, counts = [y1], [a1], list(c1)
    rem = x.shape[0] - nfull * bs
    if rem:
        y2, a2, c2 = chain.process(x[nfull * bs:], rem)
        parts_bb.append(y2); parts_a.append(a2); counts += list(c2)
    np.testing.assert_array_equal(np.array(counts, dtype=np.uint32), g["counts"])
    np.testing.assert_array_equal(np.concatenate(parts_bb), g["bb"])
    np.testing.assert_array_equal(np.concatenate(parts_a), g[key])


# ---- (2) oracle on seeded inputs ----------------------------------------------------------------

def _stream_case(cfg, x, cuts, demod=DEMOD_FM):
    """GPU fed `x` cut at `cuts` (arbitrary buffer sizes) vs the oracle fed the same cuts."""
    sc = OSC[cfg["scalar"]]
    g, o = gpu_bb(cfg, bs=max(1, max(np.diff(cuts)))), orc_bb(cfg, bs=max(1, max(np.diff(cuts))))
    chain = RxChain(g, demod)
    ofm = orc.FMDemod(sc)
    for s, e in zip(cuts[:-1], cuts[1:]):
        if e == s:
            continue
        yb, ya, _ = chain.process(x[s:e], e - s)
        ob = o.process(x[s:e])
        np.testing.assert_array_equal(yb, ob)
        if ob.shape[0]:
            if demod == DEMOD_FM:
                np.testing.assert_array_equal(ya, ofm.process(ob, inplace=True))
            elif demod == DEMOD_AM:
                np.testing.assert_array_equal(ya, orc.amdemod(ob, sc))
            else:
                np.testing.assert_array_equal(ya, orc.usbdemod(ob, sc))


def test_c1_stream_ragged_cuts():
    cfg = dict(synth.C1)
    x = synth.c1_input(300000)
    cuts = [0, 1, 2, 3, 17, 64, 4096, 4097, 70000, 70049, 70050, 70051, 200000, 299999, 300000]
    _stream_case(cfg, x, cuts, DEMOD_FM)


@pytest.mark.parametrize("order,ss,Ff,scalar", [
    (15, 50, 0.0, "s16"),      # 14 stripped taps, real and symmetric: pre-added pairs (kernel variant 4)
    (16, 50, 0.0, "s16"),      # 15 stripped taps (odd): real taps, two multiplies per tap (variant 3)
    (31, 16, 0.0, "s16"),      # shortest window the per-warp kernel takes, 30 real symmetric taps
    (33, 17, 0.0, "s16"),      # 32 taps
    (15, 300, 0.0, "s16"),     # the warp touches <= 4 windows: REDUX path
    (9, 2083, 50e3, "s16"),    # complex taps, bank-like window length
    (15, 64, 0.0, "s8"),       # int8 samples through the per-warp kernel
    (21, 255, -30e3, "s8"),
])
def test_per_warp_kernel_tap_kinds_and_window_lengths(order, ss, Ff, scalar):
    """iqbb_warp_kernels.cu: every tap kind (complex / real / real symmetric) and both window-sum paths, full-scale
    input (wrap regime), ragged cuts that split windows and warp tiles anywhere."""
    cfg = dict(scalar=scalar, Fs=2.4e6, Fc=100e3, Ff=Ff, width=40e3, order=order, sub_sample=ss, oFs=0.0)
    dt = np.int16 if scalar == "s16" else np.int8
    full = np.iinfo(dt).max
    x = synth.iq_int(90000, 2.4e6, [(0.5 * full, 103e3, 0.0), (0.3 * full, 5e3, 0.5), (0.25 * full, -300e3, 1.0)], full // 8, order + ss, dt)
    if Ff == 0.0 and scalar == "s16":
        k, _ = gpu_bb(cfg, bs=4096).design()
        assert np.all(k[:, 1] == 0), "a filter centred on 0 Hz must have real taps"
    _stream_case(cfg, x, [0, 1, 255, 256, 257, 4095, 30000, 30001, 65536, 89999, 90000], DEMOD_FM)
    _stream_case(cfg, x, [0, 90000], DEMOD_AM)


def test_c1_full_size_buffers():
    """BASELINE config 1 at its real buffer size: 8 buffers of 65536, one launch pair."""
    cfg = dict(synth.C1)
    n = 8 * cfg["buffer_size"]
    x = synth.c1_input(n)
    g, o = gpu_bb(cfg), orc_bb(cfg)
    chain = RxChain(g, DEMOD_FM)
    yb, ya, counts = chain.process(x, cfg["buffer_size"])
    ofm = orc.FMDemod(orc.S16)
    obs, ofs = [], []
    for b in range(8):
        ob = o.process(x[b * cfg["buffer_size"]:(b + 1) * cfg["buffer_size"]])
        obs.append(ob); ofs.append(ofm.process(ob, inplace=True))
        assert counts[b] == ob.shape[0]
    np.testing.assert_array_equal(yb, np.concatenate(obs))
    np.testing.assert_array_equal(ya, np.concatenate(ofs))


def test_bank_channel_shape_wrap_regime():
    """One channel of config 4 (Fs=100e6 -> ss=2083) at an amplitude where S*ss wraps 2^31."""
    cfg = dict(scalar="s16", Fs=100e6, Fc=3.90625e5, Ff=3.90625e5, width=25e3, order=15, sub_sample=1,
               oFs=48000.0, buffer_size=1 << 18)
    x = synth.iq_int(1 << 19, 100e6, [(8192, 4.0e5, 0.0), (3000, -7e6, 1.0)], 64, 77, np.int16)
    _stream_case(cfg, x, [0, 1 << 18, 1 << 19], DEMOD_AM)
    _stream_case(cfg, x, [0, 5, 2083, 2084, 4167, 300000, 1 << 19], DEMOD_USB)


@pytest.mark.parametrize("order", [1, 2, 3, 8, 9, 16, 17, 64, 255])
def test_filter_orders(order):
    cfg = dict(scalar="s16", Fs=2.4e6, Fc=-250e3, Ff=-250e3, width=100e3, order=order, sub_sample=1,
               oFs=200e3, buffer_size=5000)
    x = synth.iq_int(20000, 2.4e6, [(9000, -240e3, 0.3), (5000, 600e3, 1.0)], 100, 5 + order, np.int16)
    _stream_case(cfg, x, [0, 5000, 10000, 10001, 20000], DEMOD_FM)


@pytest.mark.parametrize("ss", [1, 2, 3, 15, 16, 17, 2047, 2048, 2049, 5000])
def test_subsampling_factors(ss):
    cfg = dict(scalar="s16", Fs=2.4e6, Fc=100e3, Ff=90e3, width=50e3, order=21, sub_sample=ss, oFs=0.0,
               buffer_size=12000)
    x = synth.iq_int(36000, 2.4e6, [(12000, 103e3, 0.0)], 64, 100 + ss, np.int16)
    _stream_case(cfg, x, [0, 12000, 12001, 24000, 36000], DEMOD_FM)


def test_int8_stream():
    cfg = dict(scalar="s8", Fs=2.4e6, Fc=-100e3, Ff=-100e3, width=30e3, order=21, sub_sample=1, oFs=48000.0,
               buffer_size=20000)
    x = synth.iq_int(100000, 2.4e6, [(100, -103e3, 0.0), (27, 400e3, 2.0)], 6, 8, np.int8)
    _stream_case(cfg, x, [0, 20000, 20001, 60000, 100000], DEMOD_FM)
    cfg.update(Fc=0.0, Ff=0.0, sub_sample=4, oFs=0.0)
    _stream_case(cfg, x, [0, 3, 50000, 100000], DEMOD_AM)


def test_setters_mid_stream():
    """setCenterFrequency restarts the NCO phase, setFilterFrequency swaps the taps; state is kept."""
    cfg = dict(synth.C1)
    x = synth.c1_input(60000)
    g, o = gpu_bb(cfg, bs=20000), orc_bb(cfg, bs=20000)
    np.testing.assert_array_equal(g.process(x[:20000]), o.process(x[:20000]))
    g.setCenterFrequency(-50e3); o.set_center_frequency(-50e3)
    np.testing.assert_array_equal(g.process(x[20000:40000]), o.process(x[20000:40000]))
    g.setFilterFrequency(-50e3); o.set_filter_frequency(-50e3)
    np.testing.assert_array_equal(g.process(x[40000:]), o.process(x[40000:]))


def test_config_mid_stream_restarts_from_a_zero_history():
    """A second config() (or setSubsample / setOutputSampleRate) restarts the stream: window grid, NCO phase AND a
    zeroed FIR history, i.e. the node then behaves like a freshly built one.  (Documented deviation, DESIGN.md 2:
    the reference's _reconfigure() resets _ring_offset but leaves the previous samples in _ring, rotated, so its
    first order-1 outputs after a re-config see stale data; from output `order` on both agree.)"""
    cfg = dict(synth.C1)
    x = synth.c1_input(40000)
    g = gpu_bb(cfg, bs=20000)
    g.process(x[:20000])
    g.config(sample_rate=cfg["Fs"], buffer_size=20000)
    fresh = orc_bb(cfg, bs=20000)
    np.testing.assert_array_equal(g.process(x[20000:]), fresh.process(x[20000:]))
    g.setSubsample(7)                                   # oFs > 0 wins in config(): still ss = 50
    fresh = orc_bb(cfg, bs=20000)
    np.testing.assert_array_equal(g.process(x[:20000]), fresh.process(x[:20000]))


def test_device_tensor_arguments_are_validated():
    import torch
    cfg = dict(synth.C1)
    g = gpu_bb(cfg, bs=4096)
    x = torch.zeros((8192, 2), dtype=torch.int16, device="cuda")
    with pytest.raises(ConfigError):
        g.process(x[::2])                               # strided view
    with pytest.raises(ConfigError):
        g.process(x.to(torch.float32))                  # wrong element type
    with pytest.raises(ConfigError):
        g.process(torch.zeros((16, 2), dtype=torch.int16))   # host tensor through the device entry point
    assert g.process(x[:4096]).shape[0] == 81


def test_device_pointer_entry_points():
    import torch
    cfg = dict(synth.C1)
    x = synth.c1_input(4 * 65536)
    g, o = gpu_bb(cfg), orc_bb(cfg)
    xd = torch.from_numpy(x).cuda()
    chain = RxChain(g, DEMOD_FM)
    yb, ya, counts = chain.process(xd, 65536)
    torch.cuda.synchronize()
    ofm = orc.FMDemod(orc.S16)
    obs = [o.process(x[b * 65536:(b + 1) * 65536]) for b in range(4)]
    np.testing.assert_array_equal(yb.cpu().numpy(), np.concatenate(obs))
    np.testing.assert_array_equal(ya.cpu().numpy(), np.concatenate([ofm.process(b, inplace=True) for b in obs]))
    # stand-alone device demods on the device-resident base band
    am = AMDemod("s16").process(yb); usb = USBDemod("s16").process(yb)
    torch.cuda.synchronize()
    np.testing.assert_array_equal(am.cpu().numpy(), orc.amdemod(np.concatenate(obs), orc.S16))
    np.testing.assert_array_equal(usb.cpu().numpy(), orc.usbdemod(np.concatenate(obs), orc.S16))


def test_fm_out_of_place_leaves_element0():
    fm = FMDemod("s16")
    x = synth.c1_input(1000)
    out = np.full(1000, 1234, dtype=np.int16)
    got = fm.process(x, in_place=False, out=out)
    assert got[0] == 1234
    ref = orc.FMDemod(orc.S16).process(x, inplace=True)
    np.testing.assert_array_equal(got[1:], ref[1:])


def test_error_behaviour():
    bb = IQBaseBand("s16", 100e3, 100e3, 12.5e3, 15, 1, 48000.0)
    with pytest.raises(RuntimeError):
        bb.process(np.zeros((8, 2), dtype=np.int16))       # process() before config()
    with pytest.raises(ConfigError):
        bb.config(Config(_lib.T_CS8, 2.4e6, 4096, 1))
    with pytest.raises(ConfigError):
        FMDemod("s16").config(Config(_lib.T_CF32, 48e3, 100, 1))
    assert bb.config(Config(_lib.T_CS16, 2.4e6, 0, 1)).type == _lib.T_UNDEFINED   # incomplete: ignored
    bb.config(sample_rate=2.4e6, buffer_size=64)
    assert bb.process(np.zeros((0, 2), dtype=np.int16)).shape[0] == 0


# ---- float path (defined by the restatement; tolerance 1e-5 relative RMS) -----------------------

def _float_case(cfg, x, bs, demod=DEMOD_FM, path=0):
    g, o = gpu_bb(cfg, bs=bs, float_path=path), orc_bb(cfg, bs=bs)
    chain = RxChain(g, demod)
    yb, ya, counts = chain.process(x, bs)
    ofm = orc.FMDemod(orc.F32)
    obs, oas = [], []
    for b in range(x.shape[0] // bs):
        ob = o.process(x[b * bs:(b + 1) * bs])
        assert counts[b] == ob.shape[0]
        obs.append(ob)
        if demod == DEMOD_FM:
            oas.append(ofm.process(ob, inplace=True))
        elif demod == DEMOD_AM:
            oas.append(orc.amdemod(ob, orc.F32))
        else:
            oas.append(orc.usbdemod(ob, orc.F32))
    ob, oa = np.concatenate(obs), np.concatenate(oas)
    assert yb.shape == ob.shape
    e_bb = rel_rms(yb.astype(np.float64).view(np.complex128), ob.astype(np.float64).view(np.complex128))
    e_a = rel_rms(ya, oa)
    assert e_bb < FLOAT_TOL, e_bb
    assert e_a < FLOAT_TOL, e_a
    return e_bb, e_a


PATHS = [(1, "direct"), (2, "folded")]


@pytest.mark.parametrize("path", [1, 2], ids=["direct", "folded"])
def test_c2_float_chain(path):
    cfg = dict(synth.C2)
    x = synth.c2_input(2 << 20)
    e = _float_case(cfg, x, 1 << 20, DEMOD_FM, path)
    print("c2 rel-rms (bb, fm):", e)


@pytest.mark.parametrize("path", [1, 2], ids=["direct", "folded"])
@pytest.mark.parametrize("demod", [DEMOD_AM, DEMOD_USB, DEMOD_FM])
def test_float_small_configs(demod, path):
    cfg = dict(scalar="f32", Fs=2.4e6, Fc=-100e3, Ff=-100e3, width=30e3, order=21, sub_sample=1, oFs=48000.0)
    x = synth.iq_f32(200000, 2.4e6, [(0.5, -103e3, 0.0), (0.2, 500e3, 1.0)], 0.01, 3)
    _float_case(cfg, x, 50000, demod, path)          # ss=50, negative shift
    cfg.update(Fc=0.0, Ff=0.0, width=200e3)
    x0 = synth.iq_f32(200000, 2.4e6, [(0.5, 3e3, 0.0), (0.2, 500e3, 1.0)], 0.01, 4)
    _float_case(cfg, x0, 50000, demod, path)         # lut_inc == 0: mixer bypassed
    if path == 1:
        cfg.update(Fc=77e3, Ff=60e3, sub_sample=7, oFs=0.0, order=33)   # ss < order-1: direct only
        _float_case(cfg, x, 40000, demod, path)


@pytest.mark.parametrize("ss,order", [(32, 33), (33, 2), (63, 64), (64, 64), (100, 2), (416, 1), (417, 64), (512, 65), (513, 65), (600, 40),
                                      (127, 128), (130, 129), (200, 129), (300, 66), (416, 128), (512, 100), (512, 129), (513, 129), (416, 130),
                                      (768, 64), (1000, 64), (2083, 15), (5000, 64), (8191, 64), (8192, 64), (8193, 64), (300000, 128)])
@pytest.mark.parametrize("path", [2], ids=["folded"])
def test_float_folded_geometry(ss, order, path):
    """Folded kernel across window/segment geometries (window << segment, window >> segment,
    ss == order-1, order 1), ragged multi-call streams."""
    # Fc = Fs/16 is exactly representable by the NCO (inc = 2048): the 1.25 MHz tone lands on DC and
    # survives even the longest boxcar, so the relative error is well conditioned
    cfg = dict(scalar="f32", Fs=20e6, Fc=1.25e6, Ff=1.2e6, width=200e3, order=order, sub_sample=ss, oFs=0.0)
    n = 700000
    x = synth.iq_f32(n, 20e6, [(0.5, 1.25e6, 0.3), (0.3, -4e6, 1.0)], 0.02, 11)
    g, o = gpu_bb(cfg, bs=n, float_path=path), orc_bb(cfg, bs=n)
    cuts = [0, 1, 31, 32, 33, 2047, 2048, 2049, 100000, 100001, 400000, n]
    ys, os_ = [], []
    for s, e in zip(cuts[:-1], cuts[1:]):
        ys.append(g.process(x[s:e])); os_.append(o.process(x[s:e]))
        assert ys[-1].shape == os_[-1].shape
    y, ob = np.concatenate(ys), np.concatenate(os_)
    if ob.shape[0]:
        e = rel_rms(y.astype(np.float64).view(np.complex128), ob.astype(np.float64).view(np.complex128))
        assert e < FLOAT_TOL, e


def test_float_folded_misaligned_device_input():
    """An 8-byte (not 16-byte) aligned device pointer takes the LDG variant of the folded kernel;
    the 16-byte aligned one the TMA variant.  Both must agree with the oracle."""
    import torch
    cfg = dict(synth.C2)
    n = 300001
    x = synth.c2_input(n + 1)
    xd = torch.from_numpy(x).cuda()
    o = orc_bb(cfg, bs=n)
    ob = o.process(x[1:])
    for view in (xd[1:], xd[1:].clone()):
        g = gpu_bb(cfg, bs=n, float_path=2)
        y = g.process(view)
        torch.cuda.synchronize()
        e = rel_rms(y.cpu().numpy().astype(np.float64).view(np.complex128), ob.astype(np.float64).view(np.complex128))
        assert e < FLOAT_TOL, e


def test_float_folded_rejects_ineligible():
    bb = IQBaseBand("f32", 0.0, 0.0, 1e5, 64, 7, 0.0)
    bb.setFloatPath(2)
    with pytest.raises(ConfigError):
        bb.config(sample_rate=2.4e6, buffer_size=4096)


# ---- (3) size-independent properties at full size ------------------------------------------------

def test_full_size_buffering_invariance_int16():
    """Config 1, 64 buffers of 65536: one launch == 64 launches (bit-exact), and the count law."""
    import torch
    cfg = dict(synth.C1)
    bs, nb = cfg["buffer_size"], cfg["n_buffers"]
    x = synth.c1_input(bs * nb)
    xd = torch.from_numpy(x).cuda()
    a, b = gpu_bb(cfg), gpu_bb(cfg)
    ca, cb = RxChain(a, DEMOD_FM), RxChain(b, DEMOD_FM)
    ya, fa, counts = ca.process(xd, bs)
    yb, fb = [], []
    for k in range(nb):
        y, f, _ = cb.process(xd[k * bs:(k + 1) * bs], bs)
        yb.append(y.clone()); fb.append(f.clone())
    torch.cuda.synchronize()
    assert torch.equal(ya, torch.cat(yb)) and torch.equal(fa, torch.cat(fb))
    ss = a.info().sub_sample
    assert int(counts.sum()) == (bs * nb - 1) // ss
    # spot-check the head against the oracle
    o = orc_bb(cfg)
    np.testing.assert_array_equal(ya[:counts[0]].cpu().numpy(), o.process(x[:bs]))

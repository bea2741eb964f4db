"""Launch set-up (libsdr_b200/csrc/launch.cu): one module owns every kernel's shared-memory opt-in and resident-CTA
count, per (kernel, device).  The opt-in is only ever raised, under one lock, so host threads that drive one device
with nodes of different geometry cannot lower each other's opt-in below what a launch needs."""
import os
import re
import threading

import numpy as np
import pytest

from conftest import rel_rms
from libsdr_b200 import synth
from libsdr_b200.nodes import ChannelBank, FilterNode, IQBaseBand

CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "libsdr_b200", "csrc")
SETUP_MODULE = {"launch.cu", "launch.cuh"}


def test_launch_setup_lives_in_one_module():
    offenders = []
    for name in sorted(os.listdir(CSRC)):
        if name in SETUP_MODULE:
            continue
        text = open(os.path.join(CSRC, name), encoding="utf-8").read()
        for call in ("cudaFuncSetAttribute", "cudaOccupancyMaxActiveBlocksPerMultiprocessor"):
            if re.search(r"\b%s\b" % call, text):
                offenders.append((name, call))
    assert not offenders, offenders


PERWIN = 5     # sdrg_iqbb_last_float_kernel
FS_F = 20e6


def _float_perwin(ss, order):
    """IQBaseBand<float> on the per-window kernel: its shared memory (table + tiles) depends on ss and the order."""
    def make():
        g = IQBaseBand("f32", 1.25e6, 1.2e6, 200e3, order, ss, 0.0)
        g.config(sample_rate=FS_F, buffer_size=1 << 17)
        return g
    x = synth.iq_f32(4 << 17, FS_F, [(0.5, 1.25e6 + 2e3, 0.3), (0.3, -4e6, 1.0)], 0.02, ss)

    def run(g, kernels):
        ys = []
        for k in range(4):
            ys.append(g.process(x[k << 17:(k + 1) << 17]))
            kernels.append(g.lastFloatKernel())
        return np.concatenate(ys)
    return make, run


def _int16_generic(order):
    """IQBaseBand<int16_t> with more than 32 taps: the generic accumulate kernel, shared memory growing with the order
    (accum_smem_int; at most 46.6 KB, reached at order 1024)."""
    def make():
        g = IQBaseBand("s16", 100e3, 100e3, 12.5e3, order, 50, 0.0)
        g.config(sample_rate=2.4e6, buffer_size=1 << 16)
        return g
    x = synth.iq_int(4 << 16, 2.4e6, [(0.5, 103e3, 0.0), (0.2, 500e3, 1.0)], 0.01, order)

    def run(g, kernels):
        return np.concatenate([g.process(x[k << 16:(k + 1) << 16]) for k in range(4)])
    return make, run


def _int16_bank(order):
    """int16 channel bank with more than 32 taps: the generic bank kernel, 16 B x 32 channels x order of taps in shared
    memory -- above 48 KB from order 70 on, and different for every order."""
    Fc = np.array([-300e3, -100e3, 50e3, 250e3])

    def make():
        b = ChannelBank("s16", Fc, None, 12.5e3, order, 256, 0.0)
        b.config(sample_rate=2.4e6, buffer_size=1 << 15)
        return b
    x = synth.iq_int(4 << 15, 2.4e6, [(0.4, 52e3, 0.0), (0.3, -298e3, 1.0)], 0.01, order)

    def run(b, kernels):
        outs = [b.process(x[k << 15:(k + 1) << 15], 1 << 15, want=("bb", "fm")) for k in range(4)]
        return np.concatenate([np.concatenate([o["bb"].reshape(len(Fc), -1) for o in outs], axis=1),
                               np.concatenate([o["fm"].astype(np.int32) for o in outs], axis=1)], axis=1)
    return make, run


def _filter(block):
    """FilterNode with two filters: block 4096 runs the radix-16 convolution kernel (107 KB of shared memory, grid and
    spectrum scratch sized by its resident-CTA count), block 1024 the single-buffer radix-16 kernels."""
    def make():
        f = FilterNode(block)
        f.addFilter(100e3, 200e3)
        f.addFilter(-500e3, -300e3)
        f.config(sample_rate=2.4e6, buffer_size=block)
        return f
    x = synth.iq_f32(40 * block, 2.4e6, [(0.5, 150e3, 0.0), (0.3, -400e3, 1.0)], 0.01, block).view(np.complex64).reshape(-1)

    def run(f, kernels):
        return np.concatenate([f.process(x[k * 10 * block:(k + 1) * 10 * block]) for k in range(4)], axis=1)
    return make, run


# each thread owns nodes whose launches need different opt-ins from the other thread's
THREAD_NODES = [
    [("f32 ss 64 order 65", _float_perwin(64, 65), 1e-5), ("s16 order 40", _int16_generic(40), 0),
     ("s16 bank order 80", _int16_bank(80), 0), ("filter 4096", _filter(4096), 1e-5)],
    [("f32 ss 100 order 15", _float_perwin(100, 15), 1e-5), ("s16 order 1000", _int16_generic(1000), 0),
     ("s16 bank order 120", _int16_bank(120), 0), ("filter 1024", _filter(1024), 1e-5)],
]


@pytest.mark.gpu
def test_two_host_threads_with_different_opt_ins():
    """Two threads drive one device at once, each with its own nodes; every output equals what the same node gives on
    one thread (int16: bit for bit; float: within the float tolerance)."""
    barrier = threading.Barrier(len(THREAD_NODES))
    results = [dict() for _ in THREAD_NODES]
    errors = []

    def worker(t):
        try:
            nodes = [(name, make(), run, []) for name, (make, run), _ in THREAD_NODES[t]]
            barrier.wait()
            for name, node, run, kernels in nodes:
                results[t][name] = (run(node, kernels), kernels)
        except Exception as e:      # noqa: BLE001 -- reported below, with the thread it came from
            errors.append((t, repr(e)))

    threads = [threading.Thread(target=worker, args=(t,)) for t in range(len(THREAD_NODES))]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors

    for t, nodes in enumerate(THREAD_NODES):
        for name, (make, run), tol in nodes:
            got, kernels = results[t][name]
            want = run(make(), [])
            assert got.shape == want.shape, name
            if name.startswith("f32"):
                assert kernels and all(k == PERWIN for k in kernels), (name, kernels)
            if tol == 0:
                np.testing.assert_array_equal(got, want, err_msg=name)
            else:
                e = rel_rms(got.astype(np.complex128) if np.iscomplexobj(got) else got.astype(np.float64).view(np.complex128),
                            want.astype(np.complex128) if np.iscomplexobj(want) else want.astype(np.float64).view(np.complex128))
                assert e < tol, (name, e)

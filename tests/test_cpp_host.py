"""The C++ host-side mirror (include/sdrg/*.hh): buffer/refcount/config conformance on the CPU, and
the sdr_fm-shaped drop-in chain against the oracle on the GPU."""
import os
import subprocess

import pytest

from conftest import ROOT

BUILD = os.path.join(ROOT, "build", "tests")
LIBDIR = os.path.join(ROOT, "libsdr_b200")


def compile_cpp(name, extra=(), compat=False):
    os.makedirs(BUILD, exist_ok=True)
    out = os.path.join(BUILD, name)
    src = os.path.join(ROOT, "tests", "cpp", name + ".cc")
    inc = ["-I" + os.path.join(ROOT, "include")] + (["-I" + os.path.join(ROOT, "include", "sdrg", "compat")] if compat else [])
    cmd = ["g++", "-std=c++17", "-O2", "-Wall"] + inc + [src] + list(extra) + [
        "-o", out, "-L" + LIBDIR, "-l:libsdrg.so", "-Wl,-rpath," + LIBDIR, "-lpthread", "-lm"]
    subprocess.run(cmd, check=True, capture_output=True, text=True)
    return out


def test_buffer_and_node_conformance():
    exe = compile_cpp("buffer_test")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "buffer_test: ok" in r.stdout


def test_compat_headers_compile_reference_style_source(tmp_path):
    """A source file written against libsdr's own header names builds unchanged with the compat dir."""
    src = tmp_path / "ref_style.cc"
    src.write_text('#include "demod.hh"\n#include "baseband.hh"\n#include "queue.hh"\n#include "filternode.hh"\n#include "fftplan.hh"\nusing namespace sdr;\n'
                   "int main() { IQBaseBand<int16_t> *bb = 0; FMDemod<int16_t> *d = 0; (void)bb; (void)d; return 0; }\n")
    subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-I" + os.path.join(ROOT, "include", "sdrg", "compat"),
                    "-I" + os.path.join(ROOT, "include"), str(src)], check=True, capture_output=True, text=True)


@pytest.mark.parametrize("typ", ["u8", "s16", "cu8", "cs16"])
def test_wav_sink_and_source_match_reference_files(typ, tmp_path):
    """WavSink writes the reference's bytes; WavSource reads a reference-written file into the same buffers."""
    import numpy as np
    from conftest import load_golden
    g = load_golden("wav_" + typ)
    exe = compile_cpp("wav_test")
    inp, ref, pre = tmp_path / "in.raw", tmp_path / "ref.wav", tmp_path / "out"
    g["x"].tofile(inp); g["wav"].tofile(ref)
    r = subprocess.run([exe, typ, str(inp), str(int(g["buffer_size"])), repr(float(g["Fs"])), str(ref), str(pre)],
                       capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "wav_test: ok" in r.stdout
    np.testing.assert_array_equal(np.fromfile(str(pre) + ".wav", dtype=np.uint8), g["wav"])
    np.testing.assert_array_equal(np.fromfile(str(pre) + ".data", dtype=np.uint8), g["data"])
    np.testing.assert_array_equal(np.fromfile(str(pre) + ".counts", dtype=np.uint32), g["byte_counts"])
    np.testing.assert_array_equal(np.fromfile(str(pre) + ".cfg"), g["cfg"])


@pytest.mark.gpu
def test_sdr_fm_shaped_chain_bit_exact():
    os.makedirs(BUILD, exist_ok=True)
    obj = os.path.join(BUILD, "sdr_oracle.o")           # the checker, linked into the TEST binary only
    subprocess.run(["gcc", "-O2", "-fwrapv", "-c", os.path.join(ROOT, "oracle", "sdr_oracle.c"), "-o", obj], check=True)
    exe = compile_cpp("chain_test", extra=[obj])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "chain_test: ok" in r.stdout


@pytest.mark.gpu
def test_filternode_and_fftplan_classes():
    os.makedirs(BUILD, exist_ok=True)
    obj = os.path.join(BUILD, "sdr_oracle.o")
    subprocess.run(["gcc", "-O2", "-fwrapv", "-c", os.path.join(ROOT, "oracle", "sdr_oracle.c"), "-o", obj], check=True)
    exe = compile_cpp("filter_test", extra=[obj])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "filter_test: ok" in r.stdout


@pytest.mark.gpu
def test_full_sdr_fm_chain_with_reference_header_names():
    os.makedirs(BUILD, exist_ok=True)
    obj = os.path.join(BUILD, "sdr_oracle.o")
    subprocess.run(["gcc", "-O2", "-fwrapv", "-c", os.path.join(ROOT, "oracle", "sdr_oracle.c"), "-o", obj], check=True)
    exe = compile_cpp("sdr_fm_test", extra=[obj], compat=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "sdr_fm_test: ok" in r.stdout


@pytest.mark.gpu
def test_sharded_bank_c_application():
    """tests/cpp/bank_sharded_test.cc: plain C ABI, 2048 channels over every visible GPU, vs the oracle."""
    os.makedirs(BUILD, exist_ok=True)
    obj = os.path.join(BUILD, "sdr_oracle.o")
    subprocess.run(["gcc", "-O2", "-fwrapv", "-c", os.path.join(ROOT, "oracle", "sdr_oracle.c"), "-o", obj], check=True)
    exe = compile_cpp("bank_sharded_test", extra=[obj])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=180)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "bank_sharded_test: ok" in r.stdout


@pytest.mark.gpu
def test_wav_to_wav_real_baseband_fm_chain(tmp_path):
    os.makedirs(BUILD, exist_ok=True)
    obj = os.path.join(BUILD, "sdr_oracle.o")
    subprocess.run(["gcc", "-O2", "-fwrapv", "-c", os.path.join(ROOT, "oracle", "sdr_oracle.c"), "-o", obj], check=True)
    exe = compile_cpp("wav_chain_test", extra=[obj], compat=True)
    r = subprocess.run([exe, str(tmp_path)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "wav_chain_test: ok" in r.stdout


@pytest.mark.parametrize("typ,dt,ncomp", [("u8", "uint8", 1), ("s16", "int16", 1), ("cu8", "uint8", 2), ("cs16", "int16", 2)])
def test_wav_nodes_vs_live_reference(typ, dt, ncomp, tmp_path):
    """Random payload, odd sizes: the file our WavSink writes and the buffers our WavSource delivers == the reference's
    (its recorded outputs, tests/recorded.py; and its WavSink/WavSource themselves when oracle/_ref/ref_harness is built)."""
    import numpy as np
    import recorded
    harness = os.path.join(ROOT, "oracle", "_ref", "ref_harness")
    g = np.random.default_rng(len(typ) * 7 + ncomp)
    frames, bs, Fs = int(g.integers(1500, 5000)), int(g.choice([333, 1024, 4000])), float(g.choice([8000.0, 44100.0, 2.4e6]))
    info = np.iinfo(dt)
    x = g.integers(info.min, info.max + 1, size=frames * ncomp).astype(dt)
    inp, ref, pre, mine = tmp_path / "in.raw", tmp_path / "ref.wav", tmp_path / "ref", tmp_path / "mine"
    x.tofile(inp)
    live = os.path.exists(harness)
    if live:
        subprocess.run([harness, "wav", typ, str(inp), str(bs), repr(Fs), str(ref), str(pre)], check=True)
    # without the reference's build, our WavSource reads the file our WavSink has just written, whose bytes the
    # recorded digest pins to the reference's file
    exe = compile_cpp("wav_test")
    src = str(ref) if live else str(mine) + ".wav"
    r = subprocess.run([exe, typ, str(inp), str(bs), repr(Fs), src, str(mine)], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stdout + r.stderr
    outs = {ext[1:]: np.fromfile(str(mine) + ext, dtype=t)
            for ext, t in ((".wav", np.uint8), (".data", np.uint8), (".counts", np.uint32), (".cfg", np.float64))}
    recorded.check("wav_" + typ, **outs)
    if live:
        np.testing.assert_array_equal(outs["wav"], np.fromfile(str(ref), dtype=np.uint8))
        for ext, t in ((".data", np.uint8), (".counts", np.uint32), (".cfg", np.float64)):
            np.testing.assert_array_equal(outs[ext[1:]], np.fromfile(str(pre) + ext, dtype=t))

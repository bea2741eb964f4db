#!/usr/bin/env python
"""bench.py -- headline benchmark of the receive-chain hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1], "c2"): IQBaseBand<float>(64 taps, shift 100 kHz, 20 MS/s ->
48 kHz) + FMDemod on complex-float IQ.  One PASS = the fused chain over a batch of 256 buffers of
2^20 samples (256 Mi samples, 2 GiB > L2, so every pass streams from HBM); one STEP = R passes
(default 80, `config.passes_per_step`), so that the default 20 timed steps cover >= 0.5 s of
steady state.  Metric: input IQ Msamples/s.

  value    : device-resident throughput (inputs already in HBM), CUDA events, max over ranks
  burst    : the same over a short region (20 passes), the round-1 definition, for comparison
  e2e      : the same through the host-pointer C-ABI call (sdrg_rxchain_process) from pinned host
             memory, H2D of the step's input and D2H of its audio inside the timed region
  roofline : the dominant kernel (iqbb accumulate) timed with CUDA events on its launching stream
  cpu_baseline : the oracle port (the reference has no float instantiation) on one host core
  c5_bank  : BASELINE configs[4], the 2048-channel int16 bank sharded over the ranks (strong
             scaling), every rank's FM/AM rows stored straight into rank 0's HBM, with a bit-exact
             check of the gathered spot channels against the oracle outside the timed region

--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed pass returned -- the
base band (n, 2) and the demodulated audio (n,), float32 -- as DIR/baseband.npy and DIR/audio.npy
(above DUMP_LIMIT bytes in all, the same seeded sample of rows of both, plus DIR/sample_index.npy).
The input is seeded and the chain state depends only on the arguments, so two builds run with the
same arguments can be compared output for output.

N > 1: one process per GPU.  C2: every rank runs its own independent stream (weak scaling, no
data-path collective).  The demodulated audio of all ranks is gathered on rank 0 WITHOUT a
collective kernel: rank 0 exports a window of its HBM (CUDA IPC), the other ranks' finalize kernels
store into it over NVLink, progress flags order producer and consumer (libsdr_b200/parallel.py,
sdrg_peer_*).  NCCL carries the rendezvous, barriers and the max-over-ranks reductions, and is the
fallback gather (SDRG_BENCH_GATHER=nccl, or when the window cannot be mapped).
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from libsdr_b200 import synth  # noqa: E402

METRIC = "iq_msamples_per_s_iqbaseband_fmdemod"
UNIT = "Msamples/s"
G_BATCH = 8                       # passes per progress flag / per NCCL collective
C5_SPOT = (0, 1, 1023, 1024, 1025, 2047, 389, 1707)
DUMP_LIMIT = 64 * 10 ** 6         # bytes written by --dump-outputs at most


def workload():
    c = dict(synth.C2)
    c["n_buffers"] = 256        # one pass = 256 buffers of 2^20 samples = 2 GiB of cf32 per GPU
    return c


def config_block(c, n_gpus, passes, gather, extra=None):
    cfg = {"workload": "c2: IQBaseBand<float> 64-tap FIR, shift 100 kHz, 20 MS/s -> 48 kHz (ss=416) + FMDemod",
           "scalar": "cf32", "order": c["order"], "sample_rate": c["Fs"], "output_rate": c["oFs"],
           "buffer_size": c["buffer_size"], "buffers_per_pass": c["n_buffers"], "passes_per_step": passes,
           "buffers_per_step": c["n_buffers"] * passes,
           "samples_per_step_per_gpu": c["buffer_size"] * c["n_buffers"] * passes,
           "l2_policy": "inputs larger than L2 (%d MiB per pass per GPU)" % (c["buffer_size"] * c["n_buffers"] * 8 >> 20),
           "input": "3 tones + uniform noise (synth.c2_input), a 4 Mi-sample segment tiled to the batch",
           "parallelism": ("independent streams per GPU (replicas); audio of every rank gathered on rank 0: " + gather)
           if n_gpus > 1 else "single GPU"}
    if extra:
        cfg.update(extra)
    return cfg


def make_input(c, out=None):
    seg = synth.c2_input(4 << 20)
    reps = (c["buffer_size"] * c["n_buffers"]) // seg.shape[0]
    if out is None:
        return np.tile(seg, (reps, 1))
    out.reshape(reps, seg.shape[0], 2)[:] = seg
    return out


# ---- clocks ----------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, period_ms=10):
        self.index, self.period = index, period_ms
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", str(self.period)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    @staticmethod
    def mark():
        """Wall-clock mark (nvidia-smi stamps its samples with local time) to cut the log into regions."""
        return time.time()

    def stop(self, region=None):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush(); self.f.seek(0)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        for line in self.f.read().splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                import datetime
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except ValueError:
                ts = 0.0
            try:
                rows.append((float(parts[1]), float(parts[2]), float(parts[3]), [v.lower().startswith("active") for v in parts[5:9]], ts))
            except ValueError:
                continue

        def summarise(rs):
            if not rs:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
            reasons = sorted({nm for r in rs for nm, v in zip(names, r[3]) if v})
            return {"sm_mhz": float(np.median([r[0] for r in rs])), "sm_max_mhz": float(max(r[1] for r in rs)),
                    "power_w_max": float(max(r[2] for r in rs)), "reasons": reasons, "samples": len(rs)}

        out = summarise(rows)
        out["period_ms"] = self.period
        if region and region[1] > region[0]:
            out["timed_region"] = summarise([r for r in rows if region[0] <= r[4] <= region[1]])
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


# ---- stdout carries exactly ONE JSON line: everything else any library prints there (NCCL's banner and
#      INFO log) is sent to stderr by pointing fd 1 at fd 2 for the life of the process ----------------------
def claim_stdout():
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return saved


def emit_line(saved_fd, line):
    os.write(saved_fd, (json.dumps(line) + "\n").encode())


def nccl_logging_setup():
    """NCCL's INIT log at INFO level (communicator lines with rank / nranks, NVLS) -> stdout -> stderr (see
    claim_stdout), whatever level the launcher's environment had: the rank check needs those lines."""
    if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
        os.environ["NCCL_DEBUG"] = os.environ.get("SDRG_NCCL_DEBUG", "INFO")
        os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")


# ---- CPU baselines ---------------------------------------------------------------------------------
def cpu_port_run(c, x, threads, n_buffers):
    """The oracle port of the float chain on `threads` independent streams; returns Msamples/s."""
    from oracle import oracle as orc
    bs = c["buffer_size"]

    def one(res, k):
        o = orc.IQBaseBand(orc.F32, c["Fc"], c["Ff"], c["width"], c["order"], c["sub_sample"], c["oFs"])
        o.config(c["Fs"], bs)
        fm = orc.FMDemod(orc.F32)
        n = 0
        for b in range(n_buffers):
            y = o.process(x[(b % c["n_buffers"]) * bs:((b % c["n_buffers"]) + 1) * bs])
            if y.shape[0]:
                fm.process(y, inplace=True)
            n += bs
        res[k] = n

    res = [0] * threads
    ths = [threading.Thread(target=one, args=(res, k)) for k in range(threads)]
    t0 = time.perf_counter()
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    return sum(res) / dt / 1e6, dt


def reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores.  The
    reference has no float IQBaseBand/FMDemod (they do not compile/link), so the float workload is
    timed on the oracle port, one independent stream per host core."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    c = workload()
    c["n_buffers"] = 8                                # the sample only touches the first buffers of the batch
    x = make_input(c)
    cores = os.cpu_count() or 1
    nb = 2                                           # buffers per thread per step (bounded sample)
    for _ in range(max(args.warmup, 0)):
        cpu_port_run(c, x, cores, 1)
    vals, tot = [], 0.0
    for _ in range(args.steps):
        v, dt = cpu_port_run(c, x, cores, nb)
        vals.append(v); tot += dt
    value = float(np.mean(vals))
    sample = "%d threads x %d buffers of %d samples per step" % (cores, nb, c["buffer_size"])
    cfg = config_block(workload(), args.gpus, 1, "n/a (CPU)")
    # what this arm really runs per step: a bounded sample of the workload above
    cfg.update({"buffers_per_pass": cores * nb, "passes_per_step": 1, "buffers_per_step": cores * nb,
                "samples_per_step_per_gpu": cores * nb * c["buffer_size"],
                "sampled_from": "the c2 workload (256 buffers of 2^20 samples per pass per GPU)",
                "l2_policy": "n/a (CPU arm)", "parallelism": "%d host threads, one independent stream each" % cores})
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (computed in f64 on CPU)",
            "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def _time_steps(fn, steps, warmup, barrier):
    import torch
    for _ in range(warmup):
        fn()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    barrier()
    return e0.elapsed_time(e1) / steps


def _steps_for(fn, barrier, target_ms=250.0, lo=3, hi=2000):
    """Number of steps that covers ~target_ms, from a 2-step probe (after 2 warm-up steps)."""
    ms = _time_steps(fn, 2, 2, barrier)
    return int(min(hi, max(lo, math.ceil(target_ms / max(ms, 1e-3)))))


class Collective:
    """The handful of host-side reductions the bench needs (max over ranks), NCCL or nothing."""

    def __init__(self, dist, world, dev):
        self.dist, self.world, self.dev = dist, world, dev

    def barrier(self):
        import torch
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max(self, v):
        import torch
        if self.world > 1:
            t = torch.tensor([float(v)], dtype=torch.float64, device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            return float(t.item())
        return float(v)


# ---- C5: the sharded 2048-channel bank ------------------------------------------------------------------
def c5_bank(coll, rank, dev, use_window):
    """BASELINE configs[4]: 2048 IQBaseBand<int16> channels (15 taps, 100 MS/s -> 48 kHz) + FM + AM on one
    stream, channels sharded by contiguous ranges over the ranks (strong scaling).  Every rank's finalize
    kernels store their (channel, sample) rows straight into the gathered arrays in rank 0's HBM."""
    import torch
    from libsdr_b200 import parallel
    from libsdr_b200.nodes import ChannelBank
    world = coll.world
    c = dict(synth.C5)
    bs, nb = c["buffer_size"], 2
    C_ = c["channels"]
    fc_all = synth.bank_frequencies(C_, c["Fs"])
    fc, lo, hi = parallel.bank_frequencies_for_rank(rank, world, fc_all)
    carriers = sorted(set(range(0, C_, 128)) | set(C5_SPOT))
    x_np = synth.bank_input(bs, c, carriers=carriers)                  # identical on every rank (seeded)
    x = torch.from_numpy(x_np).to(dev).repeat(nb, 1)
    bank = ChannelBank("s16", fc, None, c["width"], c["order"], c["sub_sample"], c["oFs"])
    bank.config(sample_rate=c["Fs"], buffer_size=bs)
    ss = 2083
    stride = (bs * nb) // ss + 2
    layout, total = parallel.bank_window_layout(C_, stride)
    gather = "none (single GPU)"
    win = None
    if world > 1 and use_window:
        win = parallel.PeerWindow(total)
        if not win.ok:
            win = None
    local = None
    if win is not None:
        gather = "p2p: finalize kernels store into rank 0's HBM (CUDA IPC window over NVLink), progress flags, no collective"
        base = win.base + win.data_offset
    else:
        local = torch.zeros(total, dtype=torch.uint8, device=dev)       # N == 1, or staging for the NCCL fallback
        base = local.data_ptr()
        if world > 1:
            gather = "nccl all_gather of the per-rank rows (fallback)"
    cons = torch.cuda.Stream(device=dev) if (win is not None and rank == 0) else None
    counter = [0]
    row0 = lo * stride * 2

    def ptrs(slot):
        return {"fm": base + layout[(slot, "fm")] + row0, "am": base + layout[(slot, "am")] + row0}

    def stream_ptr():
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def step():
        k = counter[0]; counter[0] += 1
        slot = k & 1
        if win is not None:
            if k >= 2:
                win.wait(win.ack(), 1, k - 1, stream_ptr())             # the consumer released this slot
            bank.process_into(x, bs, ptrs(slot), stride)
            win.signal(win.slot(rank), k + 1, stream_ptr())
            if cons is not None:
                sp = C.c_void_p(cons.cuda_stream)
                win.wait(win.slot(0), world, k + 1, sp)                 # every rank's rows of step k have landed
                win.signal(win.ack(), k + 1, sp)
        else:
            bank.process_into(x, bs, ptrs(slot), stride)
            if world > 1:
                for kind in ("fm", "am"):
                    o = layout[(slot, kind)]
                    rows = local[o + row0: o + row0 + (hi - lo) * stride * 2].view(torch.int16).view(hi - lo, stride)
                    parallel.gather_channel_outputs(rows, C_)

    def join():
        if cons is not None:
            torch.cuda.current_stream().wait_stream(cons)

    # ---- correctness of the gathered result, outside the timed region: a fresh stream, one step
    coll.barrier()
    bank.process_into(x, bs, ptrs(0), stride)
    coll.barrier()
    check = None
    if rank == 0:
        from oracle import oracle as orc
        n_out = (bs * nb - 1) // ss
        got = {}
        for kind in ("fm", "am"):
            if win is not None:
                raw = win.read(win.data_offset + layout[(0, kind)], C_ * stride * 2)
                got[kind] = raw.view(np.int16).reshape(C_, stride)
            elif world == 1:
                o = layout[(0, kind)]
                got[kind] = local[o:o + C_ * stride * 2].cpu().numpy().view(np.int16).reshape(C_, stride)
        if world > 1 and win is None:
            got = None
        bad, checked = 0, 0
        if got is not None:
            x2 = np.concatenate([x_np] * nb)
            for ch in C5_SPOT:
                o = orc.IQBaseBand(orc.S16, fc_all[ch], fc_all[ch], c["width"], c["order"], c["sub_sample"], c["oFs"])
                o.config(c["Fs"], bs)
                fm = orc.FMDemod(orc.S16)
                off, f_all, a_all, mask = 0, [], [], []
                for b in range(nb):
                    y = o.process(x2[b * bs:(b + 1) * bs])
                    f = fm.process(y, inplace=False)
                    f_all.append(f); a_all.append(orc.amdemod(y, orc.S16))
                    m = np.ones(y.shape[0], dtype=bool); m[0] = False          # element 0 of a buffer is never written
                    mask.append(m); off += y.shape[0]
                f_all, a_all, mask = np.concatenate(f_all), np.concatenate(a_all), np.concatenate(mask)
                assert f_all.shape[0] == n_out
                bad += int(np.count_nonzero(got["am"][ch, :n_out] != a_all))
                bad += int(np.count_nonzero(got["fm"][ch, :n_out][mask] != f_all[mask]))
                checked += 1
            check = {"channels": checked, "channel_ids": list(C5_SPOT), "outputs_per_channel": int(n_out), "kinds": ["fm", "am"],
                     "bit_exact": bad == 0, "mismatches": bad, "against": "oracle (oracle/sdr_oracle.c), gathered arrays read from rank 0"}
        else:
            check = {"channels": 0, "bit_exact": None, "note": "NCCL fallback gathers into temporaries; not checked"}
    ok = coll.max(0.0 if (check is None or check.get("bit_exact") is not False) else 1.0)
    if ok != 0.0:
        if rank == 0:
            sys.stderr.write("bench.py: C5 gathered output differs from the oracle: %r\n" % (check,))
        raise SystemExit(3)

    # ---- timing: continue the stream; flags restart from the counter
    bank.config(sample_rate=c["Fs"], buffer_size=bs)
    coll.barrier()
    steps = int(coll.max(_steps_for(lambda: (step(), join()), coll.barrier)))
    ms = coll.max(_time_steps(lambda: (step(), join()), steps, 2, coll.barrier))
    if win is not None and win.timed_out():
        raise SystemExit("bench.py: a peer-window wait timed out (C5)")
    imad_peak = 148 * 64 * 1.965e9           # FMA-heavy pipe: 64 IMAD lanes / clk / SM
    chan_ms = C_ * bs * nb / ms / 1e3
    out = {"workload": "c5: 2048-channel IQBaseBand<int16> bank (15 taps, 100 MS/s -> 48 kHz, ss=2083) + FMDemod + AMDemod, "
                       "channels sharded over %d GPU(s) by contiguous ranges, every rank reads the whole input" % world,
           "metric": "channel_msamples_per_s", "value": chan_ms, "unit": "channel*Msamples/s", "n_gpus": world,
           "input_msamples_per_s": bs * nb / ms / 1e3, "ms_per_step": ms, "steps": steps, "timed_region_s": ms * steps / 1e3,
           "buffers_per_step": nb, "buffer_size": bs, "scaling": "strong (channels fixed)", "gather": gather,
           "bound": "FMA-heavy (IMAD) pipe", "imad_pipe_frac_est": chan_ms * 1e6 * (3 * 14 + 4) / (imad_peak * world),
           "c5_check": check}
    if win is not None:
        coll.barrier()
        win.close()
    return out


def secondary_workloads(coll, dev, x_c2):
    """Short single-GPU measurements of the other shapes (not the headline line): C1, the 8(f) rows next
    to the path, C3, and the float path off the C2 geometry."""
    import torch
    from libsdr_b200 import _lib as L
    from libsdr_b200.nodes import IQBaseBand, BaseBand, RxChain, FilterNode, FFTPlan, DEMOD_FM
    out = {}
    barrier = coll.barrier
    peak = hbm_peak()[0]

    def timed(fn):
        return _time_steps(fn, _steps_for(fn, barrier, target_ms=120.0), 1, barrier)

    try:   # C1: int16, 15 taps, 2.4 MS/s -> 48 kHz + FM
        c = dict(synth.C1)
        bs, nb = c["buffer_size"], 2048
        x = torch.from_numpy(synth.c1_input(16 * bs)).to(dev).repeat(nb // 16, 1)
        bb = IQBaseBand("s16", c["Fc"], c["Ff"], c["width"], c["order"], c["sub_sample"], c["oFs"])
        bb.config(sample_rate=c["Fs"], buffer_size=bs)
        ch = RxChain(bb, DEMOD_FM)
        ms = timed(lambda: ch.process(x, bs))
        out["c1_int16"] = {"workload": "IQBaseBand<int16> 15 taps, 2.4 MS/s -> 48 kHz + FMDemod, %d buffers of %d" % (nb, bs),
                           "msamples_per_s": bs * nb / ms / 1e3, "ms_per_step": ms,
                           "algorithmic_gbs": (4 + 2 / 50) * bs * nb / ms / 1e6, "bound": "FMA-heavy (IMAD) pipe (bit-exact path)",
                           "imad_pipe_frac_est": bs * nb / (ms * 1e-3) * (3 * 14 + 4) / (148 * 64 * 1.965e9)}
        # the sdr_rec configuration: filter centred on 0 Hz (Ff == 0) => real symmetric taps
        bb0 = IQBaseBand("s16", c["Fc"], 0.0, c["width"], c["order"], c["sub_sample"], c["oFs"])
        bb0.config(sample_rate=c["Fs"], buffer_size=bs)
        ch0 = RxChain(bb0, DEMOD_FM)
        ms0 = timed(lambda: ch0.process(x, bs))
        out["c1_int16_real_taps"] = {"workload": "same with Ff = 0 (real symmetric taps, the sdr_rec configuration)",
                                     "msamples_per_s": bs * nb / ms0 / 1e3, "ms_per_step": ms0, "vs_complex_taps": ms / ms0}
        del ch, ch0, bb, bb0
    except Exception as e:  # pragma: no cover
        out["c1_int16"] = {"error": str(e)[:200]}
    try:   # SURVEY 8(f) rows next to the path: RTL-style cu8 input with AutoCast fused into the load, and the real-input BaseBand<int16>
        c = dict(synth.C1)
        bs, nb = c["buffer_size"], 2048
        g = torch.Generator(device="cpu"); g.manual_seed(0x5D12)
        x8 = torch.randint(0, 256, (nb * bs, 2), dtype=torch.uint8, generator=g).to(dev)
        bb = IQBaseBand("s16", c["Fc"], c["Ff"], c["width"], c["order"], c["sub_sample"], c["oFs"])
        bb.setInputType(L.T_CU8); bb.config(sample_rate=c["Fs"], buffer_size=bs)
        ch = RxChain(bb, DEMOD_FM)
        ms = timed(lambda: ch.process(x8, bs))
        out["c1_cu8_fused_autocast"] = {"workload": "complex uint8 -> AutoCast fused into IQBaseBand<int16> (15 taps, ss=50) + FMDemod, %d buffers of %d" % (nb, bs),
                                        "msamples_per_s": bs * nb / ms / 1e3, "ms_per_step": ms,
                                        "algorithmic_gbs": (2 + 2 / 50) * bs * nb / ms / 1e6, "bound": "FMA-heavy (IMAD) pipe (bit-exact path)"}
        xr = torch.randint(-32768, 32768, (nb * bs,), dtype=torch.int16, generator=g).to(dev)
        rb = BaseBand(300e3, 300e3, 50e3, 32, 50); rb.config(sample_rate=c["Fs"], buffer_size=bs)
        chr_ = RxChain(rb, DEMOD_FM)
        ms = timed(lambda: chr_.process(xr, bs))
        out["real_baseband_int16"] = {"workload": "BaseBand<int16> on a real int16 stream (32 taps, ss=50) + FMDemod, %d buffers of %d" % (nb, bs),
                                      "msamples_per_s": bs * nb / ms / 1e3, "ms_per_step": ms,
                                      "algorithmic_gbs": (2 + 2 / 50) * bs * nb / ms / 1e6, "bound": "FMA-heavy (IMAD) pipe (bit-exact path)"}
        del ch, chr_, bb, rb, x8, xr
    except Exception as e:  # pragma: no cover
        out["next_rows"] = {"error": str(e)[:200]}
    try:   # C3: FFT-convolution filter, block 4096; and a 4-filter bank on the same input
        c = dict(synth.C3)
        nb = c["n_buffers"]
        x = torch.from_numpy(synth.c2_input(c["buffer_size"])).to(dev).repeat(nb, 1).view(torch.complex64).reshape(-1)
        n = x.shape[0]
        f = FilterNode(c["block"]); f.addFilter(c["fmin"], c["fmax"]); f.config(sample_rate=c["Fs"], buffer_size=c["block"])
        ms = timed(lambda: f.process(x))
        out["c3_filter"] = {"workload": "FilterNode<float> block 4096 (FFT 8192), 1 band-pass filter, %d buffers of 2^20" % nb,
                            "msamples_per_s": n / ms / 1e3, "ms_per_step": ms, "algorithmic_gbs": 16 * n / ms / 1e6,
                            "hbm_frac": 16 * n / ms / 1e6 / peak, "bound": "shared memory / FP32 (Stockham FFT)"}
        f4 = FilterNode(c["block"])
        for k in range(4):
            f4.addFilter(c["fmin"] + k * 400e3, c["fmax"] + k * 400e3)
        f4.config(sample_rate=c["Fs"], buffer_size=c["block"])
        ms4 = timed(lambda: f4.process(x))
        out["c3_filter_bank4"] = {"workload": "same input, 4 band-pass filters on one FilterSink (forward FFT shared)",
                                  "input_msamples_per_s": n / ms4 / 1e3, "ms_per_step": ms4, "algorithmic_gbs": (8 + 8 * 4) * n / ms4 / 1e6,
                                  "hbm_frac": (8 + 8 * 4) * n / ms4 / 1e6 / peak}
        del f, f4
        nt = 8192
        xb = torch.view_as_complex(torch.randn((1 << 27, 2), dtype=torch.float32, device=dev))   # 1 GiB of transforms
        plan = FFTPlan(nt, FFTPlan.FORWARD)
        msf = timed(lambda: plan(xb))
        out["fft_8192_batch"] = {"workload": "FFTPlan<float> n=8192, 1 GiB of contiguous transforms", "ms_per_gib": msf,
                                 "read_write_gbs": 2 * xb.numel() * 8 / msf / 1e6, "hbm_frac": 2 * xb.numel() * 8 / msf / 1e6 / peak}
        del x, xb, plan
    except Exception as e:  # pragma: no cover
        out["c3_filter"] = {"error": str(e)[:200]}
    try:   # the float path off the C2 geometry: short windows, long windows, many taps
        xf = x_c2                                                           # the headline batch: 256 Mi samples = 2 GiB
        n = xf.shape[0]
        shapes = [("ss16_15taps", 15, 16), ("ss24_25taps", 25, 24), ("ss50_15taps", 15, 50), ("ss64_32taps", 32, 64), ("ss128_20taps", 20, 128),
                  ("ss416_64taps_c2", 64, 416),
                  ("ss1000_64taps", 64, 1000), ("ss4096_64taps", 64, 4096), ("ss20000_64taps", 64, 20000), ("ss416_128taps", 128, 416)]
        fl = {}
        for name, order, ss in shapes:
            bb = IQBaseBand("f32", 100e3, 100e3, 12.5e3, order, ss, 0.0)
            bb.config(sample_rate=20e6, buffer_size=1 << 20)
            ch = RxChain(bb, DEMOD_FM)
            ms = timed(lambda: ch.process(xf, 1 << 20))
            gbs = (8 + 4 / ss) * n / ms / 1e6
            kern = {1: "direct FIR", 2: "folded, batched", 3: "folded, window-pipelined", 4: "folded, staged short windows",
                    5: "folded, per-window (V table)", 6: "folded, TMA staging"}.get(bb.lastFloatKernel(), "?")
            fl[name] = {"order": order, "sub_sample": ss, "msamples_per_s": n / ms / 1e3, "algorithmic_gbs": gbs, "hbm_frac": gbs / peak,
                        "kernel": kern}
            del ch, bb
        out["float_shapes"] = fl
    except Exception as e:  # pragma: no cover
        out["float_shapes"] = {"error": str(e)[:200]}
    return out


def dump_outputs(path, arrays):
    """Writes path/<name>.npy for each (n, ...) array of `arrays`; above DUMP_LIMIT bytes in all, the same
    seeded sample of rows of every array, and its row numbers as sample_index.npy."""
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a[:1].nbytes for a in arrays.values())
    if n * row_bytes > DUMP_LIMIT:
        m = (DUMP_LIMIT - 4096) // (row_bytes + 8)                      # 4096: room for the .npy headers
        idx = np.sort(np.random.default_rng(0).choice(n, m, replace=False))
        arrays = dict({k: a[idx] for k, a in arrays.items()}, sample_index=idx.astype(np.float64))
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def hbm_peak():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    if "hbm_gbs" in peaks:
        return float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def pin_to_numa_node(node):
    """Run this process's threads on the CPUs of `node` (the feeding thread next to its GPU)."""
    try:
        txt = open("/sys/devices/system/node/node%d/cpulist" % node).read().strip()
        cpus = set()
        for part in txt.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


# ---- our arm -----------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the short C1/C3/float side measurements")
    ap.add_argument("--no-c5", action="store_true", help="skip the sharded 2048-channel bank")
    ap.add_argument("--buffers", type=int, default=0, help="buffers per pass (default: the workload's n_buffers)")
    ap.add_argument("--passes", type=int, default=int(os.environ.get("SDRG_BENCH_PASSES", "80")),
                    help="passes over the 2 GiB batch per step (rounded up to a multiple of %d)" % G_BATCH)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed pass as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        reference_arm(args)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    out_fd = claim_stdout()
    if world > 1:
        nccl_logging_setup()

    import torch
    from libsdr_b200 import _lib, parallel
    from libsdr_b200.nodes import IQBaseBand, RxChain, DEMOD_FM

    dist = None
    if args.gpus > 1 and world == 1:
        sys.stderr.write("bench.py: --gpus %d without torch.distributed.run (WORLD_SIZE unset): measuring ONE GPU, n_gpus=1 in the line\n" % args.gpus)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    _lib.call("sdrg_set_device", local)
    dev = torch.device("cuda", local)
    coll = Collective(dist, world, dev)
    W = max(args.warmup, 3)
    K = args.steps
    R = max(G_BATCH, (max(args.passes, 1) + G_BATCH - 1) // G_BATCH * G_BATCH)

    c = workload()
    if args.buffers:
        c["n_buffers"] = args.buffers
    bs, nb = c["buffer_size"], c["n_buffers"]
    n_pass = bs * nb

    # pinned host input next to this rank's GPU (NUMA node from sysfs), the feeding process pinned there too
    hp, node = C.c_void_p(), C.c_int(-1)
    _lib.call("sdrg_host_alloc", n_pass * 8, local, C.byref(hp), C.byref(node))
    node_cpus = pin_to_numa_node(node.value) if node.value >= 0 else 0
    x_np = np.ctypeslib.as_array(C.cast(hp, C.POINTER(C.c_float)), shape=(n_pass, 2))
    make_input(c, x_np)
    x_dev = torch.empty((n_pass, 2), dtype=torch.float32, device=dev)
    _lib.call("sdrg_memcpy_h2d_async", C.c_void_p(x_dev.data_ptr()), hp, n_pass * 8, None)
    torch.cuda.synchronize()

    bb = IQBaseBand("f32", c["Fc"], c["Ff"], c["width"], c["order"], c["sub_sample"], c["oFs"])
    bb.config(sample_rate=c["Fs"], buffer_size=bs)
    chain = RxChain(bb, DEMOD_FM)
    ss = bb.info().sub_sample
    cap = n_pass // ss + 2                                   # audio samples per pass (upper bound)
    bb_out = torch.empty((cap, 2), dtype=torch.float32, device=dev)

    # ---- the gather of the demodulated audio on rank 0 (see the module docstring)
    G = G_BATCH
    mode = os.environ.get("SDRG_BENCH_GATHER", "p2p")
    win = None
    if world > 1 and mode == "p2p":
        win = parallel.PeerWindow(world * 2 * G * cap * 4)
        if not win.ok:
            win = None
    if world == 1:
        gather = "none"
    elif win is not None:
        gather = ("p2p: finalize kernels store into rank 0's HBM (CUDA IPC window over NVLink), one progress flag per %d passes, "
                  "two rings, no collective kernel" % G)
    else:
        gather = "nccl all_gather_into_tensor, %d passes per collective, overlapped (fallback)" % G
    rings = [torch.zeros((G, cap), dtype=torch.float32, device=dev) for _ in range(2)] if win is None else None
    gathered2 = [torch.empty((world, G, cap), dtype=torch.float32, device=dev) for _ in range(2)] if (world > 1 and win is None) else None
    pending = [None, None]
    cons = torch.cuda.Stream(device=dev) if (win is not None and rank == 0) else None
    counter = [0]
    last = [None]                                            # what the latest pass returned (--dump-outputs)

    # Per-kernel CUDA events (sdrg_profile) are recorded on every 16th pass of the timed region: the event
    # records between the kernels cost ~3 % of a pass when taken on every one.
    prof_every = int(os.environ.get("SDRG_BENCH_PROFILE_EVERY", "16"))
    prof_live, prof_k0, prof_off = [False], [0], [3]

    def stream_ptr():
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def pass_dev():
        k = counter[0]
        counter[0] += 1
        if prof_live[0]:
            _lib.profile_enable((k - prof_k0[0]) % prof_every == prof_off[0])
        b, slot = divmod(k, G)
        ring = b & 1
        if win is not None:
            if slot == 0 and b >= 2:
                win.wait(win.ack(), 1, b - 1, stream_ptr())             # the consumer released this ring
            audio = win.base + win.data_offset + (((rank * 2 + ring) * G + slot) * cap) * 4
            last[0] = (chain.process_into(x_dev, bs, bb_out.data_ptr(), audio, cap), audio - win.base)
            if slot == G - 1:
                win.signal(win.slot(rank), b + 1, stream_ptr())
                if cons is not None:                                     # rank 0's consumer stream: all rows of batch b are in
                    sp = C.c_void_p(cons.cuda_stream)
                    win.wait(win.slot(0), world, b + 1, sp)
                    win.signal(win.ack(), b + 1, sp)
            return
        if slot == 0 and pending[ring] is not None:
            pending[ring].wait()                    # the gather that last read this ring has finished
            pending[ring] = None
        last[0] = chain.process(x_dev, bs, bb_out=bb_out, audio_out=rings[ring][slot])
        if world > 1 and slot == G - 1:
            pending[ring] = dist.all_gather_into_tensor(gathered2[ring], rings[ring], async_op=True)

    def drain():
        """Everything the timed passes started has completed on this rank's current stream."""
        if cons is not None:
            torch.cuda.current_stream().wait_stream(cons)
        for i, w in enumerate(pending):
            if w is not None:
                w.wait()
                pending[i] = None

    def step_dev():
        for _ in range(R):
            pass_dev()

    barrier = coll.barrier
    for _ in range(W):
        step_dev()
    drain()
    barrier()

    # burst figure (round-1 definition): 20 passes, timed alone
    bev0, bev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nburst = 24                                              # a multiple of G
    bev0.record()
    for _ in range(nburst):
        pass_dev()
    drain()
    bev1.record()
    barrier()
    burst_ms = coll.max(bev0.elapsed_time(bev1))

    sampler = ClockSampler(local, 10)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    _lib.profile_read(_lib.KERNEL_IQBB_ACCUM); _lib.profile_read(_lib.KERNEL_IQBB_FINALIZE)
    prof_live[0] = True
    prof_k0[0] = counter[0]
    l0 = _lib.kernel_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    m0 = sampler.mark() if rank == 0 else 0
    ev0.record()
    for _ in range(K):
        step_dev()
    drain()
    ev1.record()
    barrier()
    m1 = sampler.mark() if rank == 0 else 0
    launches = _lib.kernel_launch_count() - l0
    prof_live[0] = False
    _lib.profile_enable(False)
    ms = coll.max(ev0.elapsed_time(ev1))
    acc_ms, acc_n = _lib.profile_read(_lib.KERNEL_IQBB_ACCUM)
    fin_ms, fin_n = _lib.profile_read(_lib.KERNEL_IQBB_FINALIZE)
    if args.dump_outputs and rank == 0:
        if win is not None:                                  # rank 0's audio lies in its own peer window
            got, off = last[0]
            yb, ya = bb_out[:got].cpu().numpy(), win.read(off, got * 4).view(np.float32)
        else:
            yb, ya = (t.cpu().numpy() for t in last[0][:2])
        dump_outputs(args.dump_outputs, {"baseband": yb, "audio": ya})
    if win is not None and win.timed_out():
        raise SystemExit("bench.py: a peer-window wait timed out")
    value = world * n_pass * R * K / (ms * 1e-3) / 1e6
    burst_value = world * n_pass * nburst / (burst_ms * 1e-3) / 1e6

    # ---- end to end: host pointers through the C ABI, pinned input, audio read back
    n_out = bb.outputs_for(n_pass)
    ap_, anode = C.c_void_p(), C.c_int(-1)
    _lib.call("sdrg_host_alloc", (n_out + 1) * 4, local, C.byref(ap_), C.byref(anode))
    K2 = max(3, min(K, 5))

    def step_e2e():
        got = C.c_size_t(0)
        _lib.call("sdrg_rxchain_process", chain._h, hp, bs, nb, None, ap_, n_out + 1, C.byref(got), None)
        return got.value

    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    got = 0
    for _ in range(K2):
        got = step_e2e()
    barrier()
    e2e_s = coll.max(time.perf_counter() - t0)
    e2e_value = world * n_pass * K2 / e2e_s / 1e6
    # what the host can feed: the same pinned buffer through plain cudaMemcpyAsync, all ranks at once
    barrier()
    t0 = time.perf_counter()
    for _ in range(K2):
        _lib.call("sdrg_memcpy_h2d_async", C.c_void_p(x_dev.data_ptr()), hp, n_pass * 8, None)
    barrier()
    copy_s = coll.max(time.perf_counter() - t0)
    clocks = sampler.stop((m0, m1)) if rank == 0 else None

    c5 = None
    if not args.no_c5:
        c5 = c5_bank(coll, rank, dev, mode == "p2p")
    secondary = {}
    if world == 1 and not args.no_secondary:
        secondary = secondary_workloads(coll, dev, x_dev)

    if rank == 0:
        peak, peak_src = hbm_peak()
        alg_bytes = n_pass * 8 + (n_pass // ss) * 4         # cf32 in + float FM out (SURVEY.md 8d: 8 + 4/ss B/sample)
        k_ms = acc_ms / max(acc_n, 1)
        achieved = alg_bytes / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("iqbb_accum_f32_c2_bytes_per_launch")
        except Exception:
            pass
        ms_pass = ms / (K * R)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config_block(c, world, R, gather),
                "timed_region_s": ms / 1e3, "ms_per_pass": ms_pass,
                "burst": {"value": burst_value, "unit": UNIT, "passes": nburst, "ms_per_pass": burst_ms / nburst,
                          "note": "short region timed alone (round-1 definition); `value` is the sustained figure"},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(n_pass * 8),
                        "d2h_bytes_per_step": int(got * 4), "steps": K2,
                        "h2d_gbs_per_gpu": n_pass * 8 * K2 / e2e_s / 1e9,
                        "plain_copy_h2d_gbs_per_gpu": n_pass * 8 * K2 / copy_s / 1e9,
                        "frac_of_plain_copy": copy_s / e2e_s,
                        "host_numa_node": node.value, "feeder_cpus": node_cpus,
                        "note": "one step = one pass (2 GiB) per GPU through sdrg_rxchain_process: chunked upload on two copy "
                                "streams overlapped with the kernels; plain_copy = cudaMemcpyAsync of the same pinned buffer, "
                                "all ranks at once (the host-side ceiling)"},
                "gpu_launches": int(launches),
                "roofline": {"bound": "hbm", "kernel": "iqbb accumulate (FIR->NCO->window sums), float",
                             "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic, "peak_source": peak_src,
                             "kernel_timing": "CUDA events on the launching stream around the kernel, every %d-th pass of the timed region (offset %d)" % (prof_every, prof_off[0]),
                             "peak_note": "the measured peak is a copy (read + write) figure; this kernel is a pure read stream, "
                                          "which HBM3e serves slightly faster, so frac can exceed 1",
                             "kernel_ms": k_ms, "kernel_launches": int(acc_n),
                             "kernel_share_of_step": (k_ms / ms_pass) if ms > 0 and k_ms else None,
                             "finalize_ms": fin_ms / max(fin_n, 1)},
                "clocks": clocks, "c5_bank": c5, "secondary": secondary}
        if clocks and (clocks.get("timed_region") or {}).get("samples"):      # the headline fields describe the timed region
            whole = {k: clocks.get(k) for k in ("sm_mhz", "reasons", "samples", "power_w_max")}
            line["clocks"].update({k: clocks["timed_region"][k] for k in ("sm_mhz", "reasons", "power_w_max")})
            line["clocks"]["whole_run"] = whole
        if world == 1 and not args.no_cpu_baseline:
            nbuf = 24
            cc = dict(c); cc["n_buffers"] = min(nb, 24)
            v, dt = cpu_port_run(cc, x_np, 1, nbuf)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": 1, "kind": "port",
                                    "sample": "%d buffers of %d samples, oracle port of the float chain (the reference "
                                              "has no float instantiation), %.1f s" % (nbuf, bs, dt)}
            ref = os.path.join(ROOT, "oracle", "_ref", "ref_harness")
            if os.path.exists(ref):     # informational: the real reference on the int16 stand-in of the same shape
                try:
                    with tempfile.NamedTemporaryFile(suffix=".bin", delete=False) as f:
                        synth.iq_int(4 << 20, c["Fs"], [(8192, 103e3, 0.0), (4096, 99e3, 0.5)], 64, 1, np.int16).tofile(f)
                    out = subprocess.run([ref, "time", "s16", f.name, str(bs), repr(c["Fs"]), repr(c["Fc"]), repr(c["Ff"]),
                                          repr(c["width"]), str(c["order"]), "1", repr(c["oFs"]), "1", "2.0"],
                                         capture_output=True, text=True, timeout=120).stdout
                    os.unlink(f.name)
                    line["cpu_baseline"]["reference_int16_standin_msamples_per_s"] = json.loads(out)["msamples_per_s"]
                except Exception as e:  # pragma: no cover
                    line["cpu_baseline"]["reference_int16_standin_error"] = str(e)[:100]
        emit_line(out_fd, line)
    if win is not None:
        barrier()
        win.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

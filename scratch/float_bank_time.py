"""Float channel bank vs a loop of C IQBaseBand<float> + FMDemod chains (run with PYTHONPATH=.).

C4 / C5 parameters with complex float input: 100 MS/s, 15 taps, width 25 kHz, ss 2083 (oFs 48 kHz), 2^27
device-resident samples (1 GiB, larger than L2), FM output.  Bank and loop alternate inside one command; the
median of the timed passes is reported.  The bank's kernel times come from a torch.profiler pass of their own.
Bound of bank_fold_f32_kernel (DESIGN §4.7b): shared-memory wavefronts, 4.5 per warp and sample (A and U 2 each,
x 0.5), one per SM clock.  Spot channels of bank and loop are compared at the timed size (<= 1e-5).
Prints one JSON line; `--out PATH` also writes it to PATH."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

from libsdr_b200 import synth
from libsdr_b200.nodes import DEMOD_FM, ChannelBank, IQBaseBand, RxChain

N = 1 << 27
BS = 1 << 20
PASSES = int(os.environ.get("PASSES", "5"))
SMS = torch.cuda.get_device_properties(0).multi_processor_count


def smi():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True).stdout.strip().split(", ")
    return dict(card=q[0], power_limit_w=float(q[1]), max_sm_clock_mhz=float(q[2]))


def rel_rms(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.sqrt(np.mean((a - b) ** 2)) / np.sqrt(np.mean(b ** 2)))


def event_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def workload(C, x, info):
    cfg = synth.C4 if C == 256 else synth.C5
    Fs = cfg["Fs"]
    Fc = synth.bank_frequencies(C, Fs)
    bank = ChannelBank("f32", Fc, None, cfg["width"], cfg["order"], cfg["sub_sample"], cfg["oFs"])
    bank.config(sample_rate=Fs, buffer_size=BS)
    n_out = bank.outputs_for(N)
    fm = {"fm": torch.zeros((C, n_out + 8), dtype=torch.float32, device="cuda")}    # later calls may complete one more window
    nodes = []
    for c in range(C):
        nd = IQBaseBand("f32", Fc[c], Fc[c], cfg["width"], cfg["order"], cfg["sub_sample"], cfg["oFs"])
        nd.config(sample_rate=Fs, buffer_size=BS)
        nodes.append((nd, RxChain(nd, DEMOD_FM)))
    bb_out = torch.empty((n_out + 8, 2), dtype=torch.float32, device="cuda")
    au_out = torch.empty(n_out + 8, dtype=torch.float32, device="cuda")

    def run_bank():
        bank.process(x, BS, want=("fm",), out=fm)

    def run_loop():
        for nd, ch in nodes:
            ch.process(x, BS, bb_out=bb_out, audio_out=au_out)

    run_bank(); run_loop(); torch.cuda.synchronize()       # warm-up (the streams carry on: same work per pass)
    tb, tl = [], []
    for _ in range(PASSES):
        tb.append(event_ms(run_bank))
        tl.append(event_ms(run_loop))
    tb, tl = float(np.median(tb)), float(np.median(tl))

    # kernel times of one bank pass
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        run_bank(); torch.cuda.synchronize()
    k_acc = k_fin = 0.0
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / 1e3
        if "bank_fold_f32_kernel" in ev.key:
            k_acc += t
        elif "bank_finalize_kernel" in ev.key:
            k_fin += t

    # spot channels: fresh bank and chains over the same input, FM compared without the buffer-first elements
    spot = [0, 1, C // 2 - 1, C // 2, C // 2 + 1, C - 1]
    bank2 = ChannelBank("f32", Fc, None, cfg["width"], cfg["order"], cfg["sub_sample"], cfg["oFs"])
    bank2.config(sample_rate=Fs, buffer_size=BS)
    fm2 = bank2.process(x, BS, want=("fm",))["fm"]
    assert fm2.shape[1] == n_out
    errs = []
    for c in spot:
        nd = IQBaseBand("f32", Fc[c], Fc[c], cfg["width"], cfg["order"], cfg["sub_sample"], cfg["oFs"])
        nd.config(sample_rate=Fs, buffer_size=BS)
        _, ya, counts = RxChain(nd, DEMOD_FM).process(x, BS)
        first = np.concatenate([[0], np.cumsum(counts)[:-1]])[counts > 0]
        mask = np.ones(n_out, dtype=bool); mask[first] = False
        errs.append(rel_rms(fm2[c].cpu().numpy()[mask], ya.cpu().numpy()[mask]))

    cs = C * N
    clk = info["max_sm_clock_mhz"] * 1e6
    bound_ms = (C / 32) * N * 4.5 / (SMS * clk) * 1e3
    return dict(channels=C, samples=N, bank_ms=round(tb, 3), loop_ms=round(tl, 3),
                bank_cs_per_s=cs / tb * 1e3, loop_cs_per_s=cs / tl * 1e3, ratio=round(tl / tb, 3),
                bank_accum_kernel_ms=round(k_acc, 3), bank_finalize_kernel_ms=round(k_fin, 3),
                smem_bound_ms_at_max_clock=round(bound_ms, 3), share_of_smem_bound=round(bound_ms / k_acc, 3) if k_acc else None,
                spot_channels=spot, spot_fm_rel_rms_max=max(errs))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    info = smi()
    g = torch.Generator(device="cuda").manual_seed(5)
    x = (torch.randn((N, 2), device="cuda", generator=g) * 0.05).contiguous()
    # a carrier in each spot channel of both grids, 2 kHz above its centre, so that the spot comparison is well conditioned
    t = torch.arange(N, device="cuda", dtype=torch.float64) / 100e6
    for grid in (256, 2048):
        for c in (0, 1, grid // 2 - 1, grid // 2, grid // 2 + 1, grid - 1):
            ph = 2 * np.pi * ((c - grid // 2) * (100e6 / grid) + 2e3) * t
            x[:, 0] += (0.05 * torch.cos(ph)).float(); x[:, 1] += (0.05 * torch.sin(ph)).float()
    del t
    torch.cuda.synchronize()
    res = dict(info, sms=SMS, workloads=[workload(C, x, info) for C in (256, 2048)])
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    ok = all(w["spot_fm_rel_rms_max"] <= 1e-5 for w in res["workloads"])
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()

"""FFTPlan<float>, FFTPlan<double> and FilterNode on every kernel path they dispatch to, at the shapes where the grid,
chunk and stride logic of each path takes effect, with ELEMENT-WISE bounds against float64 references.

A whole-array relative RMS hides localized defects (one grid-stride iteration, one row at a chunk boundary, the block
after a call boundary): one 4096-sample block off by 1e-4 in a 16 Mi-sample output moves it by 1.6e-6.  So every case
here also checks, per row or per output block,

  FFT (float, per row):       max_k |X^_k - X_k| <= K_FFT * log2(M) * 2^-24 * s_row
  FFT (double, per row):      max_k |X^_k - X_k| <= K_F64 * log2(M) * 2^-53 * s_row
  filter (per output block):  max   |y^ - y|     <= K_FLT * log2(2N) * 2^-24 * rms(x over [block b-1 | block b])

M is the power of two actually transformed (n, or Bluestein's M); s_row = max(||x_row||_2, max_k |X_k|).  ||x_row||_2
is the typical size of an output element, and for noise-like rows max|X| is only a few times larger; but a spectrum
concentrated in one bin (a pure tone, |X_m| = n = sqrt(n) ||x||_2) carries rounding errors at the scale of that peak:
measured against ||x||_2 alone, a tone through the four-step at n = 2^21 is 218x the unit, which no single K could
allow without making the bound useless for every other row.  The filter form uses ||h_eff||_2 = 1/sqrt(2N), the
reference's normalisation (taps divided by the l2 norm of their 2N-point spectrum).  One constant per family for every
case, so a path several times less accurate than its siblings fails instead of getting its own tolerance.  Each K is
at least 4x the largest ratio observed over all cases of its family (NVIDIA B200, 148 SMs, 1000 W power limit):

  family   observed max ratio (case)                                      next largest                        K
  fft      1.95 (forward -> backward, n = 2; 2 = log2(M) makes it coarse)  1.31 (fwd->bwd n = 32)              8
  fft64    0.77 (Bluestein n = 2^22 - 1, backward)                         0.72 (n = 2^20 batch 33, backward)  4
  filter   1.64 (block 1: the 2-point transform, log2(2N) = 1)             0.81 (block 2)                      8

Large paths sit well inside: four-step 2^21 .. 2^24 <= 0.50, Bluestein (M = 2^25 and the chunked batch) <= 0.56,
filter blocks >= 16 (banks, conv8k, GeneralOla, the 2 GiB fallback) <= 0.42.

References: np.fft in complex128 for small shapes, torch.fft in complex128 on the device (cuFFT in double,
independent of the library's kernels) for large ones; the filter's full linear convolution in complex128 through
torch.fft (checked once against the oracle's time-domain convolution), and per output block the exact float64
np.convolve of the 2N input samples block b depends on (spot checks: first, last, grid / chunk / call boundaries,
seeded random blocks).  Device outputs are pre-filled with NaN wherever a test allocates them, so a skipped row or
block cannot pass on stale memory.

Path probe: each case asserts the launch count (sdrg_kernel_launch_count deltas) its intended path implies, so that a
later dispatch change cannot silently drop coverage.  The resident grid of fft8k_kernel / conv8k_kernel is 2 CTAs per
SM, 296 on a B200.

  path (gap)                        kernel(s)                                  case(s)                               launches
  fft8k grid-stride, 8192 (1)       fft8k_kernel<SPLIT>                        pow2 n=8192 batch 2049, in place       1
  fft8k paired 4096, odd batch (1)  fft8k_kernel<!SPLIT>                       pow2 n=4096 batch 4097, in place       1
  radix-16 plain FFT                fft_batch_r16_kernel                       n=256..2048, batch % per-CTA != 0      1
  small plain FFT                   fft_batch_kernel                           n=2..128                               1
  four-step, large sub-plans (2)    transpose_tw_kernel x3 + 2 sub-plans       n=2^21..2^24, batches 1,3,2 (grow);    3 + 1 + 1
                                    (fft8k_kernel inside at 2^23, 2^24)        sub-batches up to 12288
  Bluestein M=2^25 (2)              pre, mul, post + 2 four-step M-plans       n=2^23+1, 2^24-1                       3 + 2*5
  Bluestein chunk loop (3)          the same, per 1 GiB chunk                  n=100003 batch 513 (per=512)           2 * (3 + 2*5)
  in place, float plan (5)          every float path above                     pow2 in place via sdrg_fft_exec_dev    as above
  structured inputs                 fft_batch_kernel, r16, fft8k, 4-step, Bl.  impulses, tones, real input            as above
  FFTPlan<double> (4)               radix2_stage_f64 (+ Bluestein kernels)     n=2^20 batch 33, 2^22, 2^22-1          chunks*log2 M; 3 + 2*23
  Fft64 chunk loop (3)              the same, per 512 MiB chunk                n=2^20 batch 33 (per=32)               2 * 20
  sdrg_fft64_exec_dev (4)           the same                                   == host entry point, bit for bit       as above
  tiny blocks (8)                   filter_ola_kernel                          blocks 1..128, one filter              1
  single filter, r16                filter_ola1_r16_kernel<0>                  out_stride / add cases (1 filter rows)  1
  bank, small blocks (6)            filter_ola_kernel (filter loop)            blocks 16, 64, 128, 3 filters          1
  bank, radix-16 (6)                filter_ola1_r16_kernel<1>, <2>             blocks 256, 512, 2048, 3 filters       2
  bank, 2 GiB spectrum fallback (6) filter_ola_kernel                          block 1024, 2 filters, 2^27+3089 smp   1 (2 below)
  bank, block 4096 (6)              conv8k_kernel<true>                        4 filters, 4096 blocks, ragged calls   1 per call
  single node, block 4096           conv8k_kernel<false>                       bank cross-check                       1
  GeneralOla chunk loop (3)         gather, 4-step, mul, crop, roll            block 5000, 3 filters, 4097 blocks     2*(1+5+3*7)+1
  out_stride (7)                    every bank kernel above + GeneralOla       blocks 64, 1024, 4096, 5000, NaN gaps  1, 2, 1, 28
  no filters, add mid-stream (9)    filter_ola_kernel / GeneralOla w/o filter  blocks 64, 1024, 4096, 5000            1, 1, 1, 7
  ... then addFilter x2, x1         the bank kernel of the block size          == a node with the filters from start  1, 2, 1, 21 / 28

(Gap 10, the metric, is this file's element-wise bound.)  On one B200 the file takes about 80 s, about 64 s of it in the
two M = 2^25 Bluestein cases, and at most about 8 GB of device memory above its start; tensors are freed between
cases.
"""
import gc
import math
import time
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import rel_rms
from libsdr_b200 import _lib
from libsdr_b200.nodes import FFTPlan, FFTPlan64, FilterNode
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

EPS32, EPS64 = 2.0 ** -24, 2.0 ** -53
K_FFT = 8
K_F64 = 4
K_FLT = 8
RMS_FFT, RMS_FLT, RMS_F64 = 1e-5, 1e-5, 1e-12

FS = 2.4e6
BANDS3 = [(100e3, 300e3), (-200e3, -700e3), (-1.0e6, 1.1e6)]      # the second has fmax < fmin (addFilter swaps)
BANDS4 = [(100e3, 200e3), (-500e3, -300e3), (1e6, 800e3), (-1.2e6, 1.2e6)]

_OBS = {"fft": (0.0, ""), "fft64": (0.0, ""), "filter": (0.0, "")}
_MEM = {"base": 0, "peak": 0}
_ALL = []


# ---- bookkeeping ---------------------------------------------------------------------------------------------------------
def _used():
    free, total = torch.cuda.mem_get_info()
    return total - free


def _note_mem():
    _MEM["peak"] = max(_MEM["peak"], _used() - _MEM["base"])


def _record(family, label, ratio):
    if ratio > _OBS[family][0] or not math.isfinite(ratio):
        _OBS[family] = (ratio, label)
    _ALL.append((family, ratio, label))
    _note_mem()


@pytest.fixture(scope="module", autouse=True)
def _report():
    torch.cuda.init()
    torch.cuda.synchronize()
    _MEM["base"] = _used()
    t0 = time.time()
    yield
    print("\n[fft paths] wall %.1f s, peak device memory above the start about %.2f GB"
          % (time.time() - t0, _MEM["peak"] / 1e9))
    for fam, (r, lab) in _OBS.items():
        print("[fft paths] %-6s max ratio %.4g  (%s)" % (fam, r, lab))
    for fam, r, lab in sorted(_ALL, key=lambda e: (e[0], -e[1])):
        print("[fft paths]   %-6s %8.4f  %s" % (fam, r, lab))


@pytest.fixture(autouse=True)
def _free_between_cases():
    yield
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


# ---- device helpers -----------------------------------------------------------------------------------------------------
def _ptr(t):
    return C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _nan_like(shape, dtype=torch.complex64):
    t = torch.empty(shape, dtype=dtype, device="cuda")
    torch.view_as_real(t).fill_(float("nan"))
    return t


def _randn(shape, seed, dtype=torch.complex64):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return torch.randn(shape, dtype=dtype, device="cuda", generator=g)


def _launches_of(fn):
    n0 = _lib.kernel_launch_count()
    r = fn()
    torch.cuda.synchronize()
    return r, _lib.kernel_launch_count() - n0


def fft_exec(plan, x, out=None):
    """sdrg_fft_exec_dev on a (batch, n) complex64 tensor; `out` defaults to a NaN-filled tensor (pass x for in place).
    Returns (out, launches)."""
    if out is None:
        out = _nan_like(x.shape)
    _, k = _launches_of(lambda: _lib.call("sdrg_fft_exec_dev", plan._h, _ptr(x), _ptr(out), x.shape[0], _stream()))
    return out, k


def fft64_exec(plan, x):
    out = _nan_like(x.shape, torch.complex128)
    _, k = _launches_of(lambda: _lib.call("sdrg_fft64_exec_dev", plan._h, _ptr(x), _ptr(out), x.shape[0], _stream()))
    return out, k


def fft_ref(x, inverse=False):
    """Unnormalised DFT of the rows of x in complex128: np.fft on the host for small shapes, torch.fft (cuFFT in
    double) on the device for large ones.  Returns a complex128 device tensor."""
    if x.numel() <= (1 << 20):
        a = x.cpu().numpy().astype(np.complex128)
        r = np.fft.ifft(a, axis=-1, norm="forward") if inverse else np.fft.fft(a, axis=-1)
        return torch.from_numpy(r).cuda()
    a = x.to(torch.complex128)
    return torch.fft.ifft(a, dim=-1, norm="forward") if inverse else torch.fft.fft(a, dim=-1)


def _rel_rms_t(a, b):
    a = a.to(torch.complex128); b = b.to(torch.complex128)
    den = torch.sqrt(torch.mean(b.abs() ** 2)).item()
    return torch.sqrt(torch.mean((a - b).abs() ** 2)).item() / (den if den > 0 else 1.0)


def row_scale(x_in, X):
    """s_row = max(||x_row||_2, max_k |X_k|) in float64 (x_in: what the transform was applied to, X: its spectrum)."""
    return torch.maximum(torch.linalg.vector_norm(x_in.to(torch.complex128), dim=-1), X.to(torch.complex128).abs().amax(dim=-1))


def check_fft(got, ref, x_in, M, label, family="fft", rms_tol=None):
    """Per row: max|got - ref| <= K log2(M) eps s_row, plus the relative RMS over the whole array.  Returns the largest
    ratio err / (log2(M) eps s_row)."""
    got, ref, x_in = got.reshape(-1, got.shape[-1]), ref.reshape(-1, ref.shape[-1]), x_in.reshape(-1, x_in.shape[-1])
    eps, K = (EPS64, K_F64) if family == "fft64" else (EPS32, K_FFT)
    assert bool(torch.isfinite(torch.view_as_real(got)).all()), "%s: non-finite output (a row was never written?)" % label
    err = (got.to(torch.complex128) - ref).abs().amax(dim=-1)
    per_row = err / (math.log2(M) * eps * row_scale(x_in, ref))
    ratio = per_row.max().item()
    _record(family, label, ratio)
    assert ratio <= K, "%s: element-wise error %.3g x the unit bound in row %d (K = %g)" % (
        label, ratio, int(per_row.argmax()), K)
    rr = _rel_rms_t(got, ref)
    assert rr < (rms_tol or (RMS_F64 if family == "fft64" else RMS_FFT)), (label, rr)
    return ratio


# ---- filter references -------------------------------------------------------------------------------------------------
def taps_of(block, band):
    lo, hi = min(band), max(band)                  # FilterNode::addFilter swaps fmax < fmin (filternode.hh:264)
    return orc.filter_taps(block, lo, hi, FS)


def _h_eff(taps):
    h = taps.astype(np.complex128)
    return h / (np.sqrt(2 * h.shape[0]) * np.sqrt(np.sum(np.abs(h) ** 2)))


class FilterRef:
    """Causal linear convolution y[n] = sum_j h_eff[j] x[n - j] of a whole stream (from its start, zero history) in
    complex128 through torch.fft; the input's spectrum is shared by the filters."""

    def __init__(self, x):
        self.n = x.numel()
        self.x = x

    def __call__(self, taps):
        N = taps.shape[0]
        nfft = 1 << (self.n + N - 2).bit_length()
        if getattr(self, "_nfft", None) != nfft:
            self._X = torch.fft.fft(self.x.to(torch.complex128), nfft)
            self._nfft = nfft
        H = torch.fft.fft(torch.from_numpy(_h_eff(taps)).cuda(), nfft)
        return torch.fft.ifft(self._X * H)[:self.n]


def block_direct(x, taps, b):
    """Output block b computed exactly in float64 from the 2N input samples it depends on (blocks b-1 and b)."""
    N = taps.shape[0]
    seg = x[max(b - 1, 0) * N:(b + 1) * N].cpu().numpy().astype(np.complex128)
    if b == 0:
        seg = np.concatenate([np.zeros(N, np.complex128), seg])
    return np.convolve(seg, _h_eff(taps))[N:2 * N], np.sqrt(np.mean(np.abs(seg) ** 2))


def _seg_rms(x, N, b0, nb):
    """rms over [block b-1 | block b] of the stream x for blocks b0 .. b0+nb-1 (zeros before the stream's start)."""
    lo = max(b0 - 1, 0)
    p = (x[lo * N:(b0 + nb) * N].to(torch.complex128).abs() ** 2).view(-1, N).mean(dim=1)
    if b0 == 0:
        p = torch.cat([torch.zeros(1, dtype=p.dtype, device=p.device), p])
    return torch.sqrt((p[:-1] + p[1:]) / 2)


def check_filter_blocks(y, ref, x, N, label, b0=0, rms=True):
    """Per output block: max|y - ref| <= K_FLT log2(2N) 2^-24 rms(x over [b-1 | b]); y / ref cover the blocks
    b0, b0+1, ... of the stream x (x from its start)."""
    assert y.numel() % N == 0
    nb = y.numel() // N
    assert bool(torch.isfinite(torch.view_as_real(y)).all()), "%s: non-finite output" % label
    err = (y.to(torch.complex128) - ref).abs().view(nb, N).amax(dim=1)
    per_blk = err / (math.log2(2 * N) * EPS32 * _seg_rms(x, N, b0, nb))
    ratio = per_blk.max().item()
    _record("filter", label, ratio)
    assert ratio <= K_FLT, "%s: block %d off by %.3g x the unit bound (K = %g)" % (label, b0 + int(per_blk.argmax()), ratio, K_FLT)
    if rms:
        rr = _rel_rms_t(y, ref)
        assert rr < RMS_FLT, (label, rr)
    return ratio


def check_spot_blocks(y, x, taps, blocks, label, b0=0):
    """y holds blocks b0, b0+1, ... of the filtered stream x; each listed block against its exact float64 value."""
    N = taps.shape[0]
    for b in sorted(set(blocks)):
        want, seg_rms = block_direct(x, taps, b)
        got = y[(b - b0) * N:(b - b0 + 1) * N].cpu().numpy().astype(np.complex128)
        assert np.isfinite(got).all(), (label, b)
        ratio = float(np.max(np.abs(got - want))) / (math.log2(2 * N) * EPS32 * seg_rms)
        _record("filter", "%s spot %d" % (label, b), ratio)
        assert ratio <= K_FLT, "%s: spot block %d off by %.3g x the unit bound" % (label, b, ratio)


def spot_blocks(nblk, around=(), k=4, seed=0):
    s = {0, nblk - 1}
    for b in around:
        s.update(c for c in (b - 1, b, b + 1) if 0 <= c < nblk)
    s.update(int(v) for v in np.random.default_rng(seed).integers(0, nblk, k))
    return sorted(s)


def make_node(block, bands):
    f = FilterNode(block)
    for lo, hi in bands:
        f.addFilter(lo, hi)
    f.config(sample_rate=FS, buffer_size=block)
    return f


def filter_exec(node, x, n_filters, pad=0):
    """sdrg_filter_process_dev into a NaN-filled (n_filters, n_out + pad) tensor; returns (out, n_out, launches)."""
    n_out = node.outputs_for(x.numel())
    stride = n_out + pad
    out = _nan_like((max(n_filters, 1), max(stride, 1)))
    got = C.c_size_t(0)
    _, k = _launches_of(lambda: _lib.call("sdrg_filter_process_dev", node._h, _ptr(x), x.numel(), _ptr(out), stride,
                                          C.byref(got), _stream()))
    assert got.value == n_out
    return out, n_out, k


def general_ola_launches(n_blocks, n_filters, M):
    """GeneralOla::run: per chunk of per = 2^29 / (8 M) blocks: gather + forward M-plan + per filter (multiply +
    inverse M-plan + crop); then one roll.  An M-point plan above 8192 is the four-step: 3 transposes + 2 sub-plans."""
    if n_blocks == 0:
        return 0
    plan = 1 if M <= 8192 else 5
    per = max(1, min(n_blocks, 65535, (1 << 29) // (M * 8)))
    chunks = -(-n_blocks // per)
    return chunks * (1 + plan + n_filters * (2 + plan)) + 1


# ==== FFTPlan<float> ======================================================================================================
# batches: odd, above the resident grid of fft8k_kernel (4096: 2049 items of two transforms; 8192: 2049 items), and
# not multiples of the transforms per CTA of fft_batch_r16_kernel (256/16 = 16 at n = 256 ... 1 at 4096)
POW2_BATCH = {2: 131073, 4: 65537, 8: 32769, 16: 16385, 32: 8193, 64: 4097, 128: 2049,
              256: 16 * 257 + 7, 512: 8 * 257 + 3, 1024: 4 * 257 + 1, 2048: 2 * 1024 + 1, 4096: 4097, 8192: 2049}


@pytest.mark.parametrize("n", sorted(POW2_BATCH))
def test_fft_pow2_batches_over_the_grid(n):
    """Forward, backward and forward -> backward = n x, one launch each (the shared-memory kernel of the size)."""
    batch = POW2_BATCH[n]
    x = _randn((batch, n), seed=n)
    fwd, bwd = FFTPlan(n, FFTPlan.FORWARD), FFTPlan(n, FFTPlan.BACKWARD)
    X, k = fft_exec(fwd, x)
    assert k == 1                                   # fft_batch_kernel / fft_batch_r16_kernel / fft8k_kernel
    check_fft(X, fft_ref(x), x, n, "pow2 fwd n=%d" % n)
    Y, k = fft_exec(bwd, x)
    assert k == 1
    check_fft(Y, fft_ref(x, inverse=True), x, n, "pow2 bwd n=%d" % n)
    Z, k = fft_exec(bwd, X)
    assert k == 1
    check_fft(Z, x.to(torch.complex128) * n, X, n, "pow2 fwd->bwd n=%d" % n)


@pytest.mark.parametrize("n", sorted(POW2_BATCH))
def test_fft_pow2_in_place(n):
    """Pow2Fft::exec documents in == out (Bluestein and GeneralOla rely on it): the same batches with d_in == d_out."""
    batch = POW2_BATCH[n]
    x = _randn((batch, n), seed=1000 + n)
    for direction, inverse in ((FFTPlan.FORWARD, False), (FFTPlan.BACKWARD, True)):
        buf = x.clone()
        _, k = fft_exec(FFTPlan(n, direction), buf, out=buf)
        assert k == 1
        check_fft(buf, fft_ref(x, inverse), x, n, "pow2 in place %s n=%d" % ("bwd" if inverse else "fwd", n))


@pytest.mark.parametrize("log2n", [21, 22, 23, 24])
def test_fft_four_step_large_sub_plans(log2n):
    """n = 2^21 .. 2^24: sub-plans of 1024/2048 .. 4096 x 4096 points, fft8k_kernel inside the decomposition with
    sub-batches in the thousands.  One plan object is called with batches 1, 3, 2 (its scratch grows at 3)."""
    n = 1 << log2n
    x = _randn((3, n), seed=log2n)
    ref = fft_ref(x)
    fwd = FFTPlan(n, FFTPlan.FORWARD)
    for b in (1, 3, 2):
        X, k = fft_exec(fwd, x[:b])
        assert k == 3 + 1 + 1                       # transpose, sub-plan n1, transpose+twiddle, sub-plan n2, transpose
        check_fft(X, ref[:b], x[:b], n, "four-step fwd n=2^%d batch %d" % (log2n, b))
        del X
    del fwd
    bwd = FFTPlan(n, FFTPlan.BACKWARD)
    Y, k = fft_exec(bwd, x)
    assert k == 5
    check_fft(Y, fft_ref(x, inverse=True), x, n, "four-step bwd n=2^%d" % log2n)
    del Y
    X = ref.to(torch.complex64)
    Z, k = fft_exec(bwd, X)
    check_fft(Z, x.to(torch.complex128) * n, X, n, "four-step fwd->bwd n=2^%d" % log2n)


@pytest.mark.parametrize("n", [(1 << 23) + 1, (1 << 24) - 1])
def test_fft_bluestein_m_2_25(n):
    """Bluestein with M = 2^25 (the four-step engine at 4096 x 8192 underneath)."""
    M = 1 << 25
    x = _randn((1, n), seed=n % 1000)
    for direction, inverse in ((FFTPlan.FORWARD, False), (FFTPlan.BACKWARD, True)):
        X, k = fft_exec(FFTPlan(n, direction), x)
        assert k == 3 + 2 * 5                       # pre, mul, post + forward and inverse M-point four-step (5 each)
        check_fft(X, fft_ref(x, inverse), x, M, "bluestein n=%d %s" % (n, "bwd" if inverse else "fwd"))
        del X


def test_fft_bluestein_chunk_loop():
    """n = 100003 (M = 2^18), batch 513: AnyFft::exec cuts Bluestein batches at 1 GiB of scratch, per = 2^30 / (8 M)
    = 512, so the second chunk holds one row.  Every row by Parseval in float64, rows 0, 511, 512 and the last one
    element-wise."""
    n, M, batch = 100003, 1 << 18, 513
    x = _randn((batch, n), seed=3)
    X, k = fft_exec(FFTPlan(n, FFTPlan.FORWARD), x)
    assert k == 2 * (3 + 2 * 5)                     # 2 chunks x (pre, mul, post + 2 four-step plans of 2^18 = 512 x 512)
    e_out = (X.to(torch.complex128).abs() ** 2).sum(dim=1)
    e_in = n * (x.to(torch.complex128).abs() ** 2).sum(dim=1)
    dev = (e_out - e_in).abs() / e_in
    # ||X^ - X||_2 <= sqrt(n) K log2(M) 2^-24 s_row by the element-wise bound, and ||X||_2 = sqrt(n) ||x||_2, so
    # | ||X^||^2 - ||X||^2 | / ||X||^2 <= 2 u + u^2 with u = K log2(M) 2^-24 s_row / ||x||_2
    u = K_FFT * math.log2(M) * EPS32 * row_scale(x, X) / torch.linalg.vector_norm(x.to(torch.complex128), dim=-1)
    assert bool((dev <= 2 * u + u * u).all()), (int(dev.argmax()), dev.max().item())
    rows = [0, 511, 512, batch - 1]
    check_fft(X[rows], fft_ref(x[rows]), x[rows], M, "bluestein chunked rows 0/511/512/last")


STRUCT_N = [8, 256, 4096, 8192, 1 << 21, 100003]


@pytest.mark.parametrize("n", STRUCT_N)
def test_fft_structured_inputs(n):
    """Unit impulses at 0, 1 and n-1 (exp(-2 pi i k p / n) in every bin), tones on bins 1, n/2, n-1 (n delta) and a
    real input (Hermitian spectrum), in one batch of 7 rows (odd: the paired 4096-point form's last item is alone)."""
    M = n if n & (n - 1) == 0 else 1 << (2 * n - 2).bit_length()
    j = np.arange(n)
    rows = []
    for p in (0, 1, n - 1):
        r = np.zeros(n, np.complex64); r[p] = 1; rows.append(r)
    tones = (1, n // 2, n - 1)
    for m in tones:
        rows.append(np.exp(2j * np.pi * ((j * m) % n) / n).astype(np.complex64))
    rows.append(np.random.default_rng(n).standard_normal(n).astype(np.complex64))
    xh = np.stack(rows)
    x = torch.from_numpy(xh).cuda()
    X, _ = fft_exec(FFTPlan(n, FFTPlan.FORWARD), x)
    k = np.arange(n)
    exact = np.stack([np.exp(-2j * np.pi * ((k * p) % n) / n) for p in (0, 1, n - 1)])
    check_fft(X[:3], torch.from_numpy(exact).cuda(), x[:3], M, "impulses n=%d" % n)
    check_fft(X[3:], fft_ref(x[3:]), x[3:], M, "tones+real n=%d" % n)
    Xt = X[3:6].to(torch.complex128)
    for i, m in enumerate(tones):
        assert int(Xt[i].abs().argmax()) == m
        assert abs(Xt[i, m].item() - n) <= K_FFT * math.log2(M) * EPS32 * n
    Xr = X[6].to(torch.complex128)
    mirror = torch.roll(torch.flip(Xr, [0]), 1).conj()            # conj(X[(n - k) mod n])
    herm = (Xr - mirror).abs().max().item() / (math.log2(M) * EPS32 * row_scale(x[6:7], X[6:7]).item())
    _record("fft", "hermitian n=%d (/2)" % n, herm / 2)
    assert herm <= 2 * K_FFT, herm


# ==== FFTPlan<double> =====================================================================================================
@pytest.mark.parametrize("n,batch", [(1 << 20, 33), (1 << 22, 1), ((1 << 22) - 1, 1)])
def test_fft64_large_chunked_and_device_entry(n, batch):
    """Fft64 up to its 2^22 limit; n = 2^20 with batch 33 > per = 2^29 / (16 M) = 32 runs two chunks.  The device
    entry point (sdrg_fft64_exec_dev) equals the host one bit for bit on the same input."""
    M = n if n & (n - 1) == 0 else 1 << (2 * n - 2).bit_length()
    L = M.bit_length() - 1
    per = max(1, min(batch, 65535, (1 << 29) // (M * 16)))
    chunks = -(-batch // per)
    want = chunks * (L if M == n else 3 + 2 * L)    # log2 M radix-2 passes per chunk (Bluestein: pre, mul, post + 2 plans)
    if n == 1 << 20:
        assert chunks == 2
    x = _randn((batch, n), seed=n % 997, dtype=torch.complex128)
    for direction, inverse in ((FFTPlan64.FORWARD, False), (FFTPlan64.BACKWARD, True)):
        plan = FFTPlan64(n, direction)
        host = plan(x.cpu().numpy())
        X, k = fft64_exec(plan, x)
        assert k == want, (k, want)
        assert np.array_equal(X.cpu().numpy(), host)
        ref = torch.fft.ifft(x, dim=-1, norm="forward") if inverse else torch.fft.fft(x, dim=-1)
        check_fft(X, ref, x, M, "fft64 n=%d batch %d %s" % (n, batch, "bwd" if inverse else "fwd"), family="fft64")
        del X, ref, host, plan


# ==== FilterNode ==========================================================================================================
def test_filter_reference_matches_time_domain():
    """The complex128 torch.fft convolution used below equals the oracle's time-domain convolution."""
    N = 4096
    x = _randn(9 * N + 5, seed=11)
    ref = FilterRef(x)
    for band in BANDS4:
        t = taps_of(N, band)
        td = orc.filter_timedomain_f64(t, x[:8 * N].cpu().numpy())
        assert np.max(np.abs(ref(t)[:8 * N].cpu().numpy() - td)) <= 1e-12 * np.max(np.abs(td))
        want, _ = block_direct(x, t, 5)
        assert np.max(np.abs(want - td[5 * N:6 * N])) <= 1e-12 * np.max(np.abs(td))
    xs = _randn((1, 1 << 21), seed=12)             # fft_ref's device branch (cuFFT in double) against np.fft
    assert rel_rms(fft_ref(xs).cpu().numpy(), np.fft.fft(xs.cpu().numpy().astype(np.complex128))) < 1e-14


@pytest.mark.parametrize("block", [1, 2, 4, 8, 16, 32, 64, 128])
def test_filter_tiny_blocks(block):
    """Blocks 1 .. 128 (FFT sizes 2 .. 256, filter_ola_kernel), one filter, two calls, against the float64 time-domain
    convolution of the reference's taps.  Block 1: the reference's window at i = 0 is 0.42 - 0.5 + 0.08, which in double
    is -5.55e-17, not 0, so its one tap is a tiny negative number and the normalised filter is y = -x / sqrt(2)."""
    band = (100e3, 300e3)
    nblk = 600
    x = _randn(nblk * block + block // 2, seed=block)
    f = make_node(block, [band])
    t = taps_of(block, band)
    np.testing.assert_array_equal(f.design(0)[1], t)
    cut = (nblk // 3) * block + (block + 1) // 2
    y1, _, k1 = filter_exec(f, x[:cut], 1)
    y2, _, k2 = filter_exec(f, x[cut:], 1)
    assert k1 == 1 and k2 == 1                      # filter_ola_kernel
    y = torch.cat([y1[0, :cut // block * block], y2[0, :nblk * block - cut // block * block]])
    assert y.numel() == nblk * block
    ref = torch.from_numpy(orc.filter_timedomain_f64(t, x.cpu().numpy())[:nblk * block]).cuda()
    check_filter_blocks(y, ref, x, block, "tiny block %d" % block)
    if block == 1:
        check_filter_blocks(y, x[:nblk].to(torch.complex128) * -math.sqrt(0.5), x, 1, "block 1 = -x/sqrt2")


@pytest.mark.parametrize("block,launches", [(16, 1), (64, 1), (128, 1), (256, 2), (512, 2), (2048, 2)])
def test_filter_bank_paths(block, launches):
    """Three filters (one given with fmax < fmin): blocks <= 128 loop the filters inside filter_ola_kernel, blocks
    256 .. 2048 run the radix-16 bank (forward pass <1>, then one CTA per (block, filter) <2>)."""
    nblk = 2500 if block <= 512 else 700
    x = _randn(nblk * block + 3, seed=block + 7)
    f = make_node(block, BANDS3)
    cut = 777 * block // 2 + 5
    y1, n1, k1 = filter_exec(f, x[:cut], 3)
    y2, n2, k2 = filter_exec(f, x[cut:], 3)
    assert (k1, k2) == (launches, launches)
    y = torch.cat([y1[:, :n1], y2[:, :n2]], dim=1)
    ref = FilterRef(x[:nblk * block])
    for i, band in enumerate(BANDS3):
        t = taps_of(block, band)
        lab = "bank block %d filter %d" % (block, i)
        check_filter_blocks(y[i], ref(t), x, block, lab)
        check_spot_blocks(y[i], x, t, spot_blocks(nblk, around=(n1 // block,), seed=block + i), lab)


def test_filter_general_ola_chunk_loop():
    """Block 5000 (M = 16384): GeneralOla::run cuts at per = 2^29 / (8 M) = 4096 blocks; 4097 blocks in one call run two
    chunks, the next call continues from the rolled history."""
    N, M, F = 5000, 16384, 3
    nblk1, nblk2 = 4097, 3
    x = _randn((nblk1 + nblk2) * N + 1234, seed=5000)
    f = make_node(N, BANDS3)
    c1 = nblk1 * N + 17
    y1, n1, k1 = filter_exec(f, x[:c1], F)
    y2, n2, k2 = filter_exec(f, x[c1:], F)
    assert (n1, n2) == (nblk1 * N, nblk2 * N)
    assert k1 == general_ola_launches(nblk1, F, M) == 2 * (1 + 5 + 3 * 7) + 1
    assert k2 == general_ola_launches(nblk2, F, M)
    y = torch.cat([y1, y2], dim=1)
    del y1, y2
    ref = FilterRef(x[:(nblk1 + nblk2) * N])
    for i, band in enumerate(BANDS3):
        t = taps_of(N, band)
        lab = "general block 5000 filter %d" % i
        check_filter_blocks(y[i], ref(t), x, N, lab)
        check_spot_blocks(y[i], x, t, spot_blocks(nblk1 + nblk2, around=(4096, nblk1), seed=i), lab)


def test_filter_c3_bank_shape():
    """The bench's bank: block 4096, 4 filters, 16 x 2^20 samples = 4096 blocks, far above the 296-CTA grid, so each CTA
    reuses its 64 KB spectrum line for ~14 blocks.  One call and ragged calls (the pending-sample stitch), against the
    complex128 reference in full and per block; the bank equals 4 single-filter nodes (conv8k_kernel<false>)."""
    N, F = 4096, 4
    n = 16 << 20
    x = _randn(n, seed=4096)
    ref = FilterRef(x)
    refs = [ref(taps_of(N, b)) for b in BANDS4]
    del ref
    one, _, k = filter_exec(make_node(N, BANDS4), x, F)
    assert k == 1                                   # conv8k_kernel<true>
    cuts = [0, 3 * N + 1000, (1 << 23) + 12345, (1 << 23) + 300 * N + 7, n]
    fr = make_node(N, BANDS4)
    parts = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        yp, np_, k = filter_exec(fr, x[a:b], F)
        assert k == (1 if np_ else 0)
        parts.append(yp[:, :np_])
    rag = torch.cat(parts, dim=1)
    del parts
    grid_edges = [296 * i for i in range(1, 14)]
    call_edges = [c // N for c in cuts[1:-1]]
    for i, band in enumerate(BANDS4):
        t = taps_of(N, band)
        check_filter_blocks(one[i], refs[i], x, N, "c3 bank one call filter %d" % i)
        check_filter_blocks(rag[i], refs[i], x, N, "c3 bank ragged filter %d" % i)
        check_spot_blocks(one[i], x, t, spot_blocks(4096, around=grid_edges[:2] + [4095 - 296], seed=i), "c3 bank filter %d" % i)
        check_spot_blocks(rag[i], x, t, spot_blocks(4096, around=call_edges, seed=10 + i), "c3 ragged filter %d" % i)
        single, _, k = filter_exec(make_node(N, [band]), x, 1)
        assert k == 1                               # conv8k_kernel<false>
        check_filter_blocks(one[i], single[0], x, N, "c3 bank == single filter %d" % i)
        del single


def test_filter_bank_spectrum_fallback_over_2gib():
    """Block 1024, 2 filters: a call whose block spectra would exceed 2 GiB (2^27 + 3 * 1024 + 17 samples, 131075 blocks)
    falls back to filter_ola_kernel (1 launch); calls below the threshold run the radix-16 bank (2 launches).  Both
    give the same stream within the bound; spot blocks in float64."""
    N, F = 1024, 2
    bands = BANDS3[:2]
    n = (1 << 27) + 3 * N + 17
    nblk = n // N
    assert nblk * 2 * N * 8 > (2 << 30)
    x = _randn(n, seed=1024)
    big, n_out, k = filter_exec(make_node(N, bands), x, F)
    assert k == 1 and n_out == nblk * N             # filter_ola_kernel: spectrum scratch would be > 2 GiB
    taps = [taps_of(N, b) for b in bands]
    for i in range(F):
        check_spot_blocks(big[i], x, taps[i], spot_blocks(nblk, around=(1 << 16, 1 << 17), k=6, seed=i), "fallback filter %d" % i)
    small = make_node(N, bands)
    step = (1 << 24) + 333
    pos = 0
    for a in range(0, n, step):
        part, np_, k = filter_exec(small, x[a:a + step], F)
        assert k == (2 if np_ else 0)               # filter_ola1_r16_kernel<1>, <2>
        for i in range(F):
            check_filter_blocks(big[i, pos:pos + np_], part[i, :np_], x, N, "fallback == r16 bank filter %d" % i,
                                b0=pos // N, rms=False)
        pos += np_
        del part
    assert pos == nblk * N


@pytest.mark.parametrize("block", [64, 1024, 4096, 5000])
def test_filter_out_stride(block):
    """Every bank kernel writes filter f at out + f * out_stride: with out_stride = n_out + 37 into a NaN-filled buffer
    the 37 gap columns stay NaN and every row equals the call with out_stride = n_out."""
    F, pad = 3, 37
    nblk = {64: 300, 1024: 300, 4096: 700, 5000: 10}[block]
    M = 16384
    want = {64: 1, 1024: 2, 4096: 1, 5000: general_ola_launches(nblk, F, M)}[block]
    x = _randn(nblk * block + block // 3, seed=block + 37)
    a, n_out, ka = filter_exec(make_node(block, BANDS3), x, F)
    b, n_out_b, kb = filter_exec(make_node(block, BANDS3), x, F, pad=pad)
    assert n_out == n_out_b == nblk * block and ka == kb == want
    assert bool(torch.isnan(torch.view_as_real(b[:, n_out:])).all()), "a gap column was written"
    assert torch.equal(b[:, :n_out], a), "rows differ with a wider out_stride"
    t = taps_of(block, BANDS3[1])
    check_spot_blocks(b[1, :n_out], x, t, [0, nblk - 1], "out_stride block %d" % block)


def test_filter_process_without_filters_returns_no_rows():
    """No filters: FilterSink without sources emits nothing -- (0, n_out) from both entry points."""
    f = FilterNode(64)
    f.config(sample_rate=FS, buffer_size=64)
    xh = np.ones(200, np.complex64)
    assert f.process(xh).shape == (0, 192)
    y = f.process(torch.from_numpy(xh).cuda())
    torch.cuda.synchronize()
    assert tuple(y.shape) == (0, 192)               # 8 pending + 200 new samples: 3 blocks


def _bank_launches(block, F, nblk):
    """Launches of one FilterNode call with F filters and nblk completed blocks (launch_filter_ola, GeneralOla::run)."""
    if nblk == 0:
        return 0
    if block == 5000:
        return general_ola_launches(nblk, F, 16384)
    if block == 1024 and F >= 2:
        return 2                                    # filter_ola1_r16_kernel<1>, <2>
    return 1                                        # filter_ola_kernel (no filter: only the history roll), r16<0>, conv8k


@pytest.mark.parametrize("block", [64, 1024, 4096, 5000])
def test_filter_add_filters_mid_stream(block):
    """A node started with no filters still carries the stream's history: after addFilter x2, and later a third on the
    running bank, its outputs equal those of a node that had the filters from the start, over the samples after each
    add.  At block 4096 the third add regenerates the permuted spectra on a running bank and the last, larger call
    (400 blocks > the 296-CTA grid) grows the bank's spectrum scratch."""
    N = block
    calls = [5 * N + 3, 7 * N + N // 2, 40 * N + 1, 50 * N + 11, 400 * N + 5]
    adds = {2: (0, 1), 4: (2,)}                     # band indices added before call index
    x = _randn(sum(calls), seed=block + 99)
    late = FilterNode(N)
    late.config(sample_rate=FS, buffer_size=N)
    full = make_node(N, BANDS3)
    late_out, first_blk, full_out = {0: [], 1: [], 2: []}, {}, []
    pos = 0
    for ci, c in enumerate(calls):
        for bi in adds.get(ci, ()):
            assert late.addFilter(*BANDS3[bi]) == bi
            first_blk[bi] = pos // N                # the next call's output starts at the block holding sample pos
        F = late.n_filters()
        seg = x[pos:pos + c]
        if F == 0:                                  # the Python mirror: no rows, however many blocks complete
            yl, kl = _launches_of(lambda: late.process(seg))
            nl = yl.shape[1]
            assert tuple(yl.shape) == (0, ((pos % N) + c) // N * N)
        else:
            yl, nl, kl = filter_exec(late, seg, F)
        yf, nf, kf = filter_exec(full, seg, 3)
        assert nl == nf
        assert kl == _bank_launches(N, F, nl // N) and kf == _bank_launches(N, 3, nf // N), (ci, kl, kf)
        for i in range(F):
            late_out[i].append(yl[i, :nl])
        full_out.append(yf[:, :nf])
        pos += c
    full_y = torch.cat(full_out, dim=1)
    del full_out
    ref = FilterRef(x[:full_y.shape[1]])
    for i in range(3):
        got = torch.cat(late_out[i])
        s = first_blk[i] * N
        assert got.numel() == full_y.shape[1] - s
        assert torch.equal(got, full_y[i, s:]), "filter %d added mid-stream differs from the node that had it" % i
        check_filter_blocks(got, ref(taps_of(N, BANDS3[i]))[s:], x, N, "added mid-stream block %d filter %d" % (N, i),
                            b0=first_blk[i])

// fft_kernels.cu -- shared-memory Stockham FFT and the fused FFT-convolution filter.
//
// Replaces, on the device:
//   FFTPlan<float> / FFT::exec (src/fftplan.hh:11-34, src/fftplan_fftw3.hh:79-142; FFTW3 itself is
//   an external, un-vendored dependency): unnormalised c2c DFT, FORWARD = exp(-i..), any power of
//   two 2..8192, one CTA per transform, no cuFFT.
//   FilterSink + FilterSource (src/filternode.hh:81-88,164-181): per block of N samples, a forward
//   FFT of size 2N shared by all filters of the bank, then per filter a spectrum multiply, a
//   backward FFT, 1/(2N) scaling and the overlap.
// The overlap is evaluated as overlap-SAVE (each CTA transforms [previous block | current block]
// and keeps the second half) instead of the reference's overlap-ADD: both compute the same causal
// linear convolution y[n] = sum_j (h[j]/nrm) x[n-j] (SURVEY.md 8 a8), but overlap-save has no
// dependency between consecutive blocks, so all blocks of a buffer run in parallel; the carried
// state is the last N input samples instead of the last N output partials.
//
// Stockham autosort, decimation in time: at a stage with radix R and Ns = product of the radices
// already applied, butterfly j (0 <= j < n/R) reads x[j + r n/R], multiplies by w^(r (j mod Ns))
// with w = exp(-/+ 2 pi i /(Ns R)), applies the R-point DFT in registers and writes to
// (j div Ns) Ns R + (j mod Ns) + r Ns.  Twiddles come from a table of n-th roots of unity computed
// in double on the host.  Data ping-pongs between shared-memory buffers; one __syncthreads per stage.
#include "fft_kernels.cuh"
#include "fft_device.cuh"
#include "launch.cuh"

namespace sdrg {
namespace {

// Shared-memory index padding: one spare element after every 16 (= one 128-byte row of 8-byte
// elements).  Consecutive reads stay conflict free (an aligned half-warp never straddles a pad),
// while the stride-8 writes of the first stage spread over all 16 bank pairs (simulated per stage:
// 1.0 wavefronts per half-warp everywhere except the second stage's writes at 2.0; the unpadded
// layout costs 8.0 there and a pad every 8 elements makes EVERY read 2-way conflicted).
__device__ __forceinline__ int pidx(int i) { return i + (i >> 4); }
__host__ __device__ constexpr int padded_len(int n) { return n + (n >> 4) + 8; }

// One Stockham stage of radix R over `n` points: src -> dst.  `mul` (optional) is multiplied into
// the inputs as they are read (the filter's spectrum).
template <int R, bool INV>
__device__ __forceinline__ void stage(const float2 *__restrict__ src, float2 *__restrict__ dst, const int n, const int Ns,
                                      const float2 *__restrict__ tw, const float2 *__restrict__ mul) {
  const int nb = n / R;
  const int tstep = n / (Ns * R);            // index step of w = exp(-2 pi i/(Ns R)) in the n-th root table
  for (int j = threadIdx.x; j < nb; j += blockDim.x) {
    float2 v[R];
    const int k = j & (Ns - 1);              // j mod Ns (Ns is a power of two)
#pragma unroll
    for (int r = 0; r < R; ++r) {
      v[r] = src[pidx(j + r * nb)];
      if (mul) v[r] = cmulf(v[r], __ldg(mul + j + r * nb));
    }
    if (k > 0) {
      // w^r for r = 1..R-1 from ONE table load: w2 = w w, w3 = w2 w, w4 = w2 w2, ... (depth <= 3)
      float2 w1 = __ldg(tw + k * tstep);
      if (INV) w1.y = -w1.y;
      v[1] = cmulf(v[1], w1);
      if (R > 2) {
        const float2 w2 = cmulf(w1, w1), w3 = cmulf(w2, w1);
        v[2] = cmulf(v[2], w2); v[3] = cmulf(v[3], w3);
        if (R > 4) {
          const float2 w4 = cmulf(w2, w2), w5 = cmulf(w4, w1), w6 = cmulf(w4, w2), w7 = cmulf(w4, w3);
          v[4] = cmulf(v[4], w4); v[5] = cmulf(v[5], w5); v[6] = cmulf(v[6], w6); v[7] = cmulf(v[7], w7);
        }
      }
    }
    if (R == 2) dft2<INV>(v[0], v[1]);
    else if (R == 4) dft4<INV>(v);
    else dft8<INV>(v);
    const int base = (j - k) * R + k;        // (j div Ns) Ns R + (j mod Ns)
#pragma unroll
    for (int r = 0; r < R; ++r) dst[pidx(base + r * Ns)] = v[r];
  }
}

// All stages of an n-point transform (n = 2^log2n): radix 8 while possible, then 4 or 2.
// Returns the buffer holding the result.  `keep` (optional): never written, used for `a` on entry
// when the caller needs the input preserved (then results alternate between b and c).
template <bool INV>
__device__ float2 *fft_smem(float2 *a, float2 *b, float2 *c, const int n, const int log2n, const float2 *tw, const float2 *mul) {
  int Ns = 1, left = log2n;
  const float2 *src = a;
  float2 *dst = b;
  bool first = true;
  while (left > 0) {
    const float2 *m = first ? mul : nullptr;
    if (left >= 3 && left != 4) { stage<8, INV>(src, dst, n, Ns, tw, m); Ns *= 8; left -= 3; }
    else if (left >= 2) { stage<4, INV>(src, dst, n, Ns, tw, m); Ns *= 4; left -= 2; }
    else { stage<2, INV>(src, dst, n, Ns, tw, m); Ns *= 2; left -= 1; }
    __syncthreads();
    first = false;
    src = dst;
    dst = (dst == b) ? (c ? c : a) : b;
  }
  return const_cast<float2 *>(src);
}

// ---- in-place variant -------------------------------------------------------------------------------
// The same stages on ONE shared buffer: every thread first pulls all the inputs of its butterflies
// into registers, the CTA synchronises, then the outputs are written (two barriers per stage instead
// of one, half the shared memory -> two resident CTAs of 1024 threads per SM for the 8192-point
// transform).  B = butterflies per thread (n/R/blockDim), at most 8/R * 8... kept <= 8 elements/thread
// for n <= 8 * blockDim.
// SRC_G: the inputs come straight from global memory `gin` (natural order, coalesced: consecutive threads read
// consecutive j) -- nothing in `buf` is live, so the barrier between the read and the write phase is dropped.
// DST_G: the outputs go straight to global memory `gout`; legal for the LAST stage only, where Ns = n/R makes the
// output index j + r n/R coalesced as well.
template <int R, bool INV, int B, bool SRC_G = false, bool DST_G = false>
__device__ __forceinline__ void stage_inplace(float2 *__restrict__ buf, const int n, const int Ns,
                                              const float2 *__restrict__ tw, const float2 *__restrict__ mul,
                                              const int tid, const int nthr,
                                              const float2 *__restrict__ gin = nullptr, float2 *__restrict__ gout = nullptr) {
  const int nb = n / R;
  const int tstep = n / (Ns * R);
  float2 v[B][R];
#pragma unroll
  for (int b = 0; b < B; ++b) {
    const int j = tid + b * nthr;
    if (j < nb) {
      const int k = j & (Ns - 1);
#pragma unroll
      for (int r = 0; r < R; ++r) {
        v[b][r] = SRC_G ? gin[j + r * nb] : buf[pidx(j + r * nb)];
        if (mul) v[b][r] = cmulf(v[b][r], __ldg(mul + j + r * nb));
      }
      if (k > 0) {
        float2 w1 = __ldg(tw + k * tstep);
        if (INV) w1.y = -w1.y;
        if (R <= 8) {
          v[b][1] = cmulf(v[b][1], w1);
          if (R > 2) {
            const float2 w2 = cmulf(w1, w1), w3 = cmulf(w2, w1);
            v[b][2] = cmulf(v[b][2], w2); v[b][3] = cmulf(v[b][3], w3);
            if (R > 4) {
              const float2 w4 = cmulf(w2, w2), w5 = cmulf(w4, w1), w6 = cmulf(w4, w2), w7 = cmulf(w4, w3);
              v[b][4] = cmulf(v[b][4], w4); v[b][5] = cmulf(v[b][5], w5); v[b][6] = cmulf(v[b][6], w6); v[b][7] = cmulf(v[b][7], w7);
            }
          }
        } else {
          // radix 16: two chains stepping by w^2 (depth 7), only w1, w2 and the two heads stay live
          const float2 w2 = cmulf(w1, w1);
          float2 we = w2, wo = w1;
#pragma unroll
          for (int r = 1; r < R; r += 2) {
            v[b][r] = cmulf(v[b][r], wo);
            if (r + 1 < R) { v[b][r + 1] = cmulf(v[b][r + 1], we); wo = cmulf(wo, w2); we = cmulf(we, w2); }
          }
        }
      }
      if (R == 2) dft2<INV>(v[b][0], v[b][1]);
      else if (R == 4) dft4<INV>(v[b]);
      else if (R == 8) dft8<INV>(v[b]);
      else dft16<INV>(v[b]);
    }
  }
  if (!SRC_G) __syncthreads();
#pragma unroll
  for (int b = 0; b < B; ++b) {
    const int j = tid + b * nthr;
    if (j < nb) {
      const int k = j & (Ns - 1);
      const int base = (j - k) * R + k;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        if (DST_G) gout[base + r * Ns] = v[b][r];
        else buf[pidx(base + r * Ns)] = v[b][r];
      }
    }
  }
  if (!DST_G) __syncthreads();
}

// Stages for the middle `bits` bits of a transform whose first (forward) or last (inverse) radix-2
// stage is fused into the global load / store: radix 16 while possible, then 8 / 4 / 2.
template <bool INV>
__device__ void fft_smem_inplace16(float2 *buf, const int n, int Ns, int left, const float2 *tw, const float2 *mul,
                                   const int tid, const int nthr) {
  bool first = true;
  while (left > 0) {
    const float2 *m = first ? mul : nullptr;
    if (left >= 4 && left != 5) { stage_inplace<16, INV, 1>(buf, n, Ns, tw, m, tid, nthr); Ns *= 16; left -= 4; }
    else if (left >= 3) { stage_inplace<8, INV, 2>(buf, n, Ns, tw, m, tid, nthr); Ns *= 8; left -= 3; }
    else if (left >= 2) { stage_inplace<4, INV, 4>(buf, n, Ns, tw, m, tid, nthr); Ns *= 4; left -= 2; }
    else { stage_inplace<2, INV, 8>(buf, n, Ns, tw, m, tid, nthr); Ns *= 2; left -= 1; }
    first = false;
  }
}

// Single-filter overlap-save, radix-16 plan (n = 2N >= 512, 16 elements per thread).  The forward
// transform's first radix-2 stage has no twiddles (Ns = 1) and is applied while the two input blocks
// are loaded; the inverse transform's LAST radix-2 stage (Ns = N) is applied while storing, and only
// its second half -- the N valid overlap-save outputs y[N + j] = a[j] - w^j b[j] -- is evaluated.
// At n = 8192 that leaves 3 + 3 shared-memory passes (16 x 16 x 16) instead of 5 + 5.
// MODE 0: forward + inverse fused (one filter).  MODE 1: forward only, the spectrum of block b goes to
// a.spec (a filter bank shares it).  MODE 2: inverse only for filter blockIdx.y, reading a.spec.
template <int MODE>
__global__ void __launch_bounds__(512, 2) filter_ola1_r16_kernel(const FilterArgs a) {
  extern __shared__ __align__(16) unsigned char fft_smem_raw[];
  const int N = a.block, n = 2 * N;
  float2 *s0 = (float2 *)fft_smem_raw;
  const int b = blockIdx.x;
  const float2 *tw = (const float2 *)a.tw;
  if (MODE != 2) {
    const float2 *x = (const float2 *)a.x;
    const float2 *prev = b == 0 ? (const float2 *)a.hist_in : x + (size_t)(b - 1) * N;
    const float2 *cur = x + (size_t)b * N;
    const bool roll = b == (int)gridDim.x - 1;
    float2 *ho = (float2 *)a.hist_out;
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
      const float2 p = prev[i], c = cur[i];
      s0[pidx(2 * i)] = caddf(p, c);                 // Stockham radix-2, Ns = 1: dst[2j] = x[j] + x[j + n/2]
      s0[pidx(2 * i + 1)] = csubf(p, c);
      if (roll) ho[i] = c;
    }
    __syncthreads();
    fft_smem_inplace16<false>(s0, n, 2, a.log2n - 1, tw, nullptr, threadIdx.x, blockDim.x);
  }
  if (MODE == 1) {
    float2 *X = (float2 *)a.spec + (size_t)b * n;
    for (int i = threadIdx.x; i < n; i += blockDim.x) X[i] = s0[pidx(i)];
    return;
  }
  const int f = MODE == 2 ? (int)blockIdx.y : 0;
  const float2 *K = (const float2 *)a.kern + (size_t)f * n;
  if (MODE == 2) {
    const float2 *X = (const float2 *)a.spec + (size_t)b * n;
    for (int i = threadIdx.x; i < n; i += blockDim.x) s0[pidx(i)] = cmulf(X[i], __ldg(K + i));
    __syncthreads();
    fft_smem_inplace16<true>(s0, n, 1, a.log2n - 1, tw, nullptr, threadIdx.x, blockDim.x);
  } else {
    fft_smem_inplace16<true>(s0, n, 1, a.log2n - 1, tw, K, threadIdx.x, blockDim.x);
  }
  const float sc = 1.0f / (float)n;
  float2 *o = (float2 *)a.out + (size_t)f * a.out_stride + (size_t)b * N;
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    float2 w = __ldg(tw + j); w.y = -w.y;          // exp(+2 pi i j / n)
    const float2 v = csubf(s0[pidx(j)], cmulf(s0[pidx(N + j)], w));
    o[j] = make_float2(v.x * sc, v.y * sc);
  }
}

// ---- batched plain FFT (FFTPlan<float>::operator()) ---------------------------------------------
__global__ void __launch_bounds__(1024) fft_batch_kernel(const float2 *__restrict__ in, float2 *__restrict__ out, const int n,
                                                          const int log2n, const int inverse, const float2 *__restrict__ tw) {
  extern __shared__ __align__(16) unsigned char fft_smem_raw[];
  float2 *a = (float2 *)fft_smem_raw, *b = a + padded_len(n);
  const float2 *x = in + (size_t)blockIdx.x * n;
  for (int i = threadIdx.x; i < n; i += blockDim.x) a[pidx(i)] = x[i];
  __syncthreads();
  float2 *r = inverse ? fft_smem<true>(a, b, nullptr, n, log2n, tw, nullptr) : fft_smem<false>(a, b, nullptr, n, log2n, tw, nullptr);
  float2 *y = out + (size_t)blockIdx.x * n;
  for (int i = threadIdx.x; i < n; i += blockDim.x) y[i] = r[pidx(i)];
}

// Radix-16 in-place plan for the plain transform (n >= 256): n/16 threads per transform, several
// transforms per CTA when n is small; an odd log2 n sheds its radix-2 stage into the global load
// (Stockham DIT first stage, Ns = 1, no twiddles), so n = 8192 costs three shared-memory passes.
template <bool INV>
__global__ void __launch_bounds__(512, 2) fft_batch_r16_kernel(const float2 *__restrict__ in, float2 *__restrict__ out, const int n,
                                                                const int log2n, const int batch, const float2 *__restrict__ tw) {
  extern __shared__ __align__(16) unsigned char fft_smem_raw[];
  const int tpf = n >> 4;                                  // threads per transform
  const int fpc = blockDim.x / tpf;                        // transforms per CTA
  const int g = threadIdx.x / tpf, tid = threadIdx.x - g * tpf;
  int f = blockIdx.x * fpc + g;
  const bool live = f < batch;
  if (!live) f = batch - 1;                                // keeps the barriers uniform; the result goes to a dummy row
  float2 *s0 = (float2 *)fft_smem_raw + (size_t)g * padded_len(n);
  const float2 *x = in + (size_t)f * n;
  float2 *y = live ? out + (size_t)f * n : s0;             // dead groups "store" into their own shared buffer (never read again)
  // first stage: radix 16 straight from global memory (Ns = 1: no twiddles), 16 independent loads per thread
  stage_inplace<16, INV, 1, true, false>(s0, n, 1, tw, nullptr, tid, tpf, x, nullptr);
  int Ns = 16, left = log2n - 4;
  // middle stages in shared memory; the last one writes straight to global memory
  while (left > 0) {
    if (left >= 4) {                                       // 16 while possible; the remainder (8, 4 or 2) is the last stage
      if (left == 4) stage_inplace<16, INV, 1, false, true>(s0, n, Ns, tw, nullptr, tid, tpf, nullptr, y);
      else stage_inplace<16, INV, 1>(s0, n, Ns, tw, nullptr, tid, tpf);
      Ns *= 16; left -= 4;
    } else if (left == 3) {
      stage_inplace<8, INV, 2, false, true>(s0, n, Ns, tw, nullptr, tid, tpf, nullptr, y);
      Ns *= 8; left -= 3;
    } else if (left == 2) {
      stage_inplace<4, INV, 4, false, true>(s0, n, Ns, tw, nullptr, tid, tpf, nullptr, y);
      Ns *= 4; left -= 2;
    } else {
      stage_inplace<2, INV, 8, false, true>(s0, n, Ns, tw, nullptr, tid, tpf, nullptr, y);
      Ns *= 2; left -= 1;
    }
  }
}

// ---- fused overlap-save filter bank -----------------------------------------------------------------
// CTA b: X = FFT_2N([block b-1 | block b]); for every filter f: y = IFFT_2N(X K_f); out_f[block b] =
// y[N..2N) / 2N.  Block -1 is the carried history (the last N samples of the previous call).
__global__ void __launch_bounds__(1024) filter_ola_kernel(const FilterArgs a) {
  extern __shared__ __align__(16) unsigned char fft_smem_raw[];
  const int N = a.block, n = 2 * N;
  float2 *s0 = (float2 *)fft_smem_raw, *s1 = s0 + padded_len(n), *s2 = s1 + padded_len(n);
  const int b = blockIdx.x;
  const float2 *x = (const float2 *)a.x;
  const float2 *prev = b == 0 ? (const float2 *)a.hist_in : x + (size_t)(b - 1) * N;
  const float2 *cur = x + (size_t)b * N;
  for (int i = threadIdx.x; i < N; i += blockDim.x) { s0[pidx(i)] = prev[i]; s0[pidx(N + i)] = cur[i]; }
  if (b == (int)gridDim.x - 1) {             // roll the history: the last block of this call
    float2 *ho = (float2 *)a.hist_out;
    for (int i = threadIdx.x; i < N; i += blockDim.x) ho[i] = cur[i];
  }
  __syncthreads();
  const float2 *tw = (const float2 *)a.tw;
  float2 *X = fft_smem<false>(s0, s1, nullptr, n, a.log2n, tw, nullptr);    // lands in s0 or s1
  float2 *w1 = (X == s0) ? s1 : s0;
  const float sc = 1.0f / (float)n;
  for (int f = 0; f < a.n_filters; ++f) {
    const float2 *K = (const float2 *)a.kern + (size_t)f * n;
    // X is only read (first stage, with the spectrum multiplied in); later stages alternate w1 <-> s2
    float2 *y = fft_smem<true>(X, w1, s2, n, a.log2n, tw, K);
    float2 *o = (float2 *)a.out + (size_t)f * a.out_stride + (size_t)b * N;
    for (int i = threadIdx.x; i < N; i += blockDim.x) { const float2 v = y[pidx(N + i)]; o[i] = make_float2(v.x * sc, v.y * sc); }
    __syncthreads();
  }
}

}  // namespace

int launch_fft_batch(const void *in, void *out, int n, int log2n, int inverse, size_t batch, const void *tw, cudaStream_t st) {
  if (batch == 0) return SDRG_OK;
  if (n >= 256 && batch <= 0x7fffffffull) {
    const int tpf = n / 16, fpc = tpf >= 256 ? 1 : 256 / tpf;
    const size_t smem = (size_t)fpc * padded_len(n) * sizeof(float2);
    return launch("fft_batch_r16_kernel", inverse ? fft_batch_r16_kernel<true> : fft_batch_r16_kernel<false>, (unsigned)((batch + fpc - 1) / fpc),
                  tpf * fpc, smem, st, (const float2 *)in, (float2 *)out, n, log2n, (int)batch, (const float2 *)tw);
  }
  int threads = n / 8; if (threads < 32) threads = 32; if (threads > 1024) threads = 1024;
  return launch("fft_batch_kernel", fft_batch_kernel, (unsigned)batch, threads, (size_t)2 * padded_len(n) * sizeof(float2), st,
                (const float2 *)in, (float2 *)out, n, log2n, inverse, (const float2 *)tw);
}

int launch_filter_ola(const FilterArgs &a, size_t n_blocks, cudaStream_t st) {
  if (n_blocks == 0) return SDRG_OK;
  const int n = 2 * a.block;
  if (n == 8192 && a.n_filters >= 1 && a.kperm && a.tab8k) return launch_conv8k(a, n_blocks, st);
  if (n >= 512 && (a.n_filters == 1 || a.spec)) {   // in-place stages on a single buffer (n == 16 * threads)
    const size_t smem1 = (size_t)padded_len(n) * sizeof(float2);
    if (a.n_filters == 1) return launch("filter_ola1_r16_kernel", filter_ola1_r16_kernel<0>, (unsigned)n_blocks, n / 16, smem1, st, a);
    // bank: one forward pass, then every (block, filter) pair on its own CTA
    const int rc = launch("filter_ola1_r16_kernel<fwd>", filter_ola1_r16_kernel<1>, (unsigned)n_blocks, n / 16, smem1, st, a);
    if (rc) return rc;
    return launch("filter_ola1_r16_kernel<inv>", filter_ola1_r16_kernel<2>, dim3((unsigned)n_blocks, (unsigned)a.n_filters), n / 16, smem1, st, a);
  }
  int threads = n / 8; if (threads < 32) threads = 32; if (threads > 1024) threads = 1024;
  return launch("filter_ola_kernel", filter_ola_kernel, (unsigned)n_blocks, threads, (size_t)3 * padded_len(n) * sizeof(float2), st, a);
}

}  // namespace sdrg

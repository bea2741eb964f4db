// fft8k_kernels.cu -- the 8192 / 4096-point transforms (and, in conv8k_kernels.cu on the same stages, fft8k_stages.cuh,
// the block-4096 FFT convolution of BASELINE config 3),
// restructured around three facts measured on the radix-16 Stockham kernels they replace
// (profiles/r01_final_fft_filter_kernel_summary.md: 64-register cap with spills, address/twiddle arithmetic on
// the ALU pipe costing more issue slots than the butterflies, 3 + 3 shared-memory round trips):
//
//  * An 8192-point DFT is split by ONE decimation-in-frequency radix-2 step, applied while the samples are
//    loaded, into two independent 4096-point DFTs (even and odd bins); 4096 = 16 x 16 x 16, so each half is
//    three radix-16 stages, one butterfly per thread and stage (256 threads, 16 + 16 elements per thread,
//    128 registers at 2 CTAs/SM: no spills).
//  * The stages are IN PLACE in the Cooley-Tukey sense: a butterfly reads and writes the same 16 locations, so
//    a stage needs one CTA barrier and a thread may run its two butterflies (one per half) back to back.  The
//    spectrum therefore comes out digit-reversed -- which a convolution never has to undo: the filter's
//    spectrum is stored in the same permuted order (host, config time) and the inverse transform is the mirror
//    image (decimation in time) that consumes digit-reversed input and delivers natural order.  The last
//    forward stage, the spectrum multiply and the first inverse stage all happen in registers: 4 shared-memory
//    round trips per block instead of 6.  For the plain FFTPlan transform the digit reversal is absorbed by
//    the last stage's thread mapping: thread t holds bins t + 256 q of both halves, i.e. X[2(t + 256 q)] and
//    X[2(t + 256 q) + 1], and stores them as one coalesced float4.
//  * Every twiddle is a table entry (double precision on the host, rounded once): w_4096^(q u), w_256^(q c),
//    w_8192^u, w_32^a live in shared memory, indexed so that a warp reads consecutive or broadcast words.  No
//    product chains, no sincos, no per-stage index arithmetic beyond shifts and adds.
//
// Index algebra (checked against numpy.fft by scratch/fft8k_model.py, which mirrors this file line by line):
//   half h, input index j = 256 a + 16 b + c, output bin m = qa + 16 qb + 256 qc,
//   w_4096^(j m) = w_16^(a qa) . w_4096^(qa (16 b + c)) . w_16^(b qb) . w_256^(c qb) . w_16^(c qc)
//   stage 1: DFT16 over a, twiddle w_4096^(qa (16b + c));  stage 2: DFT16 over b, twiddle w_256^(qb c);
//   stage 3: DFT16 over c.  Position 256 qa + 16 qb + qc then holds U[qa + 16 qb + 256 qc].
// Reference interfaces replaced: FFTPlan<float> (src/fftplan_fftw3.hh:79-142, FFTW3 underneath) and
// FilterSink/FilterSource (src/filternode.hh:81-88,164-181).
#include "fft8k_stages.cuh"

namespace sdrg {
namespace {

// ---- FFTPlan<float>: batched 8192-point (SPLIT) or 4096-point (two transforms per iteration) DFT ----------
template <bool INV, bool SPLIT>
__global__ void __launch_bounds__(kT, 2) fft8k_kernel(const float2 *__restrict__ in, float2 *__restrict__ out, const int batch,
                                                      const float2 *__restrict__ gtab) {
  extern __shared__ __align__(16) unsigned char fft8k_smem[];
  float2 *H0 = (float2 *)fft8k_smem, *H1 = H0 + kHalfPad, *tab = H1 + kHalfPad;
  const int t = threadIdx.x;
  load_tables(tab, gtab);
  __syncthreads();
  const int items = SPLIT ? batch : (batch + 1) / 2;
  for (int it = blockIdx.x; it < items; it += gridDim.x) {
    const size_t f0 = SPLIT ? (size_t)it : (size_t)2 * it;
    const bool second = SPLIT || (f0 + 1 < (size_t)batch);
    const float2 *xa = in + f0 * (SPLIT ? 8192 : 4096);
    const float2 *xb = SPLIT ? xa + kHalf : (second ? xa + kHalf : xa);
    {
      float2 e[16], o[16];
#pragma unroll
      for (int a = 0; a < 16; ++a) { e[a] = xa[256 * a + t]; o[a] = xb[256 * a + t]; }
      if (it + (int)gridDim.x < items) {      // the next item of this CTA: 64 KB, two 128-byte lines per thread, into L2
        const char *nx = (const char *)(xa + (size_t)gridDim.x * 8192);
        prefetch_l2(nx + 128 * t); prefetch_l2(nx + 128 * (t + 256));
      }
      if (SPLIT) {
        const float2 wt = tab[kT8 + t];
#pragma unroll
        for (int a = 0; a < 16; ++a) {
          const float2 p = e[a], c = o[a];
          e[a] = caddf(p, c);
          o[a] = cmulw<INV>(csubf(p, c), root8k(wt, a));
        }
      }
      dif_stage1<INV>(e, o, H0, tab, t);
    }
    __syncthreads();
    dif_stage2<INV>(H0, tab, t);
    __syncthreads();
    {
      float2 e[16], o[16];
      const int p0 = stage3_pos(t);
      load16(e, H0, p0); load16(o, H1, p0);
      dft16<INV>(e); dft16<INV>(o);
      if (SPLIT) {               // X[2 m] = E[m], X[2 m + 1] = O[m], m = t + 256 q: one float4 per bin pair
        float4 *y = (float4 *)(out + f0 * 8192);
#pragma unroll
        for (int q = 0; q < 16; ++q) y[t + 256 * q] = make_float4(e[q].x, e[q].y, o[q].x, o[q].y);
      } else {
        float2 *ya = out + f0 * 4096, *yb = ya + kHalf;
#pragma unroll
        for (int q = 0; q < 16; ++q) { ya[t + 256 * q] = e[q]; if (second) yb[t + 256 * q] = o[q]; }
      }
    }                            // (stage 3 only read; the barrier inside the next item's stage 1 orders its stores behind this)
  }
}

}  // namespace


// host: the shared tables, double precision rounded once
void fft8k_tables(std::vector<float> &tab) {
  tab.assign(2 * (size_t)kTabLen, 0.f);
  auto put = [&](int idx, double num, double den) {
    const double ang = -2.0 * M_PI * std::fmod(num, den) / den;
    tab[2 * idx] = (float)std::cos(ang); tab[2 * idx + 1] = (float)std::sin(ang);
  };
  for (int q = 0; q < 16; ++q) for (int u = 0; u < 256; ++u) put(kT1 + 256 * q + u, (double)(q * u), 4096.0);
  for (int q = 0; q < 16; ++q) for (int c = 0; c < 16; ++c) put(kT2 + 16 * q + c, (double)(q * c), 256.0);
  for (int u = 0; u < 256; ++u) put(kT8 + u, (double)u, 8192.0);
}

// host: spectrum K (8192 complex, natural order) -> the kernel's order, scaled by 1/8192 (exact: a power of two)
void fft8k_permute_kernel(const float *kern, float *kperm) {
  for (int h = 0; h < 2; ++h)
    for (int qc = 0; qc < 16; ++qc)
      for (int t = 0; t < 256; ++t) {
        const int m = (t >> 4) + 16 * (t & 15) + 256 * qc;
        const int src = 2 * m + h, dst = (h * 16 + qc) * 256 + t;
        kperm[2 * dst] = kern[2 * src] * (1.0f / 8192.0f);
        kperm[2 * dst + 1] = kern[2 * src + 1] * (1.0f / 8192.0f);
      }
}

int launch_fft8k(const void *in, void *out, int n, int inverse, size_t batch, const void *tab, cudaStream_t st) {
  if (batch == 0) return SDRG_OK;
  if (batch > 0x7fffffffull) return set_error(SDRG_ERR_ARG, "FFT plan: batch too large");
  const bool full = n == 8192;
  auto *kern = inverse ? (full ? fft8k_kernel<true, true> : fft8k_kernel<true, false>) : (full ? fft8k_kernel<false, true> : fft8k_kernel<false, false>);
  return launch_persistent("fft8k_kernel", kern, full ? batch : (batch + 1) / 2, kT, kSmemBytes, st,
                           (const float2 *)in, (float2 *)out, (int)batch, (const float2 *)tab);
}

}  // namespace sdrg

// conv8k_kernels.cu -- the block-4096 overlap-save FFT convolution (BASELINE config 3): FilterSink / FilterSource of
// src/filternode.hh:81-88,164-181 fused into one kernel on the in-place radix-16 stages of fft8k_stages.cuh (method and
// index algebra: fft8k_kernels.cu).  This translation unit builds the butterflies from packed FP32 instructions
// (FADD2 / FMUL2 / FFMA2, fft_device.cuh): the convolution runs two transforms and a spectrum multiply per block and
// gains 2.5-3.4 % from the halved instruction count (C3 99.2 -> 101.7 GS/s, 4-filter bank 35.5 -> 36.7 GS/s of input),
// whereas the plain FFTPlan kernels, which are closer to the HBM roofline and run the same 4 warps per scheduler, lose
// 2-7 % (8192: 0.433 -> 0.440 ms/GiB, 2048: 0.524 -> 0.560) and keep the scalar form.
#define SDRG_FFT_PACKED 1
#include "fft8k_stages.cuh"

namespace sdrg {
namespace {

// ---- block-4096 overlap-save convolution, fused ------------------------------------------------------------
// y[N + j] = IDFT_8192(DFT_8192([prev | cur]) K)[N + j] / 8192 = v0[j] - conj(w_8192^j) v1[j], v_h the 4096-point
// backward DFTs of the even / odd bins.  K arrives permuted and pre-scaled: kp[(h 16 + qc) 256 + t] = K[2 m + h] / 8192,
// m = (t >> 4) + 16 (t & 15) + 256 qc the bin thread t holds after stage 3.
// BANK = false: one filter; the last forward stage, the spectrum multiply and the first inverse stage stay in registers.
// BANK = true: F filters on one FilterSink (src/filternode.hh:262-270).  The forward transform runs once per block; its
// spectrum (digit-reversed, 64 KB) goes to a CTA-private scratch line in global memory -- written and read back by the
// SAME thread, so no barrier is involved and, with at most 2 x 148 CTAs, the scratch (19 MB) never leaves L2 -- and
// every filter then runs the inverse half.
template <bool BANK>
__global__ void __launch_bounds__(kT, 2) conv8k_kernel(const FilterArgs a, const int n_blocks) {
  extern __shared__ __align__(16) unsigned char fft8k_smem[];
  float2 *H0 = (float2 *)fft8k_smem, *H1 = H0 + kHalfPad, *tab = H1 + kHalfPad;
  const int t = threadIdx.x;
  load_tables(tab, (const float2 *)a.tab8k);
  __syncthreads();
  const float2 *x = (const float2 *)a.x;
  float2 *scratch = BANK ? (float2 *)a.spec + (size_t)blockIdx.x * 8192 + t : nullptr;
  const int n_filters = BANK ? a.n_filters : 1;
  for (int blk = blockIdx.x; blk < n_blocks; blk += gridDim.x) {
    const float2 *prev = blk == 0 ? (const float2 *)a.hist_in : x + (size_t)(blk - 1) * kHalf;
    const float2 *cur = x + (size_t)blk * kHalf;
    {   // load, radix-2 DIF step, stage 1 of both halves
      float2 e[16], o[16];
#pragma unroll
      for (int q = 0; q < 16; ++q) { e[q] = prev[256 * q + t]; o[q] = cur[256 * q + t]; }
      if (blk + (int)gridDim.x < n_blocks) {   // this CTA's next block pair: 64 KB into L2 while this one is computed
        const char *nx = (const char *)(cur + ((size_t)gridDim.x - 1) * kHalf);
        prefetch_l2(nx + 128 * t); prefetch_l2(nx + 128 * (t + 256));
      }
      if (blk == n_blocks - 1) {
        float2 *ho = (float2 *)a.hist_out;
#pragma unroll
        for (int q = 0; q < 16; ++q) ho[256 * q + t] = o[q];
      }
      const float2 wt = tab[kT8 + t];
#pragma unroll
      for (int q = 0; q < 16; ++q) {
        const float2 p = e[q], c = o[q];
        e[q] = caddf(p, c);
        o[q] = cmulf(csubf(p, c), root8k(wt, q));
      }
      dif_stage1<false>(e, o, H0, tab, t);
    }
    __syncthreads();
    dif_stage2<false>(H0, tab, t);
    __syncwarp();                // stage 3 reads what lanes of this warp wrote (see stage3_pos_conv)
    const int qb = t & 15, p0 = stage3_pos_conv(t);
    if (BANK) {      // forward stage 3 -> the CTA's scratch line
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float2 v[16];
        load16(v, h ? H1 : H0, p0);
        dft16<false>(v);
#pragma unroll
        for (int q = 0; q < 16; ++q) scratch[(h * 16 + q) * 256] = v[q];
      }
    }
    for (int f = 0; f < n_filters; ++f) {
      const float2 *kp = (const float2 *)a.kperm + (size_t)f * 8192 + t;
      // (stage 3,) spectrum multiply, first inverse stage (DFT16 over qc, twiddle conj w_256^(c qb)); the filter
      // spectrum is requested first so that its latency hides behind the shared-memory reads and the DFT
      {
        float2 v0[16], v1[16];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float2 *v = h ? v1 : v0;
          float2 k[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) k[q] = __ldg(kp + (h * 16 + q) * 256);
          if (BANK) {
#pragma unroll
            for (int q = 0; q < 16; ++q) v[q] = scratch[(h * 16 + q) * 256];
          } else {
            load16(v, h ? H1 : H0, p0);
            dft16<false>(v);
          }
#pragma unroll
          for (int q = 0; q < 8; ++q) v[q] = cmulf(v[q], k[q]);
#pragma unroll
          for (int q = 8; q < 16; ++q) v[q] = cmulf(v[q], __ldg(kp + (h * 16 + q) * 256));
          dft16<true>(v);
        }
#pragma unroll
        for (int c = 1; c < 16; ++c) {
          const float2 w = tab[kT2 + 16 * c + qb];
          v0[c] = cmulw<true>(v0[c], w);
          v1[c] = cmulw<true>(v1[c], w);
        }
        store16(v0, H0, p0);
        store16(v1, H1, p0);
      }
      __syncwarp();
      {   // second inverse stage: thread t = 16 qa + c, DFT16 over qb, twiddle conj w_4096^(qa (16 b + c))
        const int qa = t >> 4, c = t & 15;
        float2 *B = H0 + pos3(qa, 0, c);
        const float2 *T = tab + kT1 + 256 * qa + c;
        float2 e[16], o[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) { e[q] = B[pos3(0, q, 0)]; o[q] = B[pos3(0, q, 0) + kHalfPad]; }
        dft16<true>(e);
        dft16<true>(o);
#pragma unroll
        for (int b = 0; b < 16; ++b) {         // (w_4096^(qa (16 b + c)) is 1 only for qa = 0: no row to skip here)
          const float2 w = T[16 * b];
          B[pos3(0, b, 0)] = cmulw<true>(e[b], w);
          B[pos3(0, b, 0) + kHalfPad] = cmulw<true>(o[b], w);
        }
      }
      __syncthreads();
      {   // third inverse stage of both halves (thread t = 16 b + c, DFT16 over qa) and the overlap-save combine
        const float2 *B = H0 + pos3(0, t >> 4, t & 15);
        float2 z[16], v[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) z[q] = B[pos3(q, 0, 0) + kHalfPad];
        dft16<true>(z);
        const float2 wt = tab[kT8 + t];
#pragma unroll
        for (int q = 0; q < 16; ++q) { z[q] = cmulw<true>(z[q], root8k(wt, q)); v[q] = B[pos3(q, 0, 0)]; }
        dft16<true>(v);
        float2 *o = (float2 *)a.out + (size_t)f * a.out_stride + (size_t)blk * kHalf + t;
#pragma unroll
        for (int q = 0; q < 16; ++q) o[256 * q] = csubf(v[q], z[q]);
      }
      if (BANK && f + 1 < n_filters) __syncthreads();   // the next filter's first-stage stores; the next BLOCK waits inside dif_stage1
    }
  }
}

}  // namespace

int conv8k_grid(size_t n_blocks, int *grid) {      // CTAs launch_conv8k will use (the bank's scratch is 64 KB per CTA)
  int resident = 0;
  const int rc = kernel_setup((const void *)conv8k_kernel<true>, kT, kSmemBytes, &resident);
  *grid = (int)(n_blocks < (size_t)resident ? n_blocks : (size_t)resident);
  return rc;
}

int launch_conv8k(const FilterArgs &a, size_t n_blocks, cudaStream_t st) {
  if (n_blocks == 0) return SDRG_OK;
  if (n_blocks > 0x7fffffffull) return set_error(SDRG_ERR_ARG, "FilterNode: too many blocks in one call");
  if (a.n_filters > 1 && !a.spec) return set_error(SDRG_ERR_RUNTIME, "FilterNode: the filter bank needs its spectrum scratch");
  return launch_persistent("conv8k_kernel", a.n_filters > 1 ? conv8k_kernel<true> : conv8k_kernel<false>, n_blocks, kT, kSmemBytes, st, a, (int)n_blocks);
}

}  // namespace sdrg

// iqbb_int_common.cuh -- the integer arithmetic of IQBaseBand<int16_t> / <int8_t>, written once for every kernel that
// computes it: the single-channel kernels (iqbb_kernels.cu, iqbb_warp_kernels.cu) and the channel bank (bank_kernels.cu).
//
// Per sample (src/baseband.hh:198-236, src/freqshift.hh:58-74): load_sample -> fir_fixed / fir_smem -> fir_result
// (>> fir_shift, int8 narrowing) -> nco_mix (LUT product, >> 16 or int8's narrow / >> 8 / narrow).  Every sum is taken
// in Z/2^32, which is associative, so the kernels' different evaluation orders are all bit-exact.  The kernels differ
// only in how they stage samples, form the LUT index and sum windows.
#pragma once
#include "iqbb_kernels.cuh"

namespace sdrg {

struct IqbbTaps { int4 t[32]; };   // Gauss-form taps {kr, ki - kr, kr + ki, 0} in the kernel's parameter (constant) bank

namespace {

constexpr int kR = kIqbbPerThread;

__device__ __forceinline__ int pad32(int i) { return i + (i >> 5); }   // 4-byte elements, 8 per thread

__device__ __forceinline__ void unpack16(uint32_t v, int &re, int &im) {
  re = (int)(short)(v & 0xffffu);
  im = ((int)v) >> 16;
}

// window bookkeeping (call-relative sample index i): q(i) = r0 + i - (first && i>0); slot = q/ss.
// n <= 2^30 and r0 < ss <= 2^30, so q and every window bound fit in 32 bits (the 64-bit division
// this used to be cost more than the FIR itself).
struct WindowGrid {
  uint32_t ss, r0, first;
  __device__ __forceinline__ uint32_t q(uint32_t i) const { return r0 + i - ((first && i > 0) ? 1u : 0u); }
  __device__ __forceinline__ uint32_t slot(uint32_t i) const { return q(i) / ss; }
  __device__ __forceinline__ int64_t begin(uint32_t s) const {
    return s == 0 ? 0 : (int64_t)(uint32_t)(s * ss - r0 + first);
  }
  __device__ __forceinline__ int64_t end(uint32_t s) const {
    return (int64_t)(uint32_t)((s + 1) * ss - r0 + first);
  }
};

// ---- samples ----------------------------------------------------------------------------------------
// One input sample as packed (re | im << 16) int16 pair.  fmt 0: complex<int16_t> as is; fmt 2/3:
// AutoCast< complex<int16_t> > fused into the load (src/autocast.hh:187-204): complex uint8 read
// through an int8_t pointer, (v - 127) << 8 (reference quirk), resp. complex int8, v << 8.
__device__ __forceinline__ uint32_t load_cs16(const void *base, int64_t idx, uint32_t fmt) {
  if (fmt == 0) return ((const uint32_t *)base)[idx];
  if (fmt == 4) return (uint32_t)((const uint16_t *)base)[idx];      // real input: imaginary part 0
  const char2 s = ((const char2 *)base)[idx];
  const int bias = fmt == 2 ? 127 : 0;
  const uint32_t re = (uint32_t)(uint16_t)(int16_t)(((int)s.x - bias) << 8);
  const uint32_t im = (uint32_t)(uint16_t)(int16_t)(((int)s.y - bias) << 8);
  return re | (im << 16);
}

// The sample at call-relative index i: from the history for i < 0 (the last Hh samples of the previous calls; anything
// older is zero), zero from n on.  int16 (IS_S8 false): the formats of load_cs16.  int8: complex<int8_t> sign-extended,
// or fmt 5, real int8 (BaseBand<int8_t>) with imaginary part 0.
template <bool IS_S8>
__device__ __forceinline__ uint32_t load_sample(const void *x, const void *hist, int64_t i, int Hh, uint32_t n, uint32_t fmt) {
  if (!IS_S8) {
    uint32_t v = 0;
    if (i < 0) { if (Hh + i >= 0) v = load_cs16(hist, Hh + i, fmt); }
    else if (i < (int64_t)n) v = load_cs16(x, i, fmt);
    return v;
  }
  if (fmt == 5) {
    signed char s = 0;
    if (i < 0) { if (Hh + i >= 0) s = ((const signed char *)hist)[Hh + i]; }
    else if (i < (int64_t)n) s = ((const signed char *)x)[i];
    return (uint32_t)(uint16_t)(int16_t)s;
  }
  char2 s = make_char2(0, 0);
  if (i < 0) { if (Hh + i >= 0) s = ((const char2 *)hist)[Hh + i]; }
  else if (i < (int64_t)n) s = ((const char2 *)x)[i];
  return ((uint32_t)(uint16_t)(int16_t)s.x) | (((uint32_t)(uint16_t)(int16_t)s.y) << 16);
}

// ---- FIR over a register window of 8 outputs ------------------------------------------------------------
// Output r of the 8 is sum_t k[t] x[r + t].  Taps are in Gauss form {kr, ki - kr, kr + ki, 0}: t1 = kr (xr + xi),
// t2 = (ki - kr) xr, t3 = (kr + ki) xi, re = t1 - t3, im = t1 + t2 (ring identities, hence exact mod 2^32).  The window
// holds 8 unpacked samples; slot u is refilled with sample u + 8 once tap u has been applied.
// `z` is an addend that is always 0: IqbbAccumArgs::zero in the per-warp kernel, 0u elsewhere.
enum FirForm {
  kFirComplex,    // complex taps on complex samples: three multiplies per tap
  kFirRealIn,     // complex taps on real samples (x_im = 0, BaseBand<int16_t>): re = sum kr x, im = re + sum (ki - kr) x
  kFirRealTaps,   // real taps (k_im = 0) on complex samples: re = sum kr xr, im = sum kr xi
};

template <int FORM>
__device__ __forceinline__ void fir_load(int &wr, int &wi, int &ws, uint32_t v, uint32_t z) {
  unpack16(v, wr, wi);
  if (FORM == kFirComplex) ws = (int)((uint32_t)wr + (uint32_t)wi + z);
}

template <int FORM>
__device__ __forceinline__ void fir_tap(uint32_t (&A1)[kR], uint32_t (&A2)[kR], uint32_t (&A3)[kR], const int4 c,
                                        const int (&wr)[kR], const int (&wi)[kR], const int (&ws)[kR], const int u) {
#pragma unroll
  for (int r = 0; r < kR; ++r) {
    const int s = (r + u) & (kR - 1);
    if (FORM == kFirRealIn) {
      A1[r] += (uint32_t)c.x * (uint32_t)wr[s];
      A2[r] += (uint32_t)c.y * (uint32_t)wr[s];
    } else if (FORM == kFirRealTaps) {
      A1[r] += (uint32_t)c.x * (uint32_t)wr[s];
      A2[r] += (uint32_t)c.x * (uint32_t)wi[s];
    } else {
      A1[r] += (uint32_t)c.x * (uint32_t)ws[s];
      A2[r] += (uint32_t)c.y * (uint32_t)wr[s];
      A3[r] += (uint32_t)c.z * (uint32_t)wi[s];
    }
  }
}

// LP taps known at compile time (in the constant bank or in shared memory), samples w[0 .. LP + 6] in registers.
template <int LP, int FORM>
__device__ __forceinline__ void fir_fixed(const uint32_t *w, const int4 *taps, uint32_t z,
                                          uint32_t (&A1)[kR], uint32_t (&A2)[kR], uint32_t (&A3)[kR]) {
  int wr[kR], wi[kR], ws[kR];
#pragma unroll
  for (int c = 0; c < kR; ++c) {
    A1[c] = A2[c] = A3[c] = 0u;
    fir_load<FORM>(wr[c], wi[c], ws[c], w[c], z);
  }
#pragma unroll
  for (int t = 0; t < LP; ++t) {
    fir_tap<FORM>(A1, A2, A3, taps[t], wr, wi, ws, t);
    if (t + 1 < LP) fir_load<FORM>(wr[t & (kR - 1)], wi[t & (kR - 1)], ws[t & (kR - 1)], w[t + kR], z);
  }
}

// Lp taps at run time, complex form; taps tp[0 .. Lp) and samples xs[pad32(ob + c)] in shared memory.
__device__ __forceinline__ void fir_smem(const uint32_t *xs, int ob, const int4 *tp, int Lp,
                                         uint32_t (&A1)[kR], uint32_t (&A2)[kR], uint32_t (&A3)[kR]) {
  int wr[kR], wi[kR], ws[kR];
#pragma unroll
  for (int c = 0; c < kR; ++c) {
    A1[c] = A2[c] = A3[c] = 0u;
    fir_load<kFirComplex>(wr[c], wi[c], ws[c], xs[pad32(ob + c)], 0u);
  }
  for (int t0 = 0; t0 < Lp; t0 += kR) {
#pragma unroll
    for (int u = 0; u < kR; ++u) {
      const int t = t0 + u;
      if (t < Lp) {
        fir_tap<kFirComplex>(A1, A2, A3, tp[t], wr, wi, ws, u);
        fir_load<kFirComplex>(wr[u], wi[u], ws[u], xs[pad32(ob + t + kR)], 0u);
      }
    }
  }
}

// int8: intermediate results are complex<int16_t>
__device__ __forceinline__ void narrow16(int &yr, int &yi) { yr = (int)(short)yr; yi = (int)(short)yi; }

// Output r of the FIR from its sums A1..A3, shifted right by `shift` (14 IQBaseBand, 16 BaseBand).  int8: narrowed to
// complex<int16_t> on the call; real8 (BaseBand<int8_t>): `res` is complex<int16_t>, so the sum wraps at 16 bits before
// the shift as well.
template <bool IS_S8, int FORM>
__device__ __forceinline__ void fir_result(uint32_t A1, uint32_t A2, uint32_t A3, uint32_t z, uint32_t shift, bool real8,
                                           int &yr, int &yi) {
  if (FORM == kFirRealTaps) { yr = ((int)A1) >> shift; yi = ((int)A2) >> shift; }
  else if (real8) { yr = ((int)(short)(A1 - A3 + z)) >> shift; yi = ((int)(short)(A1 + A2 + z)) >> shift; }
  else { yr = ((int)(A1 - A3 + z)) >> shift; yi = ((int)(A1 + A2 + z)) >> shift; }
  if (IS_S8) narrow16(yr, yi);
}

// The NCO mix with LUT entry l (freqshift.hh:67): int16 takes the product >> 16; int8 narrows the product to int16,
// shifts it by 8 and narrows again.
template <bool IS_S8>
__device__ __forceinline__ void nco_mix(int2 l, int &yr, int &yi) {
  const uint32_t pr = (uint32_t)l.x * (uint32_t)yr - (uint32_t)l.y * (uint32_t)yi;
  const uint32_t pi = (uint32_t)l.x * (uint32_t)yi + (uint32_t)l.y * (uint32_t)yr;
  if (IS_S8) { yr = (int)(short)(((int)(short)pr) >> 8); yi = (int)(short)(((int)(short)pi) >> 8); }
  else { yr = ((int)pr) >> 16; yi = ((int)pi) >> 16; }
}

// ---- prologues: zero the next call's accumulators, roll the history ------------------------------------
// (k0: this thread's first index, threadIdx.x)
template <typename Sample>
__device__ __forceinline__ void roll_history(const void *x, const void *hist_in, void *hist_out, int64_t n, int64_t H, int64_t k0) {
  for (int64_t k = k0; k < H; k += blockDim.x) {
    const int64_t i = n - H + k;                         // call-relative source index
    ((Sample *)hist_out)[k] = (i >= 0) ? ((const Sample *)x)[i] : ((const Sample *)hist_in)[H + i];
  }
}

template <typename Sample, typename Acc>
__device__ __forceinline__ void prologue(const IqbbAccumArgs &a) {
  Acc *nxt = (Acc *)a.acc_next;
  for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < a.zero_next; k += gridDim.x * blockDim.x) {
    Acc zero; zero.x = 0; zero.y = 0;
    nxt[k] = zero;
  }
  if (blockIdx.x == 0) {
    const int64_t H = a.hist_len, n = a.n;
    if (a.in_fmt == 5) roll_history<signed char>(a.x, a.hist_in, a.hist_out, n, H, threadIdx.x);      // real int8: one byte per sample
    else if (sizeof(Sample) == 4 && a.in_fmt != 0) roll_history<char2>(a.x, a.hist_in, a.hist_out, n, H, threadIdx.x);   // fused AutoCast: raw 8-bit pairs
    else roll_history<Sample>(a.x, a.hist_in, a.hist_out, n, H, threadIdx.x);
  }
}

// channel bank: the first zero_next accumulators of every channel; Sample is char2 (int8) or uint32_t (packed int16)
template <typename Sample>
__device__ __forceinline__ void bank_prologue(const BankAccumArgs &a, const int tid) {
  int2 *nxt = (int2 *)a.acc_next;
  const size_t total = (size_t)a.zero_next * a.channels;
  const size_t stride = (size_t)gridDim.x * gridDim.y * blockDim.x;
  for (size_t k = ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * blockDim.x + tid; k < total; k += stride)
    nxt[(k / a.zero_next) * a.acc_stride + (k % a.zero_next)] = make_int2(0, 0);
  if (blockIdx.x == 0 && blockIdx.y == 0) roll_history<Sample>(a.x, a.hist_in, a.hist_out, a.n, a.hist_len, tid);
}

__device__ __forceinline__ void cp_async4(void *smem_dst, const void *gmem_src) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gmem_src) : "memory");
}

}  // namespace

// iqbb_warp_kernels.cu: barrier-free per-warp variant of the fixed-tap integer kernel (sub_sample >= 16, <= 32 taps).
// `kind`: 0 complex taps (Gauss form), 3 real taps (k_im == 0 for every tap), 4 real taps symmetric about the middle
// of an even count.  Returns SDRG_OK after launching, or -1 if there is no instantiation (the caller falls back).
int launch_iqbb_accum_warp(int scalar, const IqbbAccumArgs &a, const IqbbTaps &taps, int lp, cudaStream_t st);

}  // namespace sdrg

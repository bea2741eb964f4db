// fft8k_stages.cuh -- the in-place radix-16 stages shared by the 8192 / 4096-point plan kernels (fft8k_kernels.cu) and the
// block-4096 convolution (conv8k_kernels.cu); see fft8k_kernels.cu for the method and the index algebra.  A translation
// unit that defines SDRG_FFT_PACKED before this include gets the packed-FP32 flavour of the butterflies (fft_device.cuh).
#pragma once
#include "fft_kernels.cuh"
#include "fft_device.cuh"
#include "launch.cuh"

#include <cmath>
#include <vector>

namespace sdrg {
namespace {


constexpr int kT = 256;                       // threads per CTA
constexpr int kHalf = 4096;
// shared-memory position of element i of a half: two pads per 16 and two more per 256, so that lanes striding
// by 1 (stages 1, 2: 64-bit accesses) or by 256 (stage 3: 128-bit accesses of 16 consecutive elements, whose
// first position 290 qa + 18 qb is even, i.e. 16-byte aligned) all fall on distinct banks
__device__ __forceinline__ int pos(int i) { return i + 2 * (i >> 4) + 2 * (i >> 8); }
// the same written per digit, i = 256 A + 16 B + C: every access below is then [thread base + immediate]
__host__ __device__ constexpr int pos3(int A, int B, int C) { return 290 * A + 18 * B + C; }
constexpr int kHalfPad = kHalf + 2 * (kHalf / 16) + 2 * (kHalf / 256) + 8;

// table layout (float2 entries, forward sign exp(-2 pi i k / n))
constexpr int kT1 = 0;                        // [q][u]  w_4096^(q u), q < 16, u < 256
constexpr int kT2 = kT1 + 16 * 256;           // [q][c]  w_256^(q c),  q < 16, c < 16
constexpr int kT8 = kT2 + 16 * 16;            // [u]     w_8192^u,     u < 256
constexpr int kTabLen = kT8 + 256;
constexpr size_t kSmemBytes = (size_t)(2 * kHalfPad + kTabLen) * sizeof(float2);

__device__ __forceinline__ void load_tables(float2 *tab, const float2 *__restrict__ g) {
  for (int i = threadIdx.x; i < kTabLen; i += kT) tab[i] = g[i];
}

// w_8192^(256 a + t) = w_32^a . w_8192^t; the 16 values of w_32^a are immediates
__device__ __forceinline__ float2 root8k(const float2 wt, const int a) {
  constexpr float c32[16] = {1.000000000e+00f, 9.807852804e-01f, 9.238795325e-01f, 8.314696123e-01f, 7.071067812e-01f, 5.555702330e-01f,
                             3.826834324e-01f, 1.950903220e-01f, 0.0f, -1.950903220e-01f, -3.826834324e-01f, -5.555702330e-01f,
                             -7.071067812e-01f, -8.314696123e-01f, -9.238795325e-01f, -9.807852804e-01f};
  constexpr float s32[16] = {0.000000000e+00f, 1.950903220e-01f, 3.826834324e-01f, 5.555702330e-01f, 7.071067812e-01f, 8.314696123e-01f,
                             9.238795325e-01f, 9.807852804e-01f, 1.0f, 9.807852804e-01f, 9.238795325e-01f, 8.314696123e-01f,
                             7.071067812e-01f, 5.555702330e-01f, 3.826834324e-01f, 1.950903220e-01f};
  if (a == 0) return wt;
  if (a == 8) return make_float2(wt.y, -wt.x);
  // wt * (c - i s)
  return mulw16<false>(wt, c32[a], s32[a]);
}

__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// ---- the decimation-in-frequency pass (forward; INV conjugates every root => unnormalised backward DFT) ----
// Both halves go through a stage together: twice the independent work per thread, and every table twiddle is
// loaded once for the two butterflies that need it.
// stage 1: e[a] = u0[256 a + t], o[a] = u1[256 a + t] on entry (thread t = 16 b + c)
// The CTA barrier that frees the buffers (everybody has finished READING the previous item's last stage) sits between
// the butterflies and the stores, so the global-load latency and the first DFTs of an item overlap the tail of the
// previous one.
template <bool INV>
__device__ __forceinline__ void dif_stage1(float2 *e, float2 *o, float2 *H0, const float2 *tab, const int t) {
  const int pt = pos3(0, t >> 4, t & 15);
  dft16<INV>(e);
  dft16<INV>(o);
  __syncthreads();
  H0[pt] = e[0];
  H0[pt + kHalfPad] = o[0];
#pragma unroll
  for (int q = 1; q < 16; ++q) {
    const float2 w = tab[kT1 + 256 * q + t];
    H0[pt + pos3(q, 0, 0)] = cmulw<INV>(e[q], w);
    H0[pt + pos3(q, 0, 0) + kHalfPad] = cmulw<INV>(o[q], w);
  }
}
// stage 2: thread t = 16 qa + c works on positions 256 qa + 16 b + c of both halves
template <bool INV>
__device__ __forceinline__ void dif_stage2(float2 *H0, const float2 *tab, const int t) {
  const int c = t & 15;
  float2 *B = H0 + pos3(t >> 4, 0, c);
  float2 e[16], o[16];
#pragma unroll
  for (int b = 0; b < 16; ++b) { e[b] = B[pos3(0, b, 0)]; o[b] = B[pos3(0, b, 0) + kHalfPad]; }
  dft16<INV>(e);
  dft16<INV>(o);
  B[0] = e[0];
  B[kHalfPad] = o[0];
#pragma unroll
  for (int q = 1; q < 16; ++q) {
    const float2 w = tab[kT2 + 16 * q + c];
    B[pos3(0, q, 0)] = cmulw<INV>(e[q], w);
    B[pos3(0, q, 0) + kHalfPad] = cmulw<INV>(o[q], w);
  }
}
// stage 3: thread t = qa + 16 qb reads the 16 consecutive positions of 256 qa + 16 qb + c (128-bit loads);
// on return v[qc] = U[t + 256 qc]
__device__ __forceinline__ int stage3_pos(const int t) { return pos3(t & 15, t >> 4, 0); }
// The convolution does not care in which order the bins come out, so its stage 3 uses thread t = 16 qa + qb instead:
// the 16 positions it reads were all written (stage 2, threads 16 qa + c) by lanes of the SAME warp, and the inverse
// mirror holds too -- two of the five CTA barriers per block become __syncwarp().  Bins held: qa + 16 qb + 256 qc.
__device__ __forceinline__ int stage3_pos_conv(const int t) { return pos3(t >> 4, t & 15, 0); }
__device__ __forceinline__ void load16(float2 *v, const float2 *H, const int p0) {
  const float4 *h4 = (const float4 *)(H + p0);
#pragma unroll
  for (int k = 0; k < 8; ++k) { const float4 q = h4[k]; v[2 * k] = make_float2(q.x, q.y); v[2 * k + 1] = make_float2(q.z, q.w); }
}
__device__ __forceinline__ void store16(const float2 *v, float2 *H, const int p0) {
  float4 *h4 = (float4 *)(H + p0);
#pragma unroll
  for (int k = 0; k < 8; ++k) h4[k] = make_float4(v[2 * k].x, v[2 * k].y, v[2 * k + 1].x, v[2 * k + 1].y);
}


}  // namespace
}  // namespace sdrg

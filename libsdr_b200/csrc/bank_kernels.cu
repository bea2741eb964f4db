// bank_kernels.cu -- a bank of IQBaseBand<int16_t>/<int8_t>/<float> channels on ONE input stream
// (BASELINE configs 4/5: 256..2048 channels with independent NCO offsets on a 100 MS/s stream).
//
// Every channel is an independent IQBaseBand (src/baseband.hh:198-236) fed the same buffers; the
// arithmetic per channel is iqbb_int_common.cuh's (load_sample, fir_smem / fir_fixed, fir_result,
// nco_mix, bit-exact), as in the single-channel kernels.  What changes is
// the data movement: a CTA stages one 2048-sample input tile (+ halo) in shared memory ONCE and
// loops over a group of channels (taps of the whole group preloaded in shared memory), so the
// input is read from HBM once per channel group instead of once per channel; the work is purely
// integer-multiply bound (C x (3L+7) IMAD per 4-byte sample), HBM traffic is negligible.
// With sub-sampling >= 2048 (the bank configs use 2083) a thread's 8 consecutive outputs and a
// warp's 256 touch at most two windows, so window sums are formed in registers and reduced with
// REDUX.SUM -- no shared-memory staging and no CTA barrier inside the channel loop.
// IQBaseBand<float> channels take the folded kernel further below (bank_fold_f32_kernel).
#include "iqbb_int_common.cuh"
#include "iqbb_finalize.cuh"
#include "iqbb_fold_common.cuh"

namespace sdrg {
namespace {

constexpr int kT = kIqbbThreads, kTile = kIqbbTile;
constexpr unsigned kFull = 0xffffffffu;

template <bool IS_S8>
__global__ void __launch_bounds__(kT) bank_accum_kernel(const BankAccumArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31;
  const int H = (int)a.hist_len, Lp = (int)a.taps_len;
  const int n_xs = kTile + H + 8;
  const int c0 = blockIdx.y * a.group;
  const int nch = min((int)a.group, (int)a.channels - c0);
  int4 *tp = (int4 *)smem_raw;                                   // group x Lp
  int2 *lut = (int2 *)(tp + (size_t)a.group * Lp);               // 128
  uint32_t *xs = (uint32_t *)(lut + 128);                        // pad32(n_xs)+1

  if (IS_S8) bank_prologue<char2>(a, tid); else bank_prologue<uint32_t>(a, tid);

  const int64_t tile_base = (int64_t)blockIdx.x * kTile;
  for (int k = tid; k < nch * Lp; k += kT) tp[k] = ((const int4 *)a.taps)[(size_t)c0 * Lp + k];
  if (tid < 128) lut[tid] = ((const int2 *)a.lut)[tid];
  for (int k = tid; k < n_xs; k += kT) xs[pad32(k)] = load_sample<IS_S8>(a.x, a.hist_in, tile_base - H + k, H, a.n, 0u);
  __syncthreads();

  // window geometry of this thread's 8 outputs (identical for every channel)
  const int ob = tid * kR;
  const uint32_t i0 = (uint32_t)tile_base + (uint32_t)ob;        // call-relative index of output 0
  const uint32_t tile_hi = (uint32_t)min((int64_t)a.n, tile_base + kTile);
  const WindowGrid g{a.ss, a.r0, a.first};
  const uint32_t slot_a = g.slot(i0);
  const uint32_t bnd = (uint32_t)g.end(slot_a);                  // first call-relative index of slot_a + 1
  const uint32_t slot_w = g.slot((uint32_t)tile_base + (uint32_t)((tid & ~31) * kR));   // warp-uniform
  // which of this thread's 8 outputs go to the upper of the warp's two windows (bit r), and which exist
  uint32_t upper_mask = 0, valid_mask = 0;
#pragma unroll
  for (int r = 0; r < kR; ++r) {
    const uint32_t i = i0 + r;
    const bool up = (i >= bnd) ? (slot_a + 1 != slot_w) : (slot_a != slot_w);
    upper_mask |= (up ? 1u : 0u) << r;
    valid_mask |= ((i < tile_hi) ? 1u : 0u) << r;
  }

  for (int ch = 0; ch < nch; ++ch) {
    const int c = c0 + ch;
    uint32_t A1[kR], A2[kR], A3[kR];
    fir_smem(xs, ob, tp + ch * Lp, Lp, A1, A2, A3);
    const uint32_t inc = a.inc[c] & 0x7fffu;
    const bool nco = a.inc[c] != 0, neg = (a.neg[c] != 0);
    const uint32_t phase0 = (a.consumed15 * inc) & 0x7fffu;      // (consumed * inc) mod 32768
    uint32_t lo_r = 0, lo_i = 0, hi_r = 0, hi_i = 0;             // sums for slot_w and slot_w + 1
#pragma unroll
    for (int r = 0; r < kR; ++r) {
      int yr, yi;
      fir_result<IS_S8, kFirComplex>(A1[r], A2[r], A3[r], 0u, 14, false, yr, yi);
      if (nco) {
        const uint32_t ph = (phase0 + (i0 + r) * inc) & 0x7fffu;
        uint32_t idx = ph >> 8;
        if (neg) idx = 127u - idx;
        nco_mix<IS_S8>(lut[idx], yr, yi);
      }
      if ((valid_mask >> r) & 1u) {
        if ((upper_mask >> r) & 1u) { hi_r += (uint32_t)yr; hi_i += (uint32_t)yi; } else { lo_r += (uint32_t)yr; lo_i += (uint32_t)yi; }
      }
    }
    lo_r = __reduce_add_sync(kFull, lo_r); lo_i = __reduce_add_sync(kFull, lo_i);
    hi_r = __reduce_add_sync(kFull, hi_r); hi_i = __reduce_add_sync(kFull, hi_i);
    if (lane == 0) {
      int *acc = (int *)a.acc_cur + 2 * ((size_t)c * a.acc_stride + slot_w);
      if (lo_r | lo_i) { atomicAdd(acc, (int)lo_r); atomicAdd(acc + 1, (int)lo_i); }
      if (hi_r | hi_i) { atomicAdd(acc + 2, (int)hi_r); atomicAdd(acc + 3, (int)hi_i); }
    }
  }
}

// ---- compile-time tap count ---------------------------------------------------------------------------
// As in iqbb_accum_int_fixed_kernel: the tile is staged unpadded, every thread pulls its LP+7 packed
// samples into registers ONCE (128-bit shared loads) and keeps them for ALL channels of the group;
// the channel loop then consists of broadcast tap loads, one unpack per tap step and IMADs.
template <int LP, bool IS_S8>
__global__ void __launch_bounds__(kT) bank_accum_fixed_kernel(const BankAccumArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int H = LP - 1;
  constexpr int NV = (LP + 7 + 3) / 4;
  constexpr int n_xs = kTile + 4 * NV + 8;
  const int tid = threadIdx.x, lane = tid & 31;
  const int Ls = (int)a.taps_len, pad = LP - Ls;                 // stored taps per channel; zero taps in front
  const int c0 = blockIdx.y * a.group;
  const int nch = min((int)a.group, (int)a.channels - c0);
  uint32_t *xs = (uint32_t *)smem_raw;                           // n_xs (16-byte aligned)
  int4 *tp = (int4 *)(xs + ((n_xs + 3) & ~3));                   // group x LP
  int2 *lut = (int2 *)(tp + (size_t)a.group * LP);               // 128

  if (IS_S8) bank_prologue<char2>(a, tid); else bank_prologue<uint32_t>(a, tid);

  const int64_t tile_base = (int64_t)blockIdx.x * kTile;
  for (int k = tid; k < nch * LP; k += kT) {
    const int ch = k / LP, t = k - ch * LP;
    tp[k] = t < pad ? make_int4(0, 0, 0, 0) : ((const int4 *)a.taps)[(size_t)(c0 + ch) * Ls + (t - pad)];
  }
  if (tid < 128) lut[tid] = ((const int2 *)a.lut)[tid];
  const int Hh = (int)a.hist_len;
  for (int k = tid; k < n_xs; k += kT) xs[k] = load_sample<IS_S8>(a.x, a.hist_in, tile_base - H + k, Hh, a.n, 0u);
  __syncthreads();

  uint32_t w[4 * NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const uint4 q = ((const uint4 *)xs)[tid * 2 + v];
    w[4 * v] = q.x; w[4 * v + 1] = q.y; w[4 * v + 2] = q.z; w[4 * v + 3] = q.w;
  }

  const int ob = tid * kR;
  const uint32_t i0 = (uint32_t)tile_base + (uint32_t)ob;
  const uint32_t tile_hi = (uint32_t)min((int64_t)a.n, tile_base + kTile);
  const WindowGrid g{a.ss, a.r0, a.first};
  const uint32_t slot_a = g.slot(i0);
  const uint32_t bnd = (uint32_t)g.end(slot_a);                  // first index of slot_a + 1
  const uint32_t slot_w = g.slot((uint32_t)tile_base + (uint32_t)((tid & ~31) * kR));
  // which of this thread's 8 outputs go to the upper of the warp's two windows (bit r), and which exist
  uint32_t upper_mask = 0, valid_mask = 0;
#pragma unroll
  for (int r = 0; r < kR; ++r) {
    const uint32_t i = i0 + r;
    const bool up = (i >= bnd) ? (slot_a + 1 != slot_w) : (slot_a != slot_w);
    upper_mask |= (up ? 1u : 0u) << r;
    valid_mask |= ((i < tile_hi) ? 1u : 0u) << r;
  }

  for (int ch = 0; ch < nch; ++ch) {
    const int c = c0 + ch;
    uint32_t A1[kR], A2[kR], A3[kR];
    fir_fixed<LP, kFirComplex>(w, tp + ch * LP, 0u, A1, A2, A3);
    const uint32_t inc = a.inc[c] & 0x7fffu;
    const bool nco = a.inc[c] != 0;
    const uint32_t negx = a.neg[c] ? 127u : 0u;                  // idx = 127 - idx  <=>  idx ^ 127 for idx in 0..127
    uint32_t ph = (a.consumed15 * inc + i0 * inc) & 0x7fffu;
    uint32_t lo_r = 0, lo_i = 0, hi_r = 0, hi_i = 0;
#pragma unroll
    for (int r = 0; r < kR; ++r) {
      int yr, yi;
      fir_result<IS_S8, kFirComplex>(A1[r], A2[r], A3[r], 0u, 14, false, yr, yi);
      if (nco) {
        const int2 l = lut[(ph >> 8) ^ negx];
        ph = (ph + inc) & 0x7fffu;
        nco_mix<IS_S8>(l, yr, yi);
      }
      if ((valid_mask >> r) & 1u) {
        if ((upper_mask >> r) & 1u) { hi_r += (uint32_t)yr; hi_i += (uint32_t)yi; } else { lo_r += (uint32_t)yr; lo_i += (uint32_t)yi; }
      }
    }
    lo_r = __reduce_add_sync(kFull, lo_r); lo_i = __reduce_add_sync(kFull, lo_i);
    hi_r = __reduce_add_sync(kFull, hi_r); hi_i = __reduce_add_sync(kFull, hi_i);
    if (lane == 0) {
      int *acc = (int *)a.acc_cur + 2 * ((size_t)c * a.acc_stride + slot_w);
      if (lo_r | lo_i) { atomicAdd(acc, (int)lo_r); atomicAdd(acc + 1, (int)lo_i); }
      if (hi_r | hi_i) { atomicAdd(acc + 2, (int)hi_r); atomicAdd(acc + 3, (int)hi_i); }
    }
  }
}

template <int LP, bool IS_S8>
int launch_bank_fixed(const BankAccumArgs &a, dim3 grid, cudaStream_t st) {
  constexpr int NV = (LP + 7 + 3) / 4;
  constexpr int n_xs = kTile + 4 * NV + 8;
  const size_t smem = sizeof(uint32_t) * ((n_xs + 3) & ~3) + sizeof(int4) * (size_t)a.group * LP + sizeof(int2) * 128;
  return launch("bank_accum_fixed_kernel", bank_accum_fixed_kernel<LP, IS_S8>, grid, kT, smem, st, a);
}

template <bool IS_S8>
int dispatch_bank_fixed(int lp, const BankAccumArgs &a, dim3 grid, cudaStream_t st) {
  return dispatch(lp, int_range<2, 32, 2>{}, [&](auto LP) { return launch_bank_fixed<LP, IS_S8>(a, grid, st); },
                  [&] { return set_error(SDRG_ERR_RUNTIME, "no fixed-tap bank kernel for %d taps", lp); });
}

// ---- float bank: the folded weights, one channel per lane ----------------------------------------------
// IQBaseBand<float> is linear, so FIR -> NCO -> boxcar folds into one weight per input sample
// (iqbb_fold_kernels.cu): with the channel's phase phi_p = 256 a + r at sample p, a sample whose L
// outputs all fall in its own window weighs G_c(p) = A(a) U_c(r, 0).  The last L-1 samples of a window
// feed outputs of the next one; that part,
//     sent = sum_{j=0}^{L-2} c(b+j) sum_{t=0}^{L-2-j} k[t] x[b+j-(L-1)+t]      (b = first sample of the next window),
// is computed directly from the taps and the LUT at every window end, moved out of the window and into
// the next one.  That costs L(L-1)/2 complex FMA per channel and window, at most L/2 per sample since
// ss >= 256 >= L (the direct form costs L), and 0.05 per sample at 15 taps and ss 2083; no U(r, e) table.
//
// Mapping: a CTA owns 32 channels (the lanes) and kFbSpan consecutive samples, a warp kFbWarpSpan of
// them, staged kFbChunk at a time into a warp-private buffer.  Every lane walks the same samples in
// order, so x[p] is a broadcast (one LDS.128 per two samples).  The weight costs two 8-byte shared loads:
// U_c(r, 0) stored [r][lane] (lanes hit distinct bank pairs at any r) and A(a) replicated 16 times,
// [sign][a][copy], lane l reading copy l mod 16 (each half-warp conflict free at any a).  The phase is
// kept shifted left by 8 bits, so both addresses are one mask-or (and a shift for A) of it.
// Window sums stay in registers until the window ends, then one RED.ADD per component and channel.
constexpr int kFbWarps = kT / 32;
constexpr int kFbChunk = 256;
constexpr int kFbWarpSpan = 8 * kFbChunk;
constexpr int kFbSpan = kFbWarps * kFbWarpSpan;
constexpr size_t kFbSmem = (size_t)(256 * 32 + 2 * 128 * 16 + kFbWarps * kFbChunk) * sizeof(float2);   // 112 KB: 2 CTAs per SM

__device__ __forceinline__ float2 fb_cmul(float2 a, float2 u) {         // a u: one FMUL2 and one FFMA2
  const float2 w = __fmul2_rn(u, make_float2(a.x, a.x));
  return __ffma2_rn(make_float2(-u.y, u.x), make_float2(a.y, a.y), w);
}

struct FbLane {
  const char *sA, *sU;       // shared tables (byte addressing)
  uint32_t koff, uoff;       // lane's byte offsets: A copy and sign, U column
  uint32_t inc8;             // phase increment << 8
};

__device__ __forceinline__ void fb_step(float2 &acc, uint32_t &psi, float2 xv, const FbLane &l) {
  const float2 A = *(const float2 *)(l.sA + (((psi >> 9) & 0x3f80u) | l.koff));   // a = bits 16..22 of psi, x 128 bytes
  const float2 U = *(const float2 *)(l.sU + ((psi & 0xff00u) | l.uoff));           // r = bits 8..15 of psi, x 256 bytes
  psi += l.inc8;
  foldk::cfma(acc, fb_cmul(A, U), xv);
}

// samples [s, e) of the warp's staged chunk, psi = the phase of sample s
__device__ __forceinline__ void fb_run(float2 &acc0, float2 &acc1, uint32_t psi, const float2 *xb, int s, const int e,
                                       const FbLane &l) {
  if (s < e && (s & 1)) { fb_step(acc0, psi, xb[s], l); ++s; }
  for (; s + 8 <= e; s += 8) {
    float4 q[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) q[k] = ((const float4 *)(xb + s))[k];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      fb_step(acc0, psi, make_float2(q[k].x, q[k].y), l);
      fb_step(acc1, psi, make_float2(q[k].z, q[k].w), l);
    }
  }
  for (; s + 2 <= e; s += 2) {
    const float4 q = *(const float4 *)(xb + s);
    fb_step(acc0, psi, make_float2(q.x, q.y), l);
    fb_step(acc1, psi, make_float2(q.z, q.w), l);
  }
  if (s < e) fb_step(acc0, psi, xb[s], l);
}

// the part of the window ending at b-1 that belongs to the next window (see above); b >= 1 is call-relative,
// taps = column c of the channel taps, ph = the NCO phase at b (bits 0..14)
__device__ __noinline__ float2 fb_tail(const float2 *__restrict__ x, const float2 *__restrict__ hist, const float2 *__restrict__ taps,
                                       int64_t b, int L1, uint32_t c_pad, uint32_t ph, uint32_t inc, bool nco, uint32_t negx,
                                       const char *sA, uint32_t lk) {
  float2 sent = make_float2(0.f, 0.f);
  for (int j = 0; j < L1; ++j, ph += inc) {
    float2 y = make_float2(0.f, 0.f);                   // output b+j, samples before b only
    const int64_t i0 = b + j - L1;
    for (int t = 0; t + j < L1; ++t) {
      const int64_t i = i0 + t;
      const float2 xv = i >= 0 ? __ldg(x + i) : __ldg(hist + (L1 + i));
      foldk::cfma(y, __ldg(taps + (size_t)t * c_pad), xv);
    }
    float2 cj = make_float2(1.f, 0.f);                  // lut_inc == 0: the mixer is bypassed
    if (nco) cj = *(const float2 *)(sA + (((((ph >> 8) & 127u) ^ negx) << 7) | lk));
    foldk::cfma(sent, cj, y);
  }
  return sent;
}

__device__ __forceinline__ void fb_flush(float *acc, uint32_t slot, float2 v, bool active) {
  if (active && (v.x != 0.f || v.y != 0.f)) { atomicAdd(acc + 2 * (size_t)slot, v.x); atomicAdd(acc + 2 * (size_t)slot + 1, v.y); }
}

__global__ void __launch_bounds__(kT, 2) bank_fold_f32_kernel(const BankAccumArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2 *sU = (float2 *)smem_raw;                  // [r][32]
  float2 *sA = sU + 256 * 32;                       // [sign][a][16]
  float2 *sX = sA + 2 * 128 * 16;                   // [warp][kFbChunk]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t groups = (a.channels + 31) / 32;
  const uint32_t g = blockIdx.x % groups, span = blockIdx.x / groups;   // neighbouring CTAs: the same samples, other channels

  // as in the integer kernels: zero the next call's accumulators, roll the history
  {
    float2 *nxt = (float2 *)a.acc_next;
    const size_t total = (size_t)a.zero_next * a.channels;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + tid; k < total; k += stride)
      nxt[(k / a.zero_next) * a.acc_stride + (k % a.zero_next)] = make_float2(0.f, 0.f);
    if (blockIdx.x == 0) {
      const int64_t n = a.n, H = a.hist_len;
      for (int64_t k = tid; k < H; k += blockDim.x) {
        const int64_t i = n - H + k;
        ((float2 *)a.hist_out)[k] = (i >= 0) ? ((const float2 *)a.x)[i] : ((const float2 *)a.hist_in)[H + i];
      }
    }
  }
  {
    const float4 *gu = (const float4 *)a.tab_u + (size_t)g * (256 * 32 / 2);
    for (int k = tid; k < 256 * 16; k += kT) ((float4 *)sU)[k] = gu[k];
    const float2 *lut = (const float2 *)a.lut;
    for (int k = tid; k < 2 * 128 * 16; k += kT) {
      float2 v = lut[(k >> 4) & 127];
      if (k >> 11) v.y = -v.y;                      // negative shifts: conj
      sA[k] = v;
    }
  }
  __syncthreads();

  const uint32_t c = g * 32 + lane, c_pad = groups * 32;
  const bool active = c < a.channels;
  const uint32_t inc_full = active ? a.inc[c] : 0u, inc = inc_full & 0x7fffu;
  const bool nco = inc_full != 0, neg = active && a.neg[c] != 0;
  const uint32_t lk = (uint32_t)(lane & 15) << 3;
  const FbLane l{(const char *)sA, (const char *)sU, lk | (neg ? 16384u : 0u), (uint32_t)lane << 3, inc << 8};
  float *acc_out = (float *)a.acc_cur + 2 * (size_t)(active ? c : 0) * a.acc_stride;
  float2 *xb = sX + warp * kFbChunk;
  const float2 *__restrict__ x = (const float2 *)a.x;

  const int64_t lo = (int64_t)span * kFbSpan + (int64_t)warp * kFbWarpSpan;
  if (lo >= (int64_t)a.n) return;
  const int64_t hi = min(lo + (int64_t)kFbWarpSpan, (int64_t)a.n);
  uint32_t slot = (uint32_t)(((uint64_t)a.r0 + (uint64_t)lo - ((a.first && lo > 0) ? 1u : 0u)) / a.ss);
  int64_t nb = (int64_t)(slot + 1) * a.ss + (int64_t)a.first - (int64_t)a.r0;   // first sample of the next window

  float2 pre[8];
  auto load_chunk = [&](int64_t base) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int64_t p = base + lane + 32 * u;
      pre[u] = p < hi ? foldk::ld_stream(x + p) : make_float2(0.f, 0.f);
    }
  };
  load_chunk(lo);
  float2 acc0 = make_float2(0.f, 0.f), acc1 = acc0;
  for (int64_t ck = lo; ck < hi; ck += kFbChunk) {
    __syncwarp();
#pragma unroll
    for (int u = 0; u < 8; ++u) xb[lane + 32 * u] = pre[u];
    __syncwarp();
    if (ck + kFbChunk < hi) load_chunk(ck + kFbChunk);          // in flight while this chunk is summed
    const int64_t ce = min(ck + (int64_t)kFbChunk, hi);
    for (int64_t cur = ck; cur < ce;) {
      const int64_t se = min(nb, ce);
      fb_run(acc0, acc1, ((a.consumed15 + (uint32_t)cur) * inc) << 8, xb, (int)(cur - ck), (int)(se - ck), l);
      cur = se;
      if (cur == nb) {                                          // sample nb-1 ends window `slot`
        const float2 sent = fb_tail(x, (const float2 *)a.hist_in, (const float2 *)a.taps + (active ? c : 0), nb, (int)a.taps_len - 1, c_pad,
                                    (a.consumed15 + (uint32_t)nb) * inc, inc, nco, neg ? 127u : 0u, l.sA, lk);
        fb_flush(acc_out, slot, make_float2(acc0.x + acc1.x - sent.x, acc0.y + acc1.y - sent.y), active);
        acc0 = sent; acc1 = make_float2(0.f, 0.f);
        ++slot; nb += a.ss;
      }
    }
  }
  fb_flush(acc_out, slot, make_float2(acc0.x + acc1.x, acc0.y + acc1.y), active);
}

int launch_bank_fold_f32(const BankAccumArgs &a, cudaStream_t st) {
  const uint64_t groups = (a.channels + 31) / 32, spans = ((uint64_t)a.n + kFbSpan - 1) / kFbSpan;
  if (groups * spans > 0x7fffffffull) return set_error(SDRG_ERR_RUNTIME, "bank: too many channels x samples in one call");
  return launch("bank_fold_f32_kernel", bank_fold_f32_kernel, (unsigned)(groups * spans), kT, kFbSmem, st, a);
}

// finalize for every channel: blockIdx.y = channel
template <int SCALAR>
__global__ void __launch_bounds__(256) bank_finalize_kernel(const IqbbFinalizeArgs base, const BankFinalizeStrides s) {
  __shared__ typename Fin<SCALAR>::Last sphi[256];
  __shared__ unsigned char sskip[256];
  IqbbFinalizeArgs a = base;
  const size_t c = blockIdx.y;
  a.acc_cur = (const char *)base.acc_cur + c * s.acc_stride * 8;
  a.acc_next = (char *)base.acc_next + c * s.acc_stride * 8;
  if (base.bb_out) a.bb_out = (char *)base.bb_out + c * s.out_stride * s.bb_bytes;
  if (base.audio_out) a.audio_out = (char *)base.audio_out + c * s.out_stride * s.audio_bytes;
  a.fm_last_in = (const char *)base.fm_last_in + c * 8;
  a.fm_last_out = (char *)base.fm_last_out + c * 8;
  iqbb_finalize_block<SCALAR>(a, blockIdx.x * 256u, (int)threadIdx.x, sphi, sskip);
}

}  // namespace

int launch_bank_accum(int scalar, const BankAccumArgs &a, cudaStream_t st) {
  if (a.n == 0 || a.channels == 0) return SDRG_OK;
  if (scalar == SDRG_T_F32) return launch_bank_fold_f32(a, st);
  if (scalar != SDRG_T_S8 && scalar != SDRG_T_S16) return set_error(SDRG_ERR_RUNTIME, "bank: no accumulate kernel for scalar %d", scalar);
  const size_t n_xs = kTile + a.hist_len + 8;
  const size_t smem = sizeof(int4) * (size_t)a.group * a.taps_len + sizeof(int2) * 128 + sizeof(uint32_t) * (n_xs + (n_xs >> 5) + 1);
  if (smem > 200 * 1024) return set_error(SDRG_ERR_RUNTIME, "bank: filter order too large for the bank kernel");
  dim3 grid((unsigned)((a.n + kTile - 1) / kTile), (unsigned)((a.channels + a.group - 1) / a.group));
  if (a.taps_len <= 32) {
    const int lp = (int)((a.taps_len + 1) & ~1u);
    return scalar == SDRG_T_S8 ? dispatch_bank_fixed<true>(lp, a, grid, st) : dispatch_bank_fixed<false>(lp, a, grid, st);
  }
  return launch("bank_accum_kernel", scalar == SDRG_T_S8 ? bank_accum_kernel<true> : bank_accum_kernel<false>, grid, kT, smem, st, a);
}

int launch_bank_finalize(int scalar, const IqbbFinalizeArgs &a, const BankFinalizeStrides &s, uint32_t channels, cudaStream_t st) {
  if (channels == 0) return SDRG_OK;
  const unsigned gx = (a.n_out + 255) / 256;
  dim3 grid(gx ? gx : 1, channels);
  return dispatch(scalar, std::integer_sequence<int, SDRG_T_S8, SDRG_T_S16, SDRG_T_F32>{},
                  [&](auto S) { return launch("bank_finalize_kernel", bank_finalize_kernel<S>, grid, 256, 0, st, a, s); },
                  [&] { return set_error(SDRG_ERR_RUNTIME, "bank: no finalize kernel for scalar %d", scalar); });
}

}  // namespace sdrg

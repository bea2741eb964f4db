// iqbb_kernels.cu -- IQBaseBand<Scalar> on the device: the direct (unfolded) kernels.
//
// Reference semantics: src/baseband.hh:198-236 (FIR -> NCO mix -> boxcar decimation, in this
// order, with a truncating shift after the FIR and after the mix) and src/freqshift.hh:58-74.
// Closed-form restatement used here (SURVEY.md appendix A): with n the sample index since
// config(), y[n] = (sum_t k[t] x[n-(L-1)+t]) >> 14, z[n] = (lut[idx(n)] y[n]) >> shift with
// idx(n) = ((n*inc) mod 32768) >> 8, and output m = trunc_div(wrap32(S_m*ss), wrap32(ss*ss)),
// S_m = sum of z over window W_0=[0..ss], W_m=[m*ss+1..(m+1)*ss].  All integer sums are taken in
// Z/2^32, which is associative, so the parallel evaluation order below is bit-exact.
//
// Kernel 1 (iqbb_accum_*): one CTA per tile of 2048 input samples.
//   stage tile + (L-1) halo in shared memory -> register-blocked FIR (8 outputs per thread, a
//   rotating 8-sample register window, taps broadcast from shared memory; the integer complex
//   multiply uses the 3-multiplication Gauss form, exact in Z/2^32) -> NCO -> z to shared memory
//   -> per-window partial sums (one warp or one thread per window) -> RED.ADD into the per-call
//   window accumulators in global memory (L2-resident, 8 B per OUTPUT sample).
// Kernel 2 (iqbb_finalize_*): one thread per completed window: division / narrowing, optional
//   fused FM/AM/USB demodulation, carries the open window into the next call.
#include "iqbb_int_common.cuh"
#include "launch.cuh"
#include "demod_math.cuh"

namespace sdrg {

namespace {

constexpr int kT = kIqbbThreads;
constexpr int kTile = kIqbbTile;
constexpr int kZRow = kT + 2;              // row pitch of the transposed z staging (bank spread)
constexpr unsigned kFull = 0xffffffffu;

__device__ __forceinline__ int pad64(int i) { return i + (i >> 3); }   // 8-byte elements, 8 per thread

// Per-window partial sums of one tile from the transposed z staging, added into the call's
// accumulators.  Short windows (ss <= 64: >= 32 windows per tile) take one THREAD per window --
// the issue cost is ~3 instructions per sample of ONE warp-lane instead of a warp-wide loop per
// window; long windows take one warp per window with a REDUX.SUM at the end.
__device__ __forceinline__ void window_sums_int(const IqbbAccumArgs &a, const int2 *zs, const int64_t tile_base, const int tid) {
  const int lane = tid & 31, warp = tid >> 5;
  const uint32_t tile_lo = (uint32_t)tile_base;
  const uint32_t tile_hi = (uint32_t)min((int64_t)a.n, tile_base + kTile);
  if (tile_hi <= tile_lo) return;
  WindowGrid g{a.ss, a.r0, a.first};
  const uint32_t slot_lo = g.slot(tile_lo), slot_hi = g.slot(tile_hi - 1);
  int *acc = (int *)a.acc_cur;
  const int t_hi = (int)(tile_hi - tile_lo);
  if (a.ss > 64) {
    for (uint32_t s = slot_lo + warp; s <= slot_hi; s += kT / 32) {
      const int lo = max((int)(g.begin(s) - tile_base), 0), hi = min((int)(g.end(s) - tile_base), t_hi);
      uint32_t sr = 0, si = 0;
      for (int o = lo + lane; o < hi; o += 32) {
        const int2 z = zs[(o & (kR - 1)) * kZRow + (o >> 3)];
        sr += (uint32_t)z.x; si += (uint32_t)z.y;
      }
      sr = __reduce_add_sync(kFull, sr);
      si = __reduce_add_sync(kFull, si);
      if (lane == 0) { atomicAdd(acc + 2 * (size_t)s, (int)sr); atomicAdd(acc + 2 * (size_t)s + 1, (int)si); }
    }
  } else {
    for (uint32_t s = slot_lo + tid; s <= slot_hi; s += kT) {
      const int lo = max((int)(g.begin(s) - tile_base), 0), hi = min((int)(g.end(s) - tile_base), t_hi);
      uint32_t sr = 0, si = 0;
#pragma unroll 4
      for (int o = lo; o < hi; ++o) {
        const int2 z = zs[(o & (kR - 1)) * kZRow + (o >> 3)];
        sr += (uint32_t)z.x; si += (uint32_t)z.y;
      }
      atomicAdd(acc + 2 * (size_t)s, (int)sr); atomicAdd(acc + 2 * (size_t)s + 1, (int)si);
    }
  }
}

// ---- integer kernel (arithmetic: iqbb_int_common.cuh) ---------------------------------------------
template <bool IS_S8>
__global__ void __launch_bounds__(kT) iqbb_accum_int_kernel(const IqbbAccumArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int H = (int)a.hist_len, Lp = (int)a.taps_len;
  const int n_xs = kTile + H + 8;
  int4 *tp = (int4 *)smem_raw;                                   // Lp
  int2 *lut = (int2 *)(tp + Lp);                                 // 128
  int2 *zs = lut + 128;                                          // kR * kZRow
  uint32_t *xs = (uint32_t *)(zs + kR * kZRow);                  // pad32(n_xs)+1

  if (IS_S8) prologue<char2, int2>(a); else prologue<short2, int2>(a);

  const int64_t tile_base = (int64_t)blockIdx.x * kTile;
  // stage taps / LUT / samples
  for (int k = tid; k < Lp; k += kT) tp[k] = ((const int4 *)a.taps)[k];
  if (tid < 128) lut[tid] = ((const int2 *)a.lut)[tid];
  for (int k = tid; k < n_xs; k += kT) xs[pad32(k)] = load_sample<IS_S8>(a.x, a.hist_in, tile_base - H + k, H, a.n, a.in_fmt);
  __syncthreads();

  // FIR: outputs ob..ob+7 of the tile; window sample c lives at xs[ob + c]
  const int ob = tid * kR;
  uint32_t A1[kR], A2[kR], A3[kR];
  fir_smem(xs, ob, tp, Lp, A1, A2, A3);

  // >> fir_shift, NCO, stage z (transposed: row r, column tid)
  const uint32_t i0 = (uint32_t)tile_base + (uint32_t)ob;
#pragma unroll
  for (int r = 0; r < kR; ++r) {
    int yr, yi;
    fir_result<IS_S8, kFirComplex>(A1[r], A2[r], A3[r], 0u, a.fir_shift, IS_S8 && a.in_fmt == 5, yr, yi);
    if (a.nco) {
      const uint32_t ph = (a.phase0 + (i0 + r) * a.inc) & 0x7fffu;
      uint32_t idx = ph >> 8;
      if (a.neg) idx = 127u - idx;
      nco_mix<IS_S8>(lut[idx], yr, yi);
    }
    zs[r * kZRow + tid] = make_int2(yr, yi);
  }
  __syncthreads();

  window_sums_int(a, zs, tile_base, tid);
}

// ---- integer kernel, compile-time tap count -------------------------------------------------------
// The tap count LP is fixed at compile time (taps zero-padded at the FRONT to the next even count,
// which is exact): the tile is staged unpadded, every thread pulls its LP+7 packed samples
// with 128-bit shared loads into registers ONCE, the taps sit in the
// kernel's parameter (constant) bank so the FIR inner loop is nothing but IMADs with a constant
// operand plus one unpack per sample -- no loads, no guards, no address arithmetic.
// Persistent CTAs (one per resident slot) walk the tiles grid-stride; the next tile is fetched into
// the other shared buffer with cp.async (LDGSTS: no registers, no scoreboard stall) while the current
// one is being filtered, so the global-load latency that used to head every tile is hidden.
// VAR: 0 complex int16 (also the fused 8-bit AutoCast formats), 1 complex int8, 2 REAL int16 (BaseBand<int16_t>:
// the imaginary input is 0, so the Gauss form collapses to two multiplies per tap: re = sum kr x, im = re + sum (ki-kr) x).
template <int LP, int VAR>
__global__ void __launch_bounds__(kT) iqbb_accum_int_fixed_kernel(const IqbbAccumArgs a, const __grid_constant__ IqbbTaps taps) {
  constexpr bool IS_S8 = VAR == 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int H = LP - 1;
  constexpr int NV = (LP + 7 + 3) / 4;                 // 128-bit loads per thread
  constexpr int n_xs = kTile + 4 * NV + 8;
  constexpr int xs_pitch = (n_xs + 3) & ~3;
  const int tid = threadIdx.x;
  int2 *lut = (int2 *)smem_raw;                                   // 128
  int2 *zs = lut + 128;                                          // kR * kZRow
  uint32_t *xs_all = (uint32_t *)(zs + kR * kZRow);              // 2 x xs_pitch, 16-byte aligned

  if (IS_S8) prologue<char2, int2>(a); else prologue<short2, int2>(a);
  if (tid < 128) lut[tid] = ((const int2 *)a.lut)[tid];
  const int Hh = (int)a.hist_len;                                // history kept by the handle (= stripped taps - 1 <= H)
  const uint32_t fmt = IS_S8 ? 0u : a.in_fmt;                    // int8 here is complex (BaseBand<int8_t> takes the generic kernel)
  const uint32_t n_tiles = (a.n + kTile - 1) / kTile;

  // stage tile t into xs: asynchronously when it is an interior int16 tile, synchronously otherwise
  auto stage = [&](uint32_t t, uint32_t *xs) {
    const int64_t tile_base = (int64_t)t * kTile;
    const bool interior = tile_base >= H && tile_base - H + n_xs <= (int64_t)a.n;
    if (interior && !IS_S8 && a.in_fmt == 0) {
      const uint32_t *xg = (const uint32_t *)a.x + (tile_base - H);
      for (int k = tid; k < n_xs; k += kT) cp_async4(xs + k, xg + k);
    } else if (interior && !IS_S8) {                               // 8-bit / real input formats: convert while staging, no bounds
      const int64_t i0 = tile_base - H;
      for (int k = tid; k < n_xs; k += kT) xs[k] = load_cs16(a.x, i0 + k, a.in_fmt);
    } else {
      for (int k = tid; k < n_xs; k += kT) xs[k] = load_sample<IS_S8>(a.x, a.hist_in, tile_base - H + k, Hh, a.n, fmt);
    }
    cp_async_commit();
  };

  uint32_t t = blockIdx.x;
  if (t < n_tiles) stage(t, xs_all);
  for (int buf = 0; t < n_tiles; t += gridDim.x, buf ^= 1) {
    uint32_t *xs = xs_all + buf * xs_pitch;
    if (t + gridDim.x < n_tiles) { stage(t + gridDim.x, xs_all + (buf ^ 1) * xs_pitch); cp_async_wait<1>(); }
    else cp_async_wait<0>();
    __syncthreads();
    const int64_t tile_base = (int64_t)t * kTile;

    uint32_t w[4 * NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const uint4 q = ((const uint4 *)xs)[tid * 2 + v];
      w[4 * v] = q.x; w[4 * v + 1] = q.y; w[4 * v + 2] = q.z; w[4 * v + 3] = q.w;
    }
    constexpr int FORM = VAR == 2 ? kFirRealIn : kFirComplex;
    uint32_t A1[kR], A2[kR], A3[kR];
    fir_fixed<LP, FORM>(w, taps.t, 0u, A1, A2, A3);

    const int ob = tid * kR;
    const uint32_t i0 = (uint32_t)tile_base + (uint32_t)ob;
    const uint32_t negx = a.neg ? 127u : 0u;                     // 127 - idx == idx ^ 127 on 0..127
    uint32_t ph = (a.phase0 + i0 * a.inc) & 0x7fffu;
#pragma unroll
    for (int r = 0; r < kR; ++r) {
      int yr, yi;
      fir_result<IS_S8, FORM>(A1[r], A2[r], A3[r], 0u, a.fir_shift, false, yr, yi);
      if (a.nco) {
        const int2 l = lut[(ph >> 8) ^ negx];
        ph = (ph + a.inc) & 0x7fffu;
        nco_mix<IS_S8>(l, yr, yi);
      }
      zs[r * kZRow + tid] = make_int2(yr, yi);
    }
    __syncthreads();
    window_sums_int(a, zs, tile_base, tid);
  }
}

template <int LP, int VAR>
int launch_fixed(const IqbbAccumArgs &a, const IqbbTaps &taps, unsigned n_tiles, cudaStream_t st) {
  constexpr int NV = (LP + 7 + 3) / 4;
  constexpr int xs_pitch = (kTile + 4 * NV + 8 + 3) & ~3;
  const size_t smem = sizeof(int2) * 128 + sizeof(int2) * kR * kZRow + sizeof(uint32_t) * 2 * xs_pitch;
  return launch_persistent("iqbb_accum_int_fixed_kernel", iqbb_accum_int_fixed_kernel<LP, VAR>, n_tiles, kT, smem, st, a, taps);
}

template <int VAR>
int dispatch_fixed(int lp, const IqbbAccumArgs &a, const IqbbTaps &taps, unsigned grid, cudaStream_t st) {
  return dispatch(lp, int_range<2, 32, 2>{}, [&](auto LP) { return launch_fixed<LP, VAR>(a, taps, grid, st); },
                  [&] { return set_error(SDRG_ERR_RUNTIME, "no fixed-tap kernel for %d taps", lp); });
}

// ---- float kernel (direct form; the folded fast path lives in iqbb_fold_kernels.cu) ---------------
__global__ void __launch_bounds__(kT) iqbb_accum_f32_kernel(const IqbbAccumArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int H = (int)a.hist_len, Lp = (int)a.taps_len;
  const int n_xs = kTile + H + 8;
  float2 *tp = (float2 *)smem_raw;                               // Lp (rounded up to even count)
  float2 *lut = tp + ((Lp + 1) & ~1);                            // 128
  float2 *zs = lut + 128;                                        // kR * kZRow
  float2 *xs = zs + kR * kZRow;                                  // pad64(n_xs)+1

  prologue<float2, float2>(a);

  const int64_t tile_base = (int64_t)blockIdx.x * kTile;
  for (int k = tid; k < Lp; k += kT) tp[k] = ((const float2 *)a.taps)[k];
  if (tid < 128) lut[tid] = ((const float2 *)a.lut)[tid];
  for (int k = tid; k < n_xs; k += kT) {
    const int64_t i = tile_base - H + k;
    float2 v = make_float2(0.f, 0.f);
    if (i < 0) v = ((const float2 *)a.hist_in)[H + i];
    else if (i < (int64_t)a.n) v = ((const float2 *)a.x)[i];
    xs[pad64(k)] = v;
  }
  __syncthreads();

  const int ob = tid * kR;
  float yr[kR], yi[kR];
  float2 w[kR];
#pragma unroll
  for (int c = 0; c < kR; ++c) { yr[c] = 0.f; yi[c] = 0.f; w[c] = xs[pad64(ob + c)]; }
  for (int t0 = 0; t0 < Lp; t0 += kR) {
#pragma unroll
    for (int u = 0; u < kR; ++u) {
      const int t = t0 + u;
      if (t < Lp) {
        const float2 c = tp[t];
#pragma unroll
        for (int r = 0; r < kR; ++r) {
          const int s = (r + u) & (kR - 1);
          yr[r] = fmaf(c.x, w[s].x, yr[r]); yr[r] = fmaf(-c.y, w[s].y, yr[r]);
          yi[r] = fmaf(c.x, w[s].y, yi[r]); yi[r] = fmaf(c.y, w[s].x, yi[r]);
        }
        w[u] = xs[pad64(ob + t + kR)];
      }
    }
  }
  const uint32_t i0 = (uint32_t)tile_base + (uint32_t)ob;
#pragma unroll
  for (int r = 0; r < kR; ++r) {
    float zr = yr[r], zi = yi[r];
    if (a.nco) {
      const uint32_t ph = (a.phase0 + (i0 + r) * a.inc) & 0x7fffu;
      uint32_t idx = ph >> 8;
      if (a.neg) idx = 127u - idx;
      const float2 l = lut[idx];
      zr = l.x * yr[r] - l.y * yi[r];
      zi = l.x * yi[r] + l.y * yr[r];
    }
    zs[r * kZRow + tid] = make_float2(zr, zi);
  }
  __syncthreads();

  const uint32_t tile_lo = (uint32_t)tile_base;
  const uint32_t tile_hi = (uint32_t)min((int64_t)a.n, tile_base + kTile);
  if (tile_hi <= tile_lo) return;
  WindowGrid g{a.ss, a.r0, a.first};
  const uint32_t slot_lo = g.slot(tile_lo), slot_hi = g.slot(tile_hi - 1);
  float *acc = (float *)a.acc_cur;
  if (a.ss >= 16) {
    for (uint32_t s = slot_lo + warp; s <= slot_hi; s += kT / 32) {
      const int lo = (int)(max(g.begin(s), (int64_t)tile_lo) - tile_base);
      const int hi = (int)(min(g.end(s), (int64_t)tile_hi) - tile_base);
      float sr = 0.f, si = 0.f;
      for (int o = lo + lane; o < hi; o += 32) {
        const float2 z = zs[(o & (kR - 1)) * kZRow + (o >> 3)];
        sr += z.x; si += z.y;
      }
      sr = warp_sum(sr); si = warp_sum(si);
      if (lane == 0) { atomicAdd(acc + 2 * (size_t)s, sr); atomicAdd(acc + 2 * (size_t)s + 1, si); }
    }
  } else {
    for (uint32_t s = slot_lo + tid; s <= slot_hi; s += kT) {
      const int lo = (int)(max(g.begin(s), (int64_t)tile_lo) - tile_base);
      const int hi = (int)(min(g.end(s), (int64_t)tile_hi) - tile_base);
      float sr = 0.f, si = 0.f;
      for (int o = lo; o < hi; ++o) {
        const float2 z = zs[(o & (kR - 1)) * kZRow + (o >> 3)];
        sr += z.x; si += z.y;
      }
      atomicAdd(acc + 2 * (size_t)s, sr); atomicAdd(acc + 2 * (size_t)s + 1, si);
    }
  }
}

}  // namespace
}  // namespace sdrg
#include "iqbb_finalize.cuh"
namespace sdrg {
namespace {

template <int SCALAR>
__global__ void __launch_bounds__(256) iqbb_finalize_kernel(const IqbbFinalizeArgs a) {
  __shared__ typename Fin<SCALAR>::Last sphi[256];
  __shared__ unsigned char sskip[256];
  iqbb_finalize_block<SCALAR>(a, blockIdx.x * 256u, (int)threadIdx.x, sphi, sskip);
}

size_t accum_smem_int(uint32_t Lp, uint32_t H) {
  return sizeof(int4) * Lp + sizeof(int2) * 128 + sizeof(int2) * kR * kZRow +
         sizeof(uint32_t) * ((kTile + H + 8) + ((kTile + H + 8) >> 5) + 1);
}
size_t accum_smem_f32(uint32_t Lp, uint32_t H) {
  return sizeof(float2) * ((Lp + 1) & ~1u) + sizeof(float2) * 128 + sizeof(float2) * kR * kZRow +
         sizeof(float2) * ((kTile + H + 8) + ((kTile + H + 8) >> 3) + 1);
}

}  // namespace

int launch_iqbb_accum(int scalar, const IqbbAccumArgs &a, cudaStream_t st) {
  if (a.n == 0) return SDRG_OK;
  const unsigned grid = (unsigned)((a.n + kTile - 1) / kTile);
  if (scalar != SDRG_T_F32 && a.host_taps && a.taps_len <= 32 && a.in_fmt != 5) {     // (BaseBand<int8_t> stays on the generic kernel)
    // zero taps in FRONT up to the next even count: x[n-(LP-1)+t] k'[t] with k'[t] = 0 for t < pad
    const int lp = (int)((a.taps_len + 1) & ~1u), pad = lp - (int)a.taps_len;
    IqbbTaps taps;
    for (int t = 0; t < 32; ++t) taps.t[t] = make_int4(0, 0, 0, 0);
    for (int t = 0; t < (int)a.taps_len; ++t) taps.t[pad + t] = ((const int4 *)a.host_taps)[t];
    const int rc = launch_iqbb_accum_warp(scalar, a, taps, lp, st);      // sub_sample >= 16: the barrier-free per-warp kernel
    if (rc >= 0) return rc;
    if (scalar == SDRG_T_S8) return dispatch_fixed<1>(lp, a, taps, grid, st);
    return a.in_fmt == 4 ? dispatch_fixed<2>(lp, a, taps, grid, st) : dispatch_fixed<0>(lp, a, taps, grid, st);
  }
  if (scalar == SDRG_T_F32) return launch("iqbb_accum_f32_kernel", iqbb_accum_f32_kernel, grid, kT, accum_smem_f32(a.taps_len, a.hist_len), st, a);
  return launch("iqbb_accum_int_kernel", scalar == SDRG_T_S8 ? iqbb_accum_int_kernel<true> : iqbb_accum_int_kernel<false>, grid, kT,
                accum_smem_int(a.taps_len, a.hist_len), st, a);
}

int launch_iqbb_finalize(int scalar, const IqbbFinalizeArgs &a, cudaStream_t st) {
  const unsigned grid = (unsigned)((a.n_out + 255) / 256);
  const unsigned g = grid ? grid : 1;     // the carry must be moved even when nothing completed
  return dispatch(scalar, std::integer_sequence<int, SDRG_T_S16, SDRG_T_S8, SDRG_T_F32>{},
                  [&](auto S) { return launch("iqbb_finalize_kernel", iqbb_finalize_kernel<S>, g, 256, 0, st, a); },
                  [&] { return set_error(SDRG_ERR_ARG, "finalize: unsupported scalar %d", scalar); });
}

}  // namespace sdrg

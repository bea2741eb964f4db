// iqbb_warp_kernels.cu -- IQBaseBand<int16_t>/<int8_t>, fixed tap count, one WARP per 256-sample tile and no CTA
// barrier anywhere in the loop.
//
// The arithmetic is iqbb_int_common.cuh's (load_sample, fir_fixed, fir_result, nco_mix, narrow16), as in
// iqbb_accum_int_fixed_kernel; only the symmetric-tap FIR (VAR 4) is this kernel's own, and int8's narrowing to int16
// is applied just before the NCO mix rather than inside fir_result.  What changed is the choreography.  The CTA-wide
// kernel staged 2048 samples for 256 threads, exchanged the mixed samples through a transposed shared array and summed
// each window with one thread or one warp -- two __syncthreads per tile, 41 of 256 threads busy in the window phase at
// sub_sample 50, and the barrier was the top stall (profiles/r01_final_int16_kernel_summary.md: 59 % of the IMAD pipe against the bank kernel's 86 %).
// Here a warp owns its tile end to end:
//   * it stages its own 256 + LP + 7 samples with cp.async into a private, double-buffered shared region (the next
//     tile is in flight while the current one is filtered), 16-byte chunks XOR-swizzled so that the 128-bit reads
//     of lanes j and j + 4 no longer collide;
//   * FIR (taps in the constant bank) and NCO run out of registers as in the CTA-wide kernel;
//   * the window sums never leave the warp: a lane's 8 consecutive outputs touch at most two windows
//     (sub_sample >= 16), so it forms two partial sums and adds them to a per-warp shared accumulator line
//     (native shared-memory integer atomics; their serialisation costs LSU cycles, not IMAD-pipe slots), or, when
//     the warp touches at most four windows, reduces with REDUX; one global RED per window and warp follows.
//   * window indices come from a multiply-shift by a host-computed reciprocal instead of integer divisions.
// Tap kinds (template VAR): 0 complex taps on complex int16 (Gauss 3-multiply form), 1 the same on int8 samples,
// 2 real int16 input (BaseBand<int16_t>, src/baseband.hh:304-529), 3 REAL taps (k_im == 0: a filter centred on
// 0 Hz, the sdr_rec configuration -- two multiplies per tap), 4 real taps SYMMETRIC about the middle of an even count
// (pairs of samples are added first: one multiply per component and tap pair; (x_a + x_b) k = x_a k + x_b k in Z/2^32).
#include "iqbb_int_common.cuh"
#include "launch.cuh"

namespace sdrg {
namespace {

constexpr int kT = kIqbbThreads;           // 8 warps per CTA
constexpr int kWT = 32 * kR;               // outputs per warp tile
constexpr unsigned kFull = 0xffffffffu;

// 16-byte chunk c of a warp's staging buffer lives at chunk swz(c): lanes j and j + 4 of a quarter-warp read chunks
// 2j + v and 2j + 8 + v, which would share banks; flipping bit 0 of every chunk with bit 3 set separates them.
__device__ __forceinline__ int swz(int c) { return c ^ ((c >> 3) & 1); }

__device__ __forceinline__ uint32_t div_ss(uint32_t q, uint32_t m, uint32_t s) { return (uint32_t)(((uint64_t)q * m) >> s); }

// CONV: the input needs converting while it is staged (fused AutoCast formats, real int16) -- a separate instantiation
// so that the plain complex int16 path does not carry the staging registers.
template <int LP, int VAR, bool CONV>
__global__ void __launch_bounds__(kT) iqbb_accum_int_warp_kernel(const IqbbAccumArgs a, const __grid_constant__ IqbbTaps taps) {
  constexpr bool IS_S8 = VAR == 1, SYM = VAR == 4;
  constexpr int FORM = VAR == 2 ? kFirRealIn : VAR == 3 ? kFirRealTaps : kFirComplex;
  constexpr int H = LP - 1;
  constexpr int NV = (LP + 7 + 3) / 4;                 // 128-bit loads per lane
  constexpr int n_xs = kWT - kR + 4 * NV;              // words a warp tile needs: lane 31 reads [248, 248 + 4 NV)
  constexpr int pitch = (n_xs + 7) & ~7;               // whole chunk pairs (the swizzle stays inside a pair)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int2 *lut = (int2 *)smem_raw;                                        // 128
  int2 *sacc_all = lut + 128;                                          // 8 warps x 32 window accumulators
  uint32_t *xs_all = (uint32_t *)(sacc_all + (kT / 32) * 32);          // 8 warps x 2 x pitch, 16-byte aligned
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int2 *sacc = sacc_all + warp * 32;
  uint32_t *xs_w = xs_all + warp * 2 * pitch;

  if (IS_S8) prologue<char2, int2>(a); else prologue<short2, int2>(a);
  if (tid < 128) lut[tid] = ((const int2 *)a.lut)[a.neg ? 127 - tid : tid];     // idx = 127 - idx for negative shifts (freqshift.hh:65)
  sacc[lane] = make_int2(0, 0);
  __syncthreads();                                                     // the only CTA barrier: LUT and accumulators are in place

  const int Hh = (int)a.hist_len;                                      // history the handle keeps (stripped taps - 1 <= H)
  const uint32_t fmt = IS_S8 ? 0u : a.in_fmt;                          // int8 here is complex
  const uint32_t Z = a.zero;                                           // == 0; see IqbbAccumArgs::zero
  const uint32_t n_tiles = (a.n + kWT - 1) / kWT;
  const uint32_t n_warps = gridDim.x * (kT / 32);

  // Stage tile `wt` into `xs`.  Plain complex int16 interior tiles go through cp.async (no registers, no stall).
  // The converting formats (fused AutoCast from 8-bit pairs, real int16) cannot: their loads are issued here into
  // `raw` and converted / stored only after the current tile has been filtered (finish_stage), so the load latency
  // hides behind the FIR exactly like the asynchronous copies do.  Edge tiles (history, stream end) are staged at once.
  constexpr int NL = CONV ? (n_xs + 31) / 32 : 1;
  uint32_t raw[NL];
  bool raw_pending = false;
  auto stage = [&](uint32_t wt, uint32_t *xs) {
    const int64_t base = (int64_t)wt * kWT - H;                        // call-relative index of buffer word 0
    const bool interior = base >= 0 && base + n_xs <= (int64_t)a.n;
    if (interior && !IS_S8 && !CONV) {
      const uint32_t *xg = (const uint32_t *)a.x + base;
      for (int k = lane; k < n_xs; k += 32) cp_async4(xs + ((swz(k >> 2) << 2) | (k & 3)), xg + k);
    } else if (interior && CONV) {
#pragma unroll
      for (int j = 0; j < NL; ++j) { const int k = lane + 32 * j; raw[j] = k < n_xs ? load_cs16(a.x, base + k, a.in_fmt) : 0u; }
      raw_pending = true;
    } else {
      for (int k = lane; k < n_xs; k += 32) xs[(swz(k >> 2) << 2) | (k & 3)] = load_sample<IS_S8>(a.x, a.hist_in, base + k, Hh, a.n, fmt);
    }
    cp_async_commit();
  };
  auto finish_stage = [&](uint32_t *xs) {
    if (!CONV || !raw_pending) return;
#pragma unroll
    for (int j = 0; j < NL; ++j) { const int k = lane + 32 * j; if (k < n_xs) xs[(swz(k >> 2) << 2) | (k & 3)] = raw[j]; }
    raw_pending = false;
  };

  uint32_t wt = blockIdx.x * (kT / 32) + warp;
  if (wt < n_tiles) { stage(wt, xs_w); finish_stage(xs_w); }
  for (int buf = 0; wt < n_tiles; wt += n_warps, buf ^= 1) {
    uint32_t *xs = xs_w + buf * pitch;
    if (wt + n_warps < n_tiles) { stage(wt + n_warps, xs_w + (buf ^ 1) * pitch); cp_async_wait<1>(); }
    else cp_async_wait<0>();
    __syncwarp();                                                      // every lane's copies of this tile have landed

    uint32_t w[4 * NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const uint4 q = ((const uint4 *)xs)[swz(lane * 2 + v)];
      w[4 * v] = q.x; w[4 * v + 1] = q.y; w[4 * v + 2] = q.z; w[4 * v + 3] = q.w;
    }
    __syncwarp();                                                      // all reads done before the tile after next overwrites this buffer

    int yr[kR], yi[kR];
    if (SYM) {
      // y[r] = sum_{t < LP/2} k[t] (x[r + t] + x[r + LP-1 - t]),  real k
      int xr[LP + kR - 1], xi[LP + kR - 1];
#pragma unroll
      for (int c = 0; c < LP + kR - 1; ++c) unpack16(w[c], xr[c], xi[c]);
      uint32_t Ar[kR], Ai[kR];
#pragma unroll
      for (int r = 0; r < kR; ++r) Ar[r] = Ai[r] = 0u;
#pragma unroll
      for (int tt = 0; tt < LP / 2; ++tt) {
        const uint32_t k = (uint32_t)taps.t[tt].x;
#pragma unroll
        for (int r = 0; r < kR; ++r) {
          Ar[r] += k * ((uint32_t)xr[r + tt] + (uint32_t)xr[r + LP - 1 - tt] + Z);
          Ai[r] += k * ((uint32_t)xi[r + tt] + (uint32_t)xi[r + LP - 1 - tt] + Z);
        }
      }
#pragma unroll
      for (int r = 0; r < kR; ++r) fir_result<false, kFirRealTaps>(Ar[r], Ai[r], 0u, 0u, a.fir_shift, false, yr[r], yi[r]);
    } else {
      uint32_t A1[kR], A2[kR], A3[kR];
      fir_fixed<LP, FORM>(w, taps.t, Z, A1, A2, A3);
#pragma unroll
      for (int r = 0; r < kR; ++r) fir_result<false, FORM>(A1[r], A2[r], A3[r], Z, a.fir_shift, false, yr[r], yi[r]);
    }

    // ---- NCO (in place on yr/yi).  The running phase is not masked: only bits 8..14 select the LUT entry.
    // int8: fir_result's narrowing to int16 is applied here, just before the mix, which keeps this kernel's register
    // allocation (the result is the same).
    const uint32_t i_w = wt * kWT, i0 = i_w + (uint32_t)lane * kR;
    if (a.nco) {
      uint32_t ph = a.phase0 + i0 * a.inc;
#pragma unroll
      for (int r = 0; r < kR; ++r) {
        int zr = yr[r], zi = yi[r];
        if (IS_S8) narrow16(zr, zi);
        const int2 l = lut[(ph >> 8) & 127u];                          // (the table is staged reversed for negative shifts)
        ph += a.inc + Z;
        nco_mix<IS_S8>(l, zr, zi);
        yr[r] = zr; yi[r] = zi;
      }
    } else if (IS_S8) {
#pragma unroll
      for (int r = 0; r < kR; ++r) narrow16(yr[r], yi[r]);
    }

    // ---- the lane's two partial window sums: `tot` over its valid outputs, `hi` over those past the window boundary
    const uint32_t i_end = min(a.n, i_w + kWT);                        // first index past this tile's valid outputs
    const uint32_t adj0 = (a.first && i0 > 0) ? 1u : 0u;
    const uint32_t slot_a = div_ss(a.r0 + i0 - adj0, a.div_m, a.div_s);
    const uint32_t bnd = (slot_a + 1) * a.ss - a.r0 + a.first;        // first index of window slot_a + 1 (> i0)
    const uint32_t slot_w = div_ss(a.r0 + i_w - ((a.first && i_w > 0) ? 1u : 0u), a.div_m, a.div_s);
    const uint32_t i_last = i_end - 1;
    const uint32_t n_win = div_ss(a.r0 + i_last - ((a.first && i_last > 0) ? 1u : 0u), a.div_m, a.div_s) - slot_w + 1;
    const int rb = (int)min(bnd - i0, (uint32_t)kR);                   // outputs rb.. belong to the next window
    if (i_end - i_w < (uint32_t)kWT) {                                 // the stream's last, partial tile (warp-uniform)
      const int re = max(min((int)(i_end - i0), kR), 0);
#pragma unroll
      for (int r = 0; r < kR; ++r) if (r >= re) { yr[r] = 0; yi[r] = 0; }
    }
    const uint32_t mhi = 0xffu & ~((1u << rb) - 1u);                   // bit r set: output r goes to `hi`
    uint32_t tot_r = 0, tot_i = 0, hi_r = 0, hi_i = 0;
#pragma unroll
    for (int r = 0; r < kR; r += 2) {                                  // three-input adds
      tot_r += (uint32_t)yr[r] + (uint32_t)yr[r + 1];
      tot_i += (uint32_t)yi[r] + (uint32_t)yi[r + 1];
    }
#pragma unroll
    for (int r = 1; r < kR; ++r) {                                     // (output 0 always belongs to the lane's first window)
      asm("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\tand.b32 t, %4, %5;\n\tsetp.ne.b32 p, t, 0;\n\t@p add.u32 %0, %0, %2;\n\t@p add.u32 %1, %1, %3;\n\t}"
          : "+r"(hi_r), "+r"(hi_i) : "r"(yr[r]), "r"(yi[r]), "r"(mhi), "r"(1u << r));
    }
    const uint32_t lo_r = tot_r - hi_r, lo_i = tot_i - hi_i;
    const uint32_t ka = slot_a - slot_w;                               // this lane's windows: ka and ka + 1 (relative to the warp's first)
    int *acc = (int *)a.acc_cur + 2 * (size_t)slot_w;
    if (n_win <= 4) {                                                  // long windows: REDUX per window
#pragma unroll 1
      for (uint32_t k = 0; k < n_win; ++k) {
        const uint32_t vr = (ka == k ? lo_r : 0u) + (ka + 1 == k ? hi_r : 0u);
        const uint32_t vi = (ka == k ? lo_i : 0u) + (ka + 1 == k ? hi_i : 0u);
        const uint32_t sr = __reduce_add_sync(kFull, vr), si = __reduce_add_sync(kFull, vi);
        if (lane == 0 && (sr | si)) { atomicAdd(acc + 2 * k, (int)sr); atomicAdd(acc + 2 * k + 1, (int)si); }
      }
    } else {                                                           // short windows: the warp's shared accumulator line
      if (lo_r | lo_i) { atomicAdd(&sacc[ka].x, (int)lo_r); atomicAdd(&sacc[ka].y, (int)lo_i); }
      if (hi_r | hi_i) { atomicAdd(&sacc[ka + 1].x, (int)hi_r); atomicAdd(&sacc[ka + 1].y, (int)hi_i); }
      __syncwarp();
      if ((uint32_t)lane < n_win) {
        const int2 v = sacc[lane];
        sacc[lane] = make_int2(0, 0);
        if (v.x | v.y) { atomicAdd(acc + 2 * lane, v.x); atomicAdd(acc + 2 * lane + 1, v.y); }
      }
      __syncwarp();                                                    // the line is clean before the next tile's atomics
    }
    finish_stage(xs_w + (buf ^ 1) * pitch);                            // converted samples of the next tile (if any) go to its buffer now
  }
}

// host: q / d == (q * m) >> s for every q < 2^31 (Granlund-Montgomery with N = 31: m = floor(2^(31 + l) / d) + 1, l = ceil(log2 d))
void magic_div(uint32_t d, uint32_t *m, uint32_t *s) {
  uint32_t l = 0;
  while (((uint64_t)1 << l) < d) ++l;
  *m = (uint32_t)((((uint64_t)1 << (31 + l)) / d) + 1);
  *s = 31 + l;
}

template <int LP, int VAR, bool CONV>
int launch_warp(IqbbAccumArgs a, const IqbbTaps &taps, cudaStream_t st) {
  constexpr int NV = (LP + 7 + 3) / 4;
  constexpr int pitch = ((kWT - kR + 4 * NV) + 7) & ~7;
  const size_t smem = sizeof(int2) * 128 + sizeof(int2) * (kT / 32) * 32 + sizeof(uint32_t) * (kT / 32) * 2 * pitch;
  magic_div(a.ss, &a.div_m, &a.div_s);
  const unsigned n_tiles = (a.n + kWT - 1) / kWT, want = (n_tiles + kT / 32 - 1) / (kT / 32);
  return launch_persistent("iqbb_accum_int_warp_kernel", iqbb_accum_int_warp_kernel<LP, VAR, CONV>, want, kT, smem, st, a, taps);
}

template <int VAR, bool CONV>
int dispatch_warp(int lp, const IqbbAccumArgs &a, const IqbbTaps &taps, cudaStream_t st) {
  return dispatch(lp, int_range<2, 32, 2>{}, [&](auto LP) { return launch_warp<LP, VAR, CONV>(a, taps, st); }, [] { return -1; });
}

}  // namespace

int launch_iqbb_accum_warp(int scalar, const IqbbAccumArgs &a, const IqbbTaps &taps, int lp, cudaStream_t st) {
  if (a.ss < 16 || lp > 32) return -1;
  if (scalar == SDRG_T_S8) return dispatch_warp<1, false>(lp, a, taps, st);
  if (a.in_fmt == 4) return dispatch_warp<2, true>(lp, a, taps, st);
  // fused AutoCast (complex 8-bit samples, 2-byte loads + a conversion per sample): the CTA-wide kernel, whose staging
  // phase spreads that work over all warps at once, measured faster (195 against 170 GS/s at C1's shape)
  if (a.in_fmt != 0) return -1;
  // complex int16 samples: pick the cheapest exact form the taps allow
  bool real_taps = true, sym = true;
  for (int t = 0; t < lp; ++t) {
    const int4 c = taps.t[t];                       // {kr, ki - kr, kr + ki, 0}
    if (c.y != -c.x || c.z != c.x) real_taps = false;
    if (c.x != taps.t[lp - 1 - t].x) sym = false;
  }
  if (real_taps && sym) return dispatch_warp<4, false>(lp, a, taps, st);
  if (real_taps) return dispatch_warp<3, false>(lp, a, taps, st);
  return dispatch_warp<0, false>(lp, a, taps, st);
}

}  // namespace sdrg

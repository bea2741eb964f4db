// iqbb_fold_kernels.cu -- IQBaseBand<float>: the folded (HBM-bound) accumulate kernel.
//
// The float path is linear (no truncating shifts), so FIR -> NCO -> boxcar can be folded into one
// weight per input sample (SURVEY.md appendix C.5).  With c(n) = lut[idx(n)] the NCO factor and
// window W_m = [.., n_hi], sample p contributes  x[p] * sum_{n in W_m, p <= n <= p+L-1} c(n) k[L-1-(n-p)].
// The 15-bit phase factorises exactly: phi_p = 256 a + r  =>  c(p+d) = A(a) * B(r,d) with
// A(a) = exp(-/+ 2 pi i a/128) and B depending only on (r, d); hence
//     full weight      G(p)   = A(a_p) * U(r_p, 0)
//     tail past a window end at distance e = n_hi+1-p (1 <= e <= L-1):
//                      T_e(p) = A(a_b) * U(r_b, e),   phi_b = phase at the next window's first sample
//     U(r,e) = sum_{j=0}^{L-1-e} B(r,j) k[L-1-e-j]       (256 x L table, built on the host in double)
// Each sample is read ONCE and contributes (G - T) x to its own window and T x to the next one
// (requires ss >= L-1); no halo re-reads, no FIR history: 8 bytes and ~5 flop per sample.
//
// Mapping.  The unit of work is a chunk: a window (clipped to the call), or a <= `part`-sample
// piece of a long window.  A warp owns a run of consecutive chunks and walks each in steps of 32
// lanes aligned to the chunk start.  Lane l sees samples l, l+32, ...: its low phase byte r
// advances by 32*inc per step and so cycles with period <= 8 steps; the eight U(r,0) values a lane
// needs for a chunk live in registers and the window sum factorises per residue u = step mod 8:
//     S = sum_u H_u * ( sum_{steps = u mod 8} A(a_p) x[p] )  -  (tails sent ahead)  +  (tails received)
// i.e. per sample: one 8-byte streaming load, one lookup in a 1 KB table, one complex FMA.  Loads
// are issued 8 steps (2 KB per warp) ahead of their use.  Partial sums stay in registers; at a
// chunk end the warp reduces with shuffles and issues one RED.ADD per component into the per-call
// accumulators (finalized by iqbb_finalize_kernel); tails sent ahead are carried in registers into
// the next window when the same warp processes it.
#include "iqbb_fold_common.cuh"

namespace sdrg {
using namespace foldk;
namespace {

// Ragged batch of a complete window: RS steps, only the last one predicated (per-lane constant).
template <int RS>
__device__ __forceinline__ void ragged_batch(float2 (&R)[8], const float2 *__restrict__ xk, uint32_t ph, uint32_t inc32,
                                             const float2 *sA, bool last_ok) {
  float2 xv[RS];
#pragma unroll
  for (int u = 0; u + 1 < RS; ++u) xv[u] = ld_stream(xk + 32 * u);
  xv[RS - 1] = make_float2(0.f, 0.f);
  if (last_ok) xv[RS - 1] = ld_stream(xk + 32 * (RS - 1));
#pragma unroll
  for (int u = 0; u < RS; ++u) cfma(R[u], sA[((ph + u * inc32) & 0x7fffu) >> 8], xv[u]);
}

// Persistent grid (one CTA per resident slot); chunk ids are dealt round-robin to the warps of the
// whole grid, so that at any moment the running warps read ONE compact, linearly advancing region
// of the input (DRAM row locality, like a grid-stride loop) instead of thousands of separate fronts.
__global__ void __launch_bounds__(kFoldThreads, 4) iqbb_fold_f32_kernel(const IqbbFoldArgs a) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  __shared__ float2 sA[128];
  __shared__ float2 sH[256];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  // zero the next call's accumulators (see iqbb_kernels.cu)
  for (uint32_t k = blockIdx.x * blockDim.x + tid; k < a.zero_next; k += gridDim.x * blockDim.x)
    ((float2 *)a.acc_next)[k] = make_float2(0.f, 0.f);
  if (tid < 128) sA[tid] = a.tab_a[tid];
  sH[tid] = a.tab_u[(size_t)tid * a.taps_len];              // U(r, 0)
  __syncthreads();

  const uint32_t total_warps = gridDim.x * kFoldWarps;
  const uint32_t wg = warp * gridDim.x + blockIdx.x;        // neighbouring CTAs take neighbouring chunks
  const float2 *__restrict__ x = (const float2 *)a.x;
  float *acc_out = (float *)a.acc_cur;
  WarpStage stage{(float2 *)dyn_smem + (size_t)warp * kStageRows * kStagePitch, 0u, 0u};
  const int L1 = (int)a.taps_len - 1;
  const int win_off = (int)a.first - (int)a.r0;   // begin(s) = s*ss + win_off (s>0), end(s) = (s+1)*ss + win_off
  const uint32_t inc32 = (32u * a.inc) & 0x7fffu, inc256 = (256u * a.inc) & 0x7fffu;

  // per-lane constants of the interior-window schedule
  const bool fast_last_ok = (uint32_t)lane < a.fast_pl;
  const bool fast_t0 = lane < L1, fast_t1 = lane + 32 < L1;
  const int fast_tlo = (int)a.ss - L1;

  for (uint32_t id = wg; id < a.n_chunks; id += total_warps) {
    // Complete interior window (the common case): every bound is a launch constant, so the chunk
    // arithmetic, the ragged-batch predicates and the tail addressing of the general path below fold
    // into a handful of instructions -- the kernel is issue-limited, not byte-limited, beyond ~85 %
    // of HBM (profiles/r01_final_fold_probe.md).
    if (a.fast && id > 0 && (int)((id + 1) * a.ss) + win_off <= (int)a.n) {
      const int c_lo = (int)(id * a.ss) + win_off;
      const float2 *__restrict__ xc = x + c_lo + lane;
      uint32_t ph = (a.phase0 + (uint32_t)(c_lo + lane) * a.inc) & 0x7fffu;
      const uint32_t r0 = ph & 255u;
      float2 R[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) R[u] = make_float2(0.f, 0.f);
      const float2 *__restrict__ xk = xc;
      for (uint32_t b = 0; b < a.fast_nb; ++b, xk += 256, ph = (ph + inc256) & 0x7fffu) {
        float2 xv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) xv[u] = ld_stream(xk + 32 * u);
#pragma unroll
        for (int u = 0; u < 8; ++u) cfma(R[u], sA[((ph + u * inc32) & 0x7fffu) >> 8], xv[u]);
      }
      // tails owed to the next window: loads issued together with the ragged batch
      const uint32_t pb = (a.phase0 + (uint32_t)(c_lo + (int)a.ss) * a.inc) & 0x7fffu;
      const float2 Ab = sA[pb >> 8];
      const float2 *__restrict__ ue = a.tab_u + (size_t)(pb & 255u) * a.taps_len + (L1 - lane);   // U(r_b, e), e = L1 - lane
      float2 xt0 = make_float2(0.f, 0.f), xt1 = xt0, ut0 = xt0, ut1 = xt0;
      if (fast_t0) { xt0 = __ldg(xc + fast_tlo); ut0 = __ldg(ue); }
      if (fast_t1) { xt1 = __ldg(xc + fast_tlo + 32); ut1 = __ldg(ue - 32); }
      switch (a.fast_rs) {
        case 1: ragged_batch<1>(R, xk, ph, inc32, sA, fast_last_ok); break;
        case 2: ragged_batch<2>(R, xk, ph, inc32, sA, fast_last_ok); break;
        case 3: ragged_batch<3>(R, xk, ph, inc32, sA, fast_last_ok); break;
        case 4: ragged_batch<4>(R, xk, ph, inc32, sA, fast_last_ok); break;
        case 5: ragged_batch<5>(R, xk, ph, inc32, sA, fast_last_ok); break;
        case 6: ragged_batch<6>(R, xk, ph, inc32, sA, fast_last_ok); break;
        case 7: ragged_batch<7>(R, xk, ph, inc32, sA, fast_last_ok); break;
        case 8: ragged_batch<8>(R, xk, ph, inc32, sA, fast_last_ok); break;
        default: break;
      }
      float2 sent = make_float2(0.f, 0.f);
      cfma(sent, cmul(Ab, ut0), xt0);     // zero when this lane has no such sample
      cfma(sent, cmul(Ab, ut1), xt1);
      float2 tot = make_float2(-sent.x, -sent.y);
#pragma unroll
      for (int u = 0; u < 8; ++u) cfma(tot, sH[(r0 + u * inc32) & 255u], R[u]);
      stage.push(tot, id, lane, acc_out);
      if (L1 > 0) stage.push(sent, id + 1, lane, acc_out);
      continue;
    }
    fold_chunk_general(a, id, x, sA, sH, lane, L1, win_off, inc32, inc256, stage, acc_out);
  }
  stage.drain(lane, acc_out);

}

// ---- window-pipelined variant (ss <= 512, taps <= 65) ---------------------------------------------
// A complete interior window is S = ceil(ss/32) steps, fully unrolled.  The warp keeps the S loads of
// its NEXT window in flight while it works on the current one: step i consumes ring[i] and at once
// re-issues ring[i] for step i of the next window, so the number of outstanding loads per warp is
// constant (S x 256 B) and a window costs no exposed memory round trip -- the two per window of the
// batched schedule above were what kept it at ~92 % of HBM.  Edge chunks (window 0, the clipped
// last window) go through fold_chunk_general.
template <int S, int TS = 3>     // TS: ring steps that can hold tail samples (3: taps <= 65, 5: taps <= 129)
__global__ void __launch_bounds__(kFoldThreads, S <= 8 ? 4 : (S <= 13 ? 3 : 2)) iqbb_fold_f32_win_kernel(const IqbbFoldArgs a) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  __shared__ float2 sA[128];
  __shared__ float2 sH[256];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (uint32_t k = blockIdx.x * blockDim.x + tid; k < a.zero_next; k += gridDim.x * blockDim.x)
    ((float2 *)a.acc_next)[k] = make_float2(0.f, 0.f);
  if (tid < 128) sA[tid] = a.tab_a[tid];
  sH[tid] = a.tab_u[(size_t)tid * a.taps_len];
  __syncthreads();

  const uint32_t wg = warp * gridDim.x + blockIdx.x;
  const float2 *__restrict__ x = (const float2 *)a.x;
  float *acc_out = (float *)a.acc_cur;
  WarpStage stage{(float2 *)dyn_smem + (size_t)warp * kStageRows * kStagePitch, 0u, 0u};
  const int L1 = (int)a.taps_len - 1;
  const int win_off = (int)a.first - (int)a.r0;
  const uint32_t inc32 = (32u * a.inc) & 0x7fffu, inc256 = (256u * a.inc) & 0x7fffu;
  const bool last_ok = (uint32_t)lane < a.fast_pl;
  int te[TS]; bool te_ok[TS];                 // tail distance of this lane's sample in ring step S-1-k
#pragma unroll
  for (int k = 0; k < TS; ++k) { te[k] = (int)a.ss - 32 * (S - 1 - k) - lane; te_ok[k] = te[k] >= 1 && te[k] <= L1; }

  // Edge chunks (window 0, the clipped last window and the tails behind it) are dealt statically ...
  if (wg == 0) fold_chunk_general(a, 0u, x, sA, sH, lane, L1, win_off, inc32, inc256, stage, acc_out);
  else if (a.fast_hi + wg < a.n_chunks) fold_chunk_general(a, a.fast_hi + wg, x, sA, sH, lane, L1, win_off, inc32, inc256, stage, acc_out);
  // ... the complete interior windows 1..fast_hi dynamically, kWorkChunk consecutive windows per grab of a
  // global counter: a CTA that becomes resident late (another kernel -- e.g. a collective -- holding part of
  // the SMs) or runs on a slower SM simply takes fewer windows, and ids still advance in address order.
  // The grab for the chunk after next is issued one chunk ahead and only read when it is needed.
  const uint32_t kWorkChunk = a.work_chunk;
  const uint32_t n_work = (a.fast_hi + kWorkChunk - 1) / kWorkChunk;
  uint32_t grabbed = 0;
  if (lane == 0) grabbed = atomicAdd(a.work, 1u);
  const uint32_t c0 = __shfl_sync(kFull, grabbed, 0);
  if (c0 < n_work) {
    uint32_t id = 1 + c0 * kWorkChunk, end = min(id + kWorkChunk, a.fast_hi + 1);
    if (lane == 0) grabbed = atomicAdd(a.work, 1u);               // pending: not read before this chunk's last window
    const float2 *__restrict__ xc = x + ((int)(id * a.ss) + win_off) + lane;
    float2 ring[S];
#pragma unroll
    for (int i = 0; i + 1 < S; ++i) ring[i] = ld_stream(xc + 32 * i);
    ring[S - 1] = make_float2(0.f, 0.f);
    if (last_ok) ring[S - 1] = ld_stream(xc + 32 * (S - 1));
    float2 carry = make_float2(0.f, 0.f);
    for (;;) {
      uint32_t nid = id + 1;
      bool more = nid < end, switched = false;
      if (!more) {
        const uint32_t cn = __shfl_sync(kFull, grabbed, 0);
        if (cn < n_work) { nid = 1 + cn * kWorkChunk; more = true; switched = true; }
      }
      const int c_lo = (int)(id * a.ss) + win_off;
      const float2 *__restrict__ xn = x + ((int)(nid * a.ss) + win_off) + lane;
      const uint32_t ph = a.phase0 + (uint32_t)(c_lo + lane) * a.inc;      // only bits 0..14 are used
      const uint32_t pb = a.phase0 + (uint32_t)(c_lo + (int)a.ss) * a.inc;
      // Tails owed to the next window: the last L-1 samples of the window sit in the last (up to TS)
      // ring steps already, so only their weights U(r_b, e), e = ss - 32 i - lane, are fetched (issued
      // now, used ~a window later).  e and its validity are per-lane constants of the launch.
      const float2 Ab = sA[(pb & 0x7fffu) >> 8];
      const float2 *__restrict__ urow = a.tab_u + (size_t)(pb & 255u) * a.taps_len;
      float2 ut[TS];
#pragma unroll
      for (int k = 0; k < TS; ++k) {
        ut[k] = make_float2(0.f, 0.f);
        if (k < S && te_ok[k]) ut[k] = __ldg(urow + te[k]);
      }
      float2 R[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) R[u] = make_float2(0.f, 0.f);
      float2 ts = make_float2(0.f, 0.f);
#pragma unroll
      for (int i = 0; i < S; ++i) {
        cfma(R[i & 7], sA[((ph + i * inc32) & 0x7fffu) >> 8], ring[i]);
        if (S - 1 - i < TS) cfma(ts, ut[S - 1 - i], ring[i]);    // zero weight outside the tail
        if (more) {
          if (i + 1 < S) ring[i] = ld_stream(xn + 32 * i);
          else if (last_ok) ring[i] = ld_stream(xn + 32 * i);    // lanes past the window keep their zero
        }
      }
      const float2 sent = cmul(Ab, ts);
      float2 tot = make_float2(-sent.x, -sent.y);
      const uint32_t r0 = ph & 255u;
#pragma unroll
      for (int u = 0; u < 8; ++u) cfma(tot, sH[(r0 + u * inc32) & 255u], R[u]);
      // the tails this window owes to the next one stay in registers while the warp walks consecutive windows
      // (15 of 16): one staged row per window instead of two
      tot.x += carry.x; tot.y += carry.y;
      stage.push(tot, id, lane, acc_out);
      carry = sent;
      if ((!more || switched) && L1 > 0) { stage.push(carry, id + 1, lane, acc_out); carry = make_float2(0.f, 0.f); }
      if (!more) break;
      if (switched) {
        end = min(nid + kWorkChunk, a.fast_hi + 1);
        if (lane == 0) grabbed = atomicAdd(a.work, 1u);
      }
      id = nid;
    }
  }
  stage.drain(lane, acc_out);
}

template <int S, int TS = 3>
static int launch_fold_win_s(const IqbbFoldArgs &a, cudaStream_t st) {
  const size_t smem = (size_t)kFoldWarps * kStageRows * kStagePitch * sizeof(float2);
  const uint64_t want = ((uint64_t)a.n_chunks + kFoldWarps - 1) / kFoldWarps;
  return launch_persistent("iqbb_fold_f32_win_kernel", iqbb_fold_f32_win_kernel<S, TS>, want, kFoldThreads, smem, st, a);
}

static int launch_fold_win(const IqbbFoldArgs &a, cudaStream_t st) {
  const int s = (int)((a.ss + 31) / 32);
  if (a.taps_len > 65)        // 66..129 taps: the tail reaches back up to five ring steps (ss >= taps - 1 >= 65, so S >= 3)
    return dispatch(s, int_range<3, 16>{}, [&](auto S) { return launch_fold_win_s<S, 5>(a, st); }, [] {
      return set_error(SDRG_ERR_RUNTIME, "IQBaseBand<float>: window-pipelined kernel needs 65 <= sub_sample <= 512 for more than 65 taps");
    });
  return dispatch(s, int_range<1, 16>{}, [&](auto S) { return launch_fold_win_s<S>(a, st); },
                  [] { return set_error(SDRG_ERR_RUNTIME, "IQBaseBand<float>: window-pipelined kernel needs sub_sample <= 512"); });
}

// ---- short windows (2 <= ss < 128) ------------------------------------------------------------------
// With few samples per window the per-window cost of the residue scheme above (eight H_u products, the
// tail set-up, two staged rows) dominates, so here every sample gets its complete weight instead:
//     own window   z_o = (G(p) - T_e(p)) x[p],   G = A(a_p) U(r_p, 0)
//     next window  z_n = T_e(p) x[p]   for the last L-1 samples of a window,  T_e = A(a_b) U(r_b, e), phase_b = phase_p + e inc
// (two table lookups and two complex products per sample, one more pair on tail samples).  The weighted
// samples of a 2048-sample tile are staged in shared memory and summed per window by 1, 2 or 4 threads,
// like the integer kernels do.  Loads are coalesced 8-byte streams, 8 per thread in flight.
constexpr int kSmallTile = 2048;

__global__ void __launch_bounds__(kFoldThreads, 4) iqbb_fold_f32_small_kernel(const IqbbFoldArgs a) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  __shared__ float2 sA[128];
  __shared__ float2 sH[256];
  float2 *zo = (float2 *)dyn_smem, *zn = zo + kSmallTile;
  const int tid = threadIdx.x;
  for (uint32_t k = blockIdx.x * blockDim.x + tid; k < a.zero_next; k += gridDim.x * blockDim.x)
    ((float2 *)a.acc_next)[k] = make_float2(0.f, 0.f);
  if (tid < 128) sA[tid] = a.tab_a[tid];
  sH[tid] = a.tab_u[(size_t)tid * a.taps_len];
  __syncthreads();

  const float2 *__restrict__ x = (const float2 *)a.x;
  float *acc = (float *)a.acc_cur;
  const uint32_t ss = a.ss, L = a.taps_len, L1 = L - 1;
  const uint64_t magic = ((1ull << 40) + ss - 1) / ss;     // q / ss == (q * magic) >> 40 for q < 2^31, ss < 2^9
  const int win_off = (int)a.first - (int)a.r0;            // begin(s) = s*ss + win_off (s>0), end(s) = (s+1)*ss + win_off
  const int gsh = ss >= 32 ? 2 : (ss >= 16 ? 1 : 0), G = 1 << gsh, sub = tid & (G - 1);
  const uint32_t n_tiles = (a.n + kSmallTile - 1) / kSmallTile;
  const uint32_t d256 = 256u % ss, inc256 = 256u * a.inc;

  float2 xv[8];
  auto load_tile = [&](uint32_t t) {                         // 8 coalesced streaming loads per thread
    const uint32_t b0 = t * kSmallTile, hi = min(a.n - b0, (uint32_t)kSmallTile);
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const uint32_t o = tid + 256 * r;
      xv[r] = make_float2(0.f, 0.f);
      if (o < hi) xv[r] = ld_stream(x + b0 + o);
    }
  };
  if (blockIdx.x < n_tiles) load_tile(blockIdx.x);
  for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const uint32_t base = t * kSmallTile;
    const uint32_t t_hi = min(a.n - base, (uint32_t)kSmallTile);
    // position inside its window of this thread's first sample (one division per tile), then +256 per step
    const uint32_t p0 = base + tid;
    const uint32_t q0 = a.r0 + p0 - ((a.first && p0 > 0) ? 1u : 0u);
    uint32_t m = q0 - (uint32_t)(((uint64_t)q0 * magic) >> 40) * ss;
    if (a.first && p0 == 0) m = ss - 1;                       // q(0) = q(1) = 0: sample 0 counts as position -1 (its e is set below)
    uint32_t ph = a.phase0 + p0 * a.inc;                      // bits 0..14 are the phase
#pragma unroll
    for (int r = 0; r < 8; ++r, ph += inc256) {
      const uint32_t o = tid + 256 * r;
      float2 vo = make_float2(0.f, 0.f), vn = vo;
      if (o < t_hi) {
        float2 g = cmul(sA[(ph & 0x7fffu) >> 8], sH[ph & 255u]);
        uint32_t e = ss - m;                                  // samples up to and including the window's last one
        if (a.first && base + o == 0) e = ss + 1;             // the extra first sample of window 0
        if (e <= L1) {
          const uint32_t pb = ph + e * a.inc;                 // phase of the next window's first sample
          const float2 tw = cmul(sA[(pb & 0x7fffu) >> 8], __ldg(a.tab_u + (size_t)(pb & 255u) * L + e));
          vn = cmul(tw, xv[r]);
          g.x -= tw.x; g.y -= tw.y;
        }
        vo = cmul(g, xv[r]);
      }
      m += d256; if (m >= ss) m -= ss;                        // (m + 256) mod ss, d256 = 256 mod ss
      zo[o] = vo; zn[o] = vn;
    }
    __syncthreads();
    if (t + gridDim.x < n_tiles) load_tile(t + gridDim.x);     // in flight while the windows of this tile are summed
    // per-window sums of the tile: G threads per window (outer bound CTA-uniform)
    {
      const uint32_t q_lo = a.r0 + base - ((a.first && base > 0) ? 1u : 0u);
      const uint32_t q_hi = a.r0 + (base + t_hi - 1) - ((a.first && base + t_hi - 1 > 0) ? 1u : 0u);
      const uint32_t slot_lo = (uint32_t)(((uint64_t)q_lo * magic) >> 40), slot_hi = (uint32_t)(((uint64_t)q_hi * magic) >> 40);
      for (uint32_t sb = slot_lo; sb <= slot_hi; sb += kFoldThreads >> gsh) {
        const uint32_t sl = sb + (uint32_t)(tid >> gsh);
        float sr = 0.f, si = 0.f, tr = 0.f, ti = 0.f;
        if (sl <= slot_hi) {
          const int64_t wb = sl == 0 ? 0 : (int64_t)sl * ss + win_off, we = (int64_t)(sl + 1) * ss + win_off;
          const int lo = (int)max(wb - (int64_t)base, (int64_t)0), hi = (int)min(we - (int64_t)base, (int64_t)t_hi);
          for (int o = lo + sub; o < hi; o += G) { const float2 z = zo[o]; sr += z.x; si += z.y; }
          const int tl = (int)max((int64_t)lo, we - (int64_t)L1 - (int64_t)base);
          for (int o = tl + sub; o < hi; o += G) { const float2 z = zn[o]; tr += z.x; ti += z.y; }
        }
        for (int d = G >> 1; d > 0; d >>= 1) {
          sr += __shfl_xor_sync(kFull, sr, d); si += __shfl_xor_sync(kFull, si, d);
          tr += __shfl_xor_sync(kFull, tr, d); ti += __shfl_xor_sync(kFull, ti, d);
        }
        if (sub == 0 && sl <= slot_hi) {
          if (sr != 0.f || si != 0.f) { atomicAdd(acc + 2 * (size_t)sl, sr); atomicAdd(acc + 2 * (size_t)sl + 1, si); }
          if (tr != 0.f || ti != 0.f) { atomicAdd(acc + 2 * (size_t)sl + 2, tr); atomicAdd(acc + 2 * (size_t)sl + 3, ti); }
        }
      }
    }
    __syncthreads();
  }
}

static int launch_fold_small(const IqbbFoldArgs &a, cudaStream_t st) {
  const uint64_t n_tiles = ((uint64_t)a.n + kSmallTile - 1) / kSmallTile;
  return launch_persistent("iqbb_fold_f32_small_kernel", iqbb_fold_f32_small_kernel, n_tiles, kFoldThreads, (size_t)2 * kSmallTile * sizeof(float2), st, a);
}

}  // namespace

// Grids are sized to the machine: 148 SMs x 3 resident CTAs of 8 warps.
int launch_iqbb_fold(const IqbbFoldArgs &a_in, cudaStream_t st, int *which_out) {
  int which_local = 0;
  int *which = which_out ? which_out : &which_local;
  if (a_in.n == 0) return SDRG_OK;
  IqbbFoldArgs a = a_in;
  // slots touched by this call: slot of the last sample + 1
  const uint64_t q_last = (uint64_t)a.r0 + (a.n - 1) - ((a.first && a.n > 1) ? 1 : 0);
  const uint64_t n_slots = q_last / a.ss + 1;
  a.part = 8192;
  a.cpw = (uint32_t)(((uint64_t)a.ss + 1 + a.part - 1) / a.part);
  const uint64_t n_chunks = n_slots * a.cpw;
  if (n_chunks > 0xffffffffull) return set_error(SDRG_ERR_RUNTIME, "IQBaseBand<float>: too many windows in one call");
  a.n_chunks = (uint32_t)n_chunks;
  a.fast = (a.cpw == 1 && a.taps_len <= 65 && a.ss + 1 >= a.taps_len) ? 1u : 0u;   // batched kernel: two tail steps
  const bool win_ok = a.cpw == 1 && a.taps_len <= 129 && a.ss + 1 >= a.taps_len && a.ss <= 512;   // window-pipelined: up to five
  a.fast_nb = a.ss / 256;
  a.fast_rs = (a.ss % 256 + 31) / 32;
  a.fast_pl = a.ss % 32 ? a.ss % 32 : 32;
  a.fast_hi = 0;
  if (a.fast || win_ok) {      // ids 1..fast_hi: (id + 1) * ss + first - r0 <= n
    const int64_t hi = ((int64_t)a.n + (int64_t)a.r0 - (int64_t)a.first) / (int64_t)a.ss - 1;
    a.fast_hi = hi >= 1 ? (uint32_t)hi : 0u;
  }
  a.work_chunk = 16;
  if (a.cpw == 1 && fold_perwin_eligible(a)) { *which = 5; return launch_fold_perwin(a, st); }
  // ss <= 55: the short-window kernel (measured crossover with the window-pipelined one)
  if (a.cpw == 1 && a.ss + 1 >= a.taps_len && a.ss <= 55) { *which = 4; return launch_fold_small(a, st); }
  if (win_ok && a.fast_hi >= 1) { *which = 3; return launch_fold_win(a, st); }
  *which = 2;
  const size_t smem = (size_t)kFoldWarps * kStageRows * kStagePitch * sizeof(float2);
  return launch_persistent("iqbb_fold_f32_kernel", iqbb_fold_f32_kernel, (n_chunks + kFoldWarps - 1) / kFoldWarps, kFoldThreads, smem, st, a);
}

}  // namespace sdrg

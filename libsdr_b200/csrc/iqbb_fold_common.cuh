// iqbb_fold_common.cuh -- helpers shared by the folded float kernels (iqbb_fold_kernels.cu, iqbb_fold_perwin.cu).
// See iqbb_fold_kernels.cu for the method.
#pragma once
#include "iqbb_kernels.cuh"
#include "launch.cuh"

namespace sdrg {
namespace foldk {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kFoldThreads = 256;
constexpr int kFoldWarps = kFoldThreads / 32;

__device__ __forceinline__ float2 ld_stream(const float2 *p) {
  float2 v;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
  return v;
}
__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
  return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
// acc += w x (complex) as two packed FP32 FMAs (sm_100 FFMA2: the half swap and the sign of one half are operand
// modifiers): half the issue slots of four scalar FFMA at the same FMA-pipe time.  These kernels run 16-32 warps per SM
// and are issue-limited once the SM clock drops under the power cap, so this is what keeps them on the HBM roofline
// (C2 sustained: 0.959 -> 0.987 of the measured peak).
__device__ __forceinline__ void cfma(float2 &acc, float2 w, float2 x) {
  acc = __ffma2_rn(x, make_float2(w.x, w.x), acc);
  acc = __ffma2_rn(make_float2(-x.y, x.x), make_float2(w.y, w.y), acc);
}
__device__ __forceinline__ void flush(float *acc, uint32_t slot, float2 v, int lane) {
  const float sr = warp_sum(v.x), si = warp_sum(v.y);
  if (lane == 0 && (sr != 0.f || si != 0.f)) { atomicAdd(acc + 2 * (size_t)slot, sr); atomicAdd(acc + 2 * (size_t)slot + 1, si); }
}

// Per-warp staging of window partials: row w holds the 32 per-lane partial sums of the w-th window
// this warp finished; once 32 rows are full lane l sums row l (one LDS.64 per element, rows padded
// to 33 to stay conflict free) and issues the RED.ADDs for its window.  This replaces a 5-step
// shuffle reduction per component per window by ~3 instructions per window.
constexpr int kStageRows = 16, kStagePitch = 33;

struct WarpStage {
  float2 *rows;      // [kStageRows][kStagePitch]
  uint32_t my_slot;  // lane l: slot of row l
  uint32_t count;
  __device__ __forceinline__ void push(float2 v, uint32_t slot, int lane, float *acc_out) {
    rows[count * kStagePitch + lane] = v;
    if ((uint32_t)lane == count) my_slot = slot;
    if (++count == kStageRows) drain(lane, acc_out);
  }
  __device__ __forceinline__ void drain(int lane, float *acc_out) {
    __syncwarp();
    if ((uint32_t)lane < count) {
      float sr = 0.f, si = 0.f;
      const float2 *r = rows + lane * kStagePitch;
#pragma unroll 8
      for (int i = 0; i < 32; ++i) { const float2 v = r[i]; sr += v.x; si += v.y; }   // the 32 lane partials of row `lane`
      if (sr != 0.f || si != 0.f) { atomicAdd(acc_out + 2 * (size_t)my_slot, sr); atomicAdd(acc_out + 2 * (size_t)my_slot + 1, si); }
    }
    __syncwarp();
    count = 0;
  }
};

// chunk id -> (slot, first sample, length, tail start); false for an empty piece
struct Chunk { uint32_t s; int c_lo, len, t_lo, full_end; };
__device__ __forceinline__ bool chunk_of(const IqbbFoldArgs &a, uint32_t id, int win_off, int L1, Chunk &c) {
  const uint32_t s = a.cpw == 1 ? id : id / a.cpw, part = a.cpw == 1 ? 0u : id % a.cpw;
  c.s = s;
  c.full_end = (int)((s + 1) * a.ss) + win_off;                          // exclusive, may exceed n
  const int w_lo = s == 0 ? 0 : (int)(s * a.ss) + win_off;
  const int w_hi = min(c.full_end, (int)a.n);
  c.c_lo = w_lo + (int)(part * a.part);
  if (c.c_lo >= w_hi) return false;
  c.len = min(c.c_lo + (int)a.part, w_hi) - c.c_lo;
  c.t_lo = max(0, min(c.len, c.full_end - L1 - c.c_lo));                 // samples >= t_lo send a tail ahead
  return true;
}

// One chunk on the general path: any clipping, any piece of a long window, any tap count.
// `what`: bit 0 = add the samples' contributions to their own window, bit 1 = add the tails they owe to the next one
// (the per-window kernel computes whole windows itself and needs only one of the two from its neighbours);
// STAGED = false reduces with shuffles and issues the RED.ADDs at once (no per-warp staging rows needed).
template <bool STAGED = true>
__device__ __forceinline__ void fold_chunk_general(const IqbbFoldArgs &a, const uint32_t id,
                                                   const float2 *__restrict__ x, const float2 *sA, const float2 *sH,
                                                   const int lane, const int L1, const int win_off,
                                                   const uint32_t inc32, const uint32_t inc256,
                                                   WarpStage &stage, float *acc_out, const uint32_t what = 3u) {
    Chunk c;
    if (!chunk_of(a, id, win_off, L1, c)) return;
    const int len = c.len;
    uint32_t ph = (a.phase0 + (uint32_t)(c.c_lo + lane) * a.inc) & 0x7fffu;         // this lane's phase in step 0
    const uint32_t r0 = ph & 255u;        // low phase byte in step 0; step u has (r0 + u*inc32) & 255 in every batch
    float2 R[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) R[u] = make_float2(0.f, 0.f);
    const float2 *__restrict__ xc = x + c.c_lo + lane;

    // every sample: R_u += A(a_p) x[p]   (its full weight G = H_u A)
    int k = 0;
    for (; k + 256 <= len; k += 256, ph = (ph + inc256) & 0x7fffu) {
      float2 xv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) xv[u] = ld_stream(xc + k + 32 * u);
#pragma unroll
      for (int u = 0; u < 8; ++u) cfma(R[u], sA[((ph + u * inc32) & 0x7fffu) >> 8], xv[u]);
    }
    // The last L-1 samples of the window also owe T_e x to the next window.  Their loads (a re-read
    // of x, L2 resident, and the U(r_b, e) row) are issued together with the ragged batch so that
    // the window costs two memory round trips, not three.
    float2 sent = make_float2(0.f, 0.f);
    const bool has_tail = c.t_lo < len;
    const int jt = c.t_lo + lane;                                   // this lane's first tail sample
    float2 Ab = make_float2(0.f, 0.f), xt0 = Ab, xt1 = Ab, ut0 = Ab, ut1 = Ab;
    const float2 *__restrict__ ue = a.tab_u;
    if (has_tail) {
      const uint32_t pb = (a.phase0 + (uint32_t)c.full_end * a.inc) & 0x7fffu;
      Ab = sA[pb >> 8];
      ue = a.tab_u + (size_t)(pb & 255u) * a.taps_len + (c.full_end - c.c_lo - lane);   // U(r_b, e), e = end - j
      if (jt < len) { xt0 = __ldg(xc + (jt - lane)); ut0 = __ldg(ue - (jt - lane)); }
      if (jt + 32 < len) { xt1 = __ldg(xc + (jt + 32 - lane)); ut1 = __ldg(ue - (jt + 32 - lane)); }
    }
    if (k < len) {                        // ragged last batch
      const int rem = len - k;
      float2 xv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        xv[u] = make_float2(0.f, 0.f);
        if (32 * u < rem && 32 * u + lane < rem) xv[u] = ld_stream(xc + k + 32 * u);
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (32 * u >= rem) break;
        cfma(R[u], sA[((ph + u * inc32) & 0x7fffu) >> 8], xv[u]);
      }
    }
    if (has_tail) {
      cfma(sent, cmul(Ab, ut0), xt0);     // zero when this lane has no such sample
      cfma(sent, cmul(Ab, ut1), xt1);
      for (int j = jt + 64; j < len; j += 32)       // L > 65 only
        cfma(sent, cmul(Ab, __ldg(ue - (j - lane))), __ldg(xc + (j - lane)));
    }
    float2 tot = make_float2(-sent.x, -sent.y);
#pragma unroll
    for (int u = 0; u < 8; ++u) cfma(tot, sH[(r0 + u * inc32) & 255u], R[u]);   // H_u = U(r_u, 0)
    if (STAGED) {
      if (what & 1u) stage.push(tot, c.s, lane, acc_out);
      if (c.t_lo < len && (what & 2u)) stage.push(sent, c.s + 1, lane, acc_out);
    } else {
      if (what & 1u) flush(acc_out, c.s, tot, lane);
      if (c.t_lo < len && (what & 2u)) flush(acc_out, c.s + 1, sent, lane);
    }
}


}  // namespace foldk

// iqbb_fold_perwin.cu: whole windows per thread group (short windows); false when the call has no eligible window
bool fold_perwin_eligible(IqbbFoldArgs &a);
int launch_fold_perwin(const IqbbFoldArgs &a, cudaStream_t st);

}  // namespace sdrg

// iqbb_fold_perwin.cu -- IQBaseBand<float>, short windows (ss <= 256): one whole window per thread group.
//
// The per-sample weights of iqbb_fold_kernels.cu cost two table look-ups and two complex products per sample;
// for a window of a few dozen samples that set-up, not HBM, is the bound (0.20-0.37 of the roofline).  Regrouped
// by window, the same folded sum reads
//     out[w] = A(a_b) * sum_{j=0}^{ss+L-2} V(r_b, j) * x[n_b - (L-1) + j],     256 a_b + r_b = phase at n_b,
//     V(r, j) = sum_{d = max(0, j-L+1)}^{min(j, ss-1)} B(r, d) k[j-d],         B(r, d) = lut[((r + d inc) >> 8) & 127]
// (n_b = first sample of the window; this is SURVEY.md appendix C.5's g_m with the phase factored out exactly).
// B(r, d) = B0(d) * rho^carry(r, d) with carry(r, d) = [r + (d inc & 255) >= 256], so V(r, .) changes only where r
// crosses one of at most ss thresholds: there are <= ss + 1 DISTINCT rows, not 256, and the whole table
// ((ss+1)(ss+L-1) float2) fits into shared memory for the window lengths this kernel is for.  Per multiply-add:
// one LDS of x, one LDS of V, four FFMA -- (ss+L-1)/ss of them per input sample, no per-sample index arithmetic.
//
// Mapping.  Tiles of consecutive windows (+ L-1 halo, read once from HBM) go through two shared-memory buffers per
// thread group, so the copy of the next tile is in flight while one is summed.  The shared-memory pipe is what bounds
// these kernels (16 bytes of LDS per multiply-add), so both mappings are built around conflict-free accesses:
//  * ss >= 23 (iqbb_fold_f32_perwin16_kernel<K>, K = 1, 2, 4): a half warp per window, lanes over j.  x and V are read
//    as 16 consecutive float2 (no conflicts, no padding, halo and window contiguous), every half warp sums K windows one
//    after the other and the 16 x K partial sums are combined by a transposed reduction (K/2 + K/4 + ... + 4 shuffles
//    per component instead of 4 K).  The V table exists once per CTA and can take most of the shared memory, so there
//    is ONE CTA per SM, split into up to four groups of 256 threads that run independent tile pipelines (own buffers,
//    own mbarriers, own named barrier) -- several "CTAs" sharing one table.  Tiles are staged by 1-D bulk copies
//    (cp.async.bulk, SASS UBLKCP): no LSU issue slots, no registers.
//  * ss <= 22 (iqbb_fold_f32_perwin1_kernel): a thread per window (a reduction per window would cost more than the
//    window); windows are laid out with an odd pitch ss + delta so that the 16 lanes of a half warp hit 16 different
//    banks, and for ss <= 16 the rows of V land in different banks as well (measured crossover with the half-warp mapping: ss = 23); tiles are staged with 8-byte cp.async.
// A window whose halo is inside the call is summed and STORED by its thread group alone (nothing else contributes to
// its slot); the first and last windows of a call -- cut by the call boundary -- take the per-sample path of
// fold_chunk_general(), restricted to the (sample, window) pairs the whole windows do not cover.
#include "iqbb_fold_common.cuh"

namespace sdrg {
using namespace foldk;
namespace {


struct PerwinGeom {
  uint32_t n_tiles, pitch, delta, magic;    // thread-per-window layout: window pitch ss + delta, magic = ceil(2^32 / ss)
  uint32_t n_edge;                          // edge chunks: ids 0..d_lo-1 and d_hi..n_chunks-1
  uint32_t x_tile;                          // float2 elements of one staged tile (even)
  uint32_t stages;                          // ring depth, 2 or 3
  uint32_t chunk;                           // thread-per-window staging: samples per half warp (see issue_tile)
};

__device__ __forceinline__ void cp_async8(float2 *dst_smem, const float2 *src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}

// 1-D bulk async copies (TMA, SASS UBLKCP) completing on an mbarrier: the staging of the half-warp kernels costs no
// LSU issue slots and no registers (an 8-byte LDGSTS occupies the LSU pipe for ~8 cycles per warp instruction)
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  } while (!ok);
}
constexpr int kPwBulk = 512;               // samples per bulk copy (4 KB)

__device__ __forceinline__ void mac_run(float2 &a0, float2 &a1, const float2 *__restrict__ pv, const float2 *__restrict__ px, int cnt) {
  int t = 0;
  for (; t + 4 <= cnt; t += 4, pv += 4, px += 4) {
    const float2 v0 = pv[0], v1 = pv[1], v2 = pv[2], v3 = pv[3];
    const float2 x0 = px[0], x1 = px[1], x2 = px[2], x3 = px[3];
    cfma(a0, v0, x0); cfma(a1, v1, x1); cfma(a0, v2, x2); cfma(a1, v3, x3);
  }
  for (; t < cnt; ++t, ++pv, ++px) cfma(a0, pv[0], px[0]);
}

// Transposed reduction of K accumulators over the 16 lanes of a half warp: each exchange halves the number of
// values a lane holds; afterwards lane l holds the total of window (l * K) >> 4 (replicated over 16/K lanes).
template <int K>
__device__ __forceinline__ float2 reduce16(float2 (&acc)[K], int l16) {
  int mask = 8;
#pragma unroll
  for (int cnt = K; cnt > 1; cnt >>= 1, mask >>= 1) {
    const bool upper = (l16 & mask) != 0;
#pragma unroll
    for (int i = 0; i < cnt / 2; ++i) {
      const float2 send = upper ? acc[i] : acc[i + cnt / 2], keep = upper ? acc[i + cnt / 2] : acc[i];
      acc[i].x = keep.x + __shfl_xor_sync(kFull, send.x, mask);
      acc[i].y = keep.y + __shfl_xor_sync(kFull, send.y, mask);
    }
  }
#pragma unroll
  for (; mask > 0; mask >>= 1) {
    acc[0].x += __shfl_xor_sync(kFull, acc[0].x, mask);
    acc[0].y += __shfl_xor_sync(kFull, acc[0].y, mask);
  }
  return acc[0];
}

// Prologue shared by both kernels: zero the next call's accumulators, copy the tables.
__device__ __forceinline__ void perwin_tables(const IqbbFoldArgs &a, float2 *sA, float2 *sH, uint16_t *sC, float2 *sV) {
  const uint32_t tid = threadIdx.x;
  for (uint32_t k = blockIdx.x * blockDim.x + tid; k < a.zero_next; k += gridDim.x * blockDim.x)
    ((float2 *)a.acc_next)[k] = make_float2(0.f, 0.f);
  if (tid < 128) sA[tid] = a.tab_a[tid];
  if (tid < 256) { sH[tid] = a.tab_u[(size_t)tid * a.taps_len]; sC[tid] = a.tab_cls[tid]; }
  for (uint32_t k = tid; k < a.v_rows * a.v_pitch; k += blockDim.x) sV[k] = a.tab_v[k];
}

// Edge chunks, one per warp of the last CTA: windows before d_lo keep their own sums (their tails into d_lo are
// part of that whole window), window d_hi only sends its tails ahead, everything behind it takes both.
__device__ __forceinline__ void perwin_edges(const IqbbFoldArgs &a, const PerwinGeom &geo, const float2 *sA, const float2 *sH) {
  if (blockIdx.x != gridDim.x - 1) return;
  const int lane = threadIdx.x & 31, L1 = (int)a.taps_len - 1, win_off = (int)a.first - (int)a.r0;
  const uint32_t inc32 = (32u * a.inc) & 0x7fffu, inc256 = (256u * a.inc) & 0x7fffu;
  WarpStage none{nullptr, 0u, 0u};
  for (uint32_t e = threadIdx.x >> 5; e < geo.n_edge; e += blockDim.x >> 5) {
    const uint32_t id = e < a.d_lo ? e : a.d_hi + (e - a.d_lo);
    const uint32_t what = e < a.d_lo ? (e + 1 < a.d_lo ? 3u : 1u) : (id == a.d_hi ? 2u : 3u);
    fold_chunk_general<false>(a, id, (const float2 *)a.x, sA, sH, lane, L1, win_off, inc32, inc256, none, (float *)a.acc_cur, what);
  }
}

// ---- ss <= 22: a thread per window -----------------------------------------------------------------------------
constexpr int kPw1Threads = 256;

__global__ void __launch_bounds__(kPw1Threads, 4) iqbb_fold_f32_perwin1_kernel(const IqbbFoldArgs a, const PerwinGeom geo) {
  constexpr int TW = kPw1Threads;                    // windows per tile
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  __shared__ float2 sA[128];
  __shared__ float2 sH[256];
  __shared__ uint16_t sC[256];
  float2 *sV = (float2 *)dyn_smem;
  float2 *sX = sV + (((size_t)a.v_rows * a.v_pitch + 1) & ~(size_t)1);
  const int tid = threadIdx.x;
  const float2 *__restrict__ x = (const float2 *)a.x;
  const int ss = (int)a.ss, L1 = (int)a.taps_len - 1;
  const int win_off = (int)a.first - (int)a.r0;
  const int pitch = (int)geo.pitch, delta = (int)geo.delta;
  const uint32_t stages = geo.stages;

  // tile t: windows s0 .. s0+nw-1, samples [s0*ss + win_off - L1, (s0+nw)*ss + win_off) -> ring buffer `stage`.
  // Padded layout: a half warp copies `chunk` consecutive samples whose positions span <= 16 slots, so that its 16
  // stores hit different banks (with 16 samples the first and last would collide across a window border).
  auto issue_tile = [&](uint32_t t, uint32_t stage) {
    if (t < geo.n_tiles) {
      const uint32_t s0 = a.d_lo + t * TW;
      const int nw = (int)min((uint32_t)TW, a.d_hi + 1 - s0);
      const int count = nw * ss + L1;
      float2 *dst = sX + (size_t)stage * geo.x_tile;
      const int chunk = (int)geo.chunk, per_pass = (kPw1Threads / 16) * chunk;
      const int m0 = (tid >> 4) * chunk + (tid & 15);
      if ((tid & 15) < chunk) {
        const float2 *__restrict__ xh = x + ((int64_t)s0 * ss + win_off - L1) + m0;
        for (int m = m0; m < count; m += per_pass, xh += per_pass)
          cp_async8(dst + m + delta * (int)__umulhi((uint32_t)(m + ss - L1), geo.magic), xh);
      }
    }
    cp_async_commit();                               // always: keeps the group count in step with the tiles
  };
  issue_tile(blockIdx.x, 0);                         // on their way while the tables are copied
  if (stages > 2) issue_tile(blockIdx.x + gridDim.x, 1);
  perwin_tables(a, sA, sH, sC, sV);
  __syncthreads();
  perwin_edges(a, geo, sA, sH);

  uint32_t stage = 0;
  for (uint32_t t = blockIdx.x; t < geo.n_tiles; t += gridDim.x) {
    if (stages > 2) cp_async_wait<1>(); else cp_async_wait<0>();    // this thread's copies of tile t have landed ...
    __syncthreads();                                                // ... everybody's have, and the buffer of tile t-1 is free
    issue_tile(t + (stages - 1) * gridDim.x, stage == 0 ? stages - 1 : stage - 1);
    const float2 *xs = sX + (size_t)stage * geo.x_tile;
    const uint32_t s0 = a.d_lo + t * TW;
    const int nw = (int)min((uint32_t)TW, a.d_hi + 1 - s0);
    if (tid < nw) {
      const uint32_t phb = a.phase0 + (uint32_t)((int)((s0 + tid) * a.ss) + win_off) * a.inc;   // bits 0..14: phase at the window's first sample
      const float2 *v = sV + (uint32_t)sC[phb & 255u] * a.v_pitch;
      float2 a0 = make_float2(0.f, 0.f), a1 = a0;
      mac_run(a0, a1, v, xs + tid * pitch, L1);                               // halo: the previous window's last L-1 samples
      mac_run(a0, a1, v + L1, xs + (L1 + delta + tid * pitch), ss);           // the window itself
      ((float2 *)a.acc_cur)[s0 + tid] = cmul(sA[(phb & 0x7fffu) >> 8], make_float2(a0.x + a1.x, a0.y + a1.y));
    }
    stage = stage + 1 == stages ? 0 : stage + 1;
  }
  cp_async_wait<0>();
}

// One window of a half warp, NS steps of 16 lanes fully unrolled (immediate offsets, no loop): the last step is the only
// one that can be partial.  NS = 0: any number of steps (loop).
template <int NS>
__device__ __forceinline__ float2 mac_window(const float2 *__restrict__ pv, const float2 *__restrict__ px, int n_steps, bool last_ok) {
  float2 b0 = make_float2(0.f, 0.f), b1 = b0;
  if (NS > 0) {
#pragma unroll
    for (int s = 0; s + 1 < NS; ++s) cfma((s & 1) ? b1 : b0, pv[16 * s], px[16 * s]);
    if (last_ok) cfma(((NS - 1) & 1) ? b1 : b0, pv[16 * (NS - 1)], px[16 * (NS - 1)]);
  } else {
    int s = 0;
    for (; s + 3 <= n_steps; s += 2, pv += 32, px += 32) {
      const float2 v0 = pv[0], v1 = pv[16], x0 = px[0], x1 = px[16];
      cfma(b0, v0, x0); cfma(b1, v1, x1);
    }
    if (s + 2 <= n_steps) { cfma(b0, pv[0], px[0]); pv += 16; px += 16; }
    if (last_ok) cfma(b1, pv[0], px[0]);
  }
  return make_float2(b0.x + b1.x, b0.y + b1.y);
}

// ---- ss >= 23: a half warp per window ----------------------------------------------------------------------------
// The V table exists once per CTA and can take most of the shared memory, so there is ONE CTA per SM; to keep the SM
// busy across tile hand-overs the CTA is split into groups of 256 threads that run independent tile pipelines (own ring
// of buffers, own mbarriers, own named barrier) -- several "CTAs" sharing one table.
constexpr int kPwGroup = 256;

template <int K>
__global__ void __launch_bounds__(1024, 1) iqbb_fold_f32_perwin16_kernel(const IqbbFoldArgs a, const PerwinGeom geo) {
  constexpr int TW = (kPwGroup / 16) * K;            // windows per tile (of one group)
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  __shared__ float2 sA[128];
  __shared__ float2 sH[256];
  __shared__ uint16_t sC[256];
  __shared__ __align__(8) uint64_t bars[4][3];
  float2 *sV = (float2 *)dyn_smem;
  const int tid = threadIdx.x, grp = tid / kPwGroup, gt = tid % kPwGroup, lane = tid & 31, gwarp = gt >> 5;
  const uint32_t stages = geo.stages;
  float2 *sX = sV + (((size_t)a.v_rows * a.v_pitch + 1) & ~(size_t)1) + (size_t)grp * stages * geo.x_tile;
  if (tid == 0) {
    for (int i = 0; i < 12; ++i) mbar_init(smem_u32(&bars[0][0] + i), 1);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  const float2 *__restrict__ x = (const float2 *)a.x;
  const int ss = (int)a.ss, L1 = (int)a.taps_len - 1, len = ss + L1;
  const int win_off = (int)a.first - (int)a.r0;
  const uint32_t n_groups = blockDim.x / kPwGroup;
  const uint32_t vcta = blockIdx.x * n_groups + grp, vgrid = gridDim.x * n_groups;     // tiles are dealt to the groups of the grid
  // bulk copies need 16-byte aligned addresses on both sides: sample i of a tile sits at element par + i of its buffer,
  // par = 1 when the tile's first sample is only 8-byte aligned (the same for every tile: a tile holds an even number of samples)
  const int par = (int)((reinterpret_cast<uintptr_t>(x + ((int64_t)a.d_lo * ss + win_off - L1)) >> 3) & 1u);

  // tile t: windows s0 .. s0+nw-1 -> elements par + [w ss, w ss + len) of ring buffer `stage`.  The group's first warp
  // issues the 16-byte aligned middle as bulk copies of 4 KB; an unaligned first / last sample is copied by a thread
  // (visible after the group's next barrier, which precedes the tile's use by at least one iteration).
  auto issue_tile = [&](uint32_t t, uint32_t stage) {
    if (t >= geo.n_tiles || gwarp > 1) return;
    const uint32_t s0 = a.d_lo + t * TW;
    const int nw = (int)min((uint32_t)TW, a.d_hi + 1 - s0);
    const int count = nw * ss + L1;
    const float2 *__restrict__ src0 = x + ((int64_t)s0 * ss + win_off - L1);
    float2 *dst = sX + (size_t)stage * geo.x_tile;
    const int n_bulk = (count - par) & ~1;
    if (gwarp == 0) {
      const uint32_t bar = smem_u32(&bars[grp][stage]);
      if (lane == 0) mbar_expect_tx(bar, (uint32_t)n_bulk * 8u);
      __syncwarp();
      for (int c = lane * kPwBulk; c < n_bulk; c += 32 * kPwBulk)
        tma_load_1d(smem_u32(dst + 2 * par + c), src0 + par + c, (uint32_t)min(kPwBulk, n_bulk - c) * 8u, bar);
    } else {
      if (lane == 0 && par) dst[1] = src0[0];
      if (lane == 1 && ((count - par) & 1)) dst[par + count - 1] = src0[count - 1];
    }
  };
  issue_tile(vcta, 0);                               // on their way while the tables are copied
  if (stages > 2) issue_tile(vcta + vgrid, 1);
  perwin_tables(a, sA, sH, sC, sV);
  __syncthreads();
  perwin_edges(a, geo, sA, sH);

  const int l16 = tid & 15, hw = gt >> 4;
  const int n_steps = (len + 15) >> 4;                              // steps of 16 lanes; only the last one can be partial
  const bool last_ok = (len & 15) == 0 || l16 < (len & 15);         // this lane's part of it
  const int w_mine = hw * K + ((l16 * K) >> 4);                     // the window whose total this lane holds after reduce16()
  const bool writer = (l16 & (16 / K - 1)) == 0;
  const uint32_t ph_step = a.ss * a.inc;                            // phase advance per window
  const uint32_t ph_mine = (uint32_t)((int)(hw * K * a.ss) + win_off) * a.inc + a.phase0;     // + s0 * ph_step: phase of this half warp's first window
  const int x_mine = hw * K * ss + l16;

  uint32_t stage = 0, phases = 0;
  for (uint32_t t = vcta; t < geo.n_tiles; t += vgrid) {
    // One warp polls the tile's mbarrier (256 spinning threads would take issue slots from the groups that are summing);
    // the group's named barrier then publishes the landed tile to the other warps and, at the same time, tells the
    // first warp that everybody is done with tile t-1, whose buffer the next bulk copies overwrite.
    if (gwarp == 0) mbar_wait(smem_u32(&bars[grp][stage]), (phases >> stage) & 1u);
    phases ^= 1u << stage;
    asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "n"(kPwGroup) : "memory");
    issue_tile(t + (stages - 1) * vgrid, stage == 0 ? stages - 1 : stage - 1);
    const float2 *xs = sX + (size_t)stage * geo.x_tile + par + x_mine;
    const uint32_t s0 = a.d_lo + t * TW;
    const int nw = (int)min((uint32_t)TW, a.d_hi + 1 - s0);
    const uint32_t ph0 = ph_mine + s0 * ph_step;
    float2 acc[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      acc[k] = make_float2(0.f, 0.f);
      if (hw * K + k < nw) {
        const uint32_t phb = ph0 + k * ph_step;
        const float2 *pv = sV + (uint32_t)sC[phb & 255u] * a.v_pitch + l16;
        const float2 *px = xs + k * ss;
        switch (n_steps) {        // CTA-uniform
          case 2: acc[k] = mac_window<2>(pv, px, n_steps, last_ok); break;
          case 3: acc[k] = mac_window<3>(pv, px, n_steps, last_ok); break;
          case 4: acc[k] = mac_window<4>(pv, px, n_steps, last_ok); break;
          case 5: acc[k] = mac_window<5>(pv, px, n_steps, last_ok); break;
          case 6: acc[k] = mac_window<6>(pv, px, n_steps, last_ok); break;
          case 7: acc[k] = mac_window<7>(pv, px, n_steps, last_ok); break;
          case 8: acc[k] = mac_window<8>(pv, px, n_steps, last_ok); break;
          case 9: acc[k] = mac_window<9>(pv, px, n_steps, last_ok); break;
          case 10: acc[k] = mac_window<10>(pv, px, n_steps, last_ok); break;
          case 11: acc[k] = mac_window<11>(pv, px, n_steps, last_ok); break;
          case 12: acc[k] = mac_window<12>(pv, px, n_steps, last_ok); break;
          case 13: acc[k] = mac_window<13>(pv, px, n_steps, last_ok); break;
          case 14: acc[k] = mac_window<14>(pv, px, n_steps, last_ok); break;
          case 15: acc[k] = mac_window<15>(pv, px, n_steps, last_ok); break;
          case 16: acc[k] = mac_window<16>(pv, px, n_steps, last_ok); break;
          default: acc[k] = mac_window<0>(pv, px, n_steps, last_ok); break;
        }
      }
    }
    const float2 tot = reduce16<K>(acc, l16);
    if (writer && w_mine < nw) {
      const uint32_t phb = ph0 + (uint32_t)((l16 * K) >> 4) * ph_step;
      ((float2 *)a.acc_cur)[s0 + w_mine] = cmul(sA[(phb & 0x7fffu) >> 8], tot);
    }
    stage = stage + 1 == stages ? 0 : stage + 1;
  }
}

constexpr uint32_t kPw1MaxSs = 22;        // ss <= this: a thread per window; above: a half warp per window

constexpr size_t kPwMaxSmem = 220 * 1024;

int k_max_of(uint32_t ss) {      // windows per half warp: a group's tile (16 K windows) stays within 2048 samples where it can
  int k = 4;
  while (k > 1 && 16u * k * ss > 2048u) k >>= 1;
  return k;
}

// float2 elements of one tile buffer (even, so that every buffer starts 16-byte aligned); k = 0: thread-per-window layout
size_t tile_elems(const IqbbFoldArgs &a, int k, uint32_t *delta_out) {
  const size_t L1 = a.taps_len - 1;
  uint32_t delta = 0;
  size_t t;
  if (k == 0) {
    delta = (a.ss & 1u) ? 0u : 1u;                               // odd pitch
    t = L1 + delta + 256u * (size_t)(a.ss + delta);
  } else {
    t = L1 + 16u * (size_t)k * a.ss + 2;                         // + alignment slack of the bulk copies
  }
  if (delta_out) *delta_out = delta;
  return (t + 1) & ~(size_t)1;
}

// Half-warp kernels: what matters most is how many 256-thread groups are resident (measured on B200, ss 32..128:
// 4 groups x 2 buffers beat 2 groups x 3 buffers by 1.3-1.7x), then the tile size.  Two buffers per group; the largest
// K <= k_max that still lets four groups fit next to the table, else the K with the most groups.
void shape16(const IqbbFoldArgs &a, size_t table, int *k_out, int *groups_out) {
  int best_k = 1, best_g = 0;
  for (int k = k_max_of(a.ss); k >= 1; k >>= 1) {
    int g = 4;
    while (g > 1 && (table + (size_t)g * 2 * tile_elems(a, k, nullptr)) * sizeof(float2) > kPwMaxSmem) g >>= 1;
    if (g > best_g) { best_g = g; best_k = k; }
    if (g == 4) break;
  }
  *k_out = best_k; *groups_out = best_g > 0 ? best_g : 1;
}

}  // namespace

// Fills in d_lo / d_hi; true when the call has whole windows and the table + two tile buffers fit into shared memory.
bool fold_perwin_eligible(IqbbFoldArgs &a) {
  if (!a.tab_v || !a.tab_cls || a.v_rows == 0 || a.ss < 2 || a.ss > 256 || a.taps_len > a.ss + 1) return false;
  const int64_t ss = a.ss, L1 = (int64_t)a.taps_len - 1, win_off = (int64_t)a.first - (int64_t)a.r0;
  int64_t lo = 1;
  while (lo * ss + win_off - L1 < 0) ++lo;
  const int64_t hi = ((int64_t)a.n - win_off) / ss - 1;        // (hi + 1) ss + win_off <= n
  if (hi < lo) return false;
  a.d_lo = (uint32_t)lo; a.d_hi = (uint32_t)hi;
  if (((size_t)a.v_rows * a.v_pitch + 1 + 2 * tile_elems(a, a.ss <= kPw1MaxSs ? 0 : 1, nullptr)) * sizeof(float2) > kPwMaxSmem) return false;
  if (a.ss > kPw1MaxSs && a.taps_len <= 129) {
    // a table that leaves room for fewer than four thread groups: the window-pipelined kernel is faster (measured, 2 groups:
    // ss 96 / 97 taps 2.7 vs 3.5 TB/s, 100 / 101 2.8 vs 3.3, 128 / 20 4.2 vs 4.3; 4 groups: 96 / 64 5.2 vs 3.5)
    int k = 1, groups = 1;
    shape16(a, ((size_t)a.v_rows * a.v_pitch + 1) & ~(size_t)1, &k, &groups);
    if (groups < 4) return false;
  }
  return true;
}

int launch_fold_perwin(const IqbbFoldArgs &a_in, cudaStream_t st) {
  IqbbFoldArgs a = a_in;
  const uint64_t q_last = (uint64_t)a.r0 + (a.n - 1) - ((a.first && a.n > 1) ? 1 : 0);
  a.part = 8192; a.cpw = 1; a.fast = 0;
  a.n_chunks = (uint32_t)(q_last / a.ss + 1);
  PerwinGeom geo{};
  geo.n_edge = a.d_lo + (a.n_chunks > a.d_hi ? a.n_chunks - a.d_hi : 0u);
  geo.magic = (uint32_t)(((1ull << 32) + a.ss - 1) / a.ss);
  geo.stages = 2;
  const size_t table = ((size_t)a.v_rows * a.v_pitch + 1) & ~(size_t)1;
  if (a.ss <= kPw1MaxSs) {
    // small table, several CTAs per SM with two buffers each (measured: 3 CTAs x 2 buffers beat 2 CTAs x 3)
    geo.x_tile = (uint32_t)tile_elems(a, 0, &geo.delta);
    geo.pitch = a.ss + geo.delta;
    geo.chunk = 16;
    if (geo.delta) while (geo.chunk + (geo.chunk + a.ss - 2) / a.ss > 16u) --geo.chunk;   // samples + window borders crossed <= 16 slots
    geo.n_tiles = (a.d_hi - a.d_lo + 1 + 255u) / 256u;
    return launch_persistent("iqbb_fold_f32_perwin_kernel", iqbb_fold_f32_perwin1_kernel, geo.n_tiles, kPw1Threads,
                             (table + geo.stages * (size_t)geo.x_tile) * sizeof(float2), st, a, geo);
  }
  int k = 1, groups = 1;
  shape16(a, table, &k, &groups);
  geo.x_tile = (uint32_t)tile_elems(a, k, nullptr);
  geo.pitch = a.ss;
  const size_t smem = (table + (size_t)groups * geo.stages * geo.x_tile) * sizeof(float2);
  const uint32_t tw = 16u * (uint32_t)k;
  geo.n_tiles = (a.d_hi - a.d_lo + 1 + tw - 1) / tw;
  const uint64_t want = (geo.n_tiles + groups - 1) / groups;
  return dispatch(k, std::integer_sequence<int, 1, 2, 4>{}, [&](auto K) {
    return launch_persistent("iqbb_fold_f32_perwin_kernel", iqbb_fold_f32_perwin16_kernel<K>, want > 0 ? want : 1, groups * kPwGroup, smem, st, a, geo);
  }, [&] { return set_error(SDRG_ERR_RUNTIME, "IQBaseBand<float>: no per-window kernel for %d windows per half warp", k); });
}

}  // namespace sdrg

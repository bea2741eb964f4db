// iqbb_fold_experimental.cu -- variants of the folded float kernel that are NOT on the default path:
//   * the TMA bulk-copy staging variant (sdrg_iqbb_set_float_path(h, 3)): correct, issue-bound, not faster;
//   * the bandwidth probes behind SDRG_FOLD_PROBE (profiles/r01_final_fold_probe.md): same grid, chunk dealing
//     and staging as the production kernel with the arithmetic stripped -- their output is NOT the IQBaseBand result.
#include "iqbb_fold_common.cuh"

namespace sdrg {
using namespace foldk;
namespace {

// ---- TMA variant ---------------------------------------------------------------------------------
// Same arithmetic, different data movement: every warp owns a contiguous, 2 KB-aligned segment of
// the call and streams it through a private shared-memory ring of kTmaTiles x 2 KB tiles filled by
// 1-D bulk async copies (cp.async.bulk, SASS UBLKCP) that complete on per-tile mbarriers.  Bytes in
// flight no longer cost registers: 3 CTAs x 8 warps x 3 tiles x 2 KB = 144 KB per SM are outstanding
// while the warps compute from shared memory.  No cross-warp synchronisation after the prologue.
constexpr int kTmaTile = 256;                   // samples per tile (2 KB)
constexpr int kTmaTiles = 4;                    // ring depth per warp
constexpr int kTmaRing = kTmaTile * kTmaTiles;  // samples per ring

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

__global__ void __launch_bounds__(kFoldThreads, 3) iqbb_fold_f32_tma_kernel(const IqbbFoldArgs a) {
  extern __shared__ __align__(128) unsigned char dyn_smem[];
  __shared__ float2 sA[128];
  __shared__ float2 sH[256];
  __shared__ __align__(8) unsigned long long bars[kFoldWarps][kTmaTiles];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  for (uint32_t k = blockIdx.x * blockDim.x + tid; k < a.zero_next; k += gridDim.x * blockDim.x)
    ((float2 *)a.acc_next)[k] = make_float2(0.f, 0.f);
  if (tid < 128) sA[tid] = a.tab_a[tid];
  sH[tid] = a.tab_u[(size_t)tid * a.taps_len];
  if (lane == 0) {
#pragma unroll
    for (int t = 0; t < kTmaTiles; ++t) mbar_init(smem_u32(&bars[warp][t]), 1);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  const uint64_t seg_lo64 = ((uint64_t)blockIdx.x * kFoldWarps + warp) * a.seg;
  if (seg_lo64 >= a.n) return;
  const uint32_t S_lo = (uint32_t)seg_lo64;
  const uint32_t S_hi = (uint32_t)min((uint64_t)a.n, seg_lo64 + a.seg);
  const float2 *__restrict__ x = (const float2 *)a.x;
  float2 *ring = (float2 *)dyn_smem + (size_t)warp * kTmaRing;
  const uint32_t ring_u32 = smem_u32(ring), bar_u32 = smem_u32(&bars[warp][0]);
  const uint32_t n_tiles = (S_hi - S_lo + kTmaTile - 1) / kTmaTile;

  // producer side (lane 0): tile t -> ring slot t % kTmaTiles
  auto issue = [&](uint32_t t) {
    const uint32_t start = S_lo + t * kTmaTile;
    const uint32_t cnt = min((uint32_t)kTmaTile, S_hi - start);
    const uint32_t bytes16 = (cnt * 8u) & ~15u;
    const uint32_t slot = t % kTmaTiles;
    mbar_expect_tx(bar_u32 + slot * 8, bytes16);
    if (bytes16) tma_load_1d(ring_u32 + slot * (kTmaTile * 8), x + start, bytes16, bar_u32 + slot * 8);
    if (cnt & 1u) ring[slot * kTmaTile + cnt - 1] = x[start + cnt - 1];     // odd tail of the call
  };
  if (lane == 0) {
    for (uint32_t t = 0; t < min(n_tiles, (uint32_t)kTmaTiles); ++t) issue(t);
  }
  __syncwarp();
  uint32_t landed = 0;      // tiles [0, landed) are known to be in shared memory
  uint32_t issued = min(n_tiles, (uint32_t)kTmaTiles);

  float *acc_out = (float *)a.acc_cur;
  const int L1 = (int)a.taps_len - 1;
  const int64_t win_off = (int64_t)a.first - (int64_t)a.r0;
  const uint32_t inc32 = (32u * a.inc) & 0x7fffu, inc256 = (256u * a.inc) & 0x7fffu;

  float2 base = make_float2(0.f, 0.f);
  uint32_t base_slot = 0;
  uint32_t s = (uint32_t)(((uint64_t)a.r0 + S_lo - ((a.first && S_lo > 0) ? 1u : 0u)) / a.ss);
  for (uint32_t pos = S_lo; pos < S_hi; ++s) {
    const int64_t full_end = (int64_t)((uint64_t)(s + 1) * a.ss) + win_off;
    const uint32_t c_lo = pos;
    const uint32_t c_hi = (uint32_t)min(full_end, (int64_t)S_hi);
    const uint32_t len = c_hi - c_lo;
    const int64_t t_lo64 = full_end - L1 - (int64_t)c_lo;
    const uint32_t t_lo = t_lo64 < 0 ? 0u : (t_lo64 > (int64_t)len ? len : (uint32_t)t_lo64);
    const uint32_t end_rel = (uint32_t)(full_end - (int64_t)c_lo);
    pos = c_hi;

    if (base_slot != s) { flush(acc_out, base_slot, base, lane); base = make_float2(0.f, 0.f); }
    uint32_t ph = (a.phase0 + (c_lo + (uint32_t)lane) * a.inc) & 0x7fffu;
    float2 H[8], R[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) { H[u] = sH[(ph + u * inc32) & 255u]; R[u] = make_float2(0.f, 0.f); }
    float2 sent = make_float2(0.f, 0.f);
    uint32_t pb = 0; float2 Ab = make_float2(0.f, 0.f);
    const float2 *__restrict__ urow = a.tab_u;
    if (t_lo < len) {
      pb = (a.phase0 + (uint32_t)full_end * a.inc) & 0x7fffu;
      Ab = sA[pb >> 8];
      urow = a.tab_u + (size_t)(pb & 255u) * a.taps_len;
    }
    const uint32_t roff = c_lo - S_lo + lane;             // segment-relative index of this lane's sample in step 0

    for (uint32_t k = 0; k < len; k += 256, ph = (ph + inc256) & 0x7fffu) {
      // tiles needed by this batch: up to the one holding its last sample
      const uint32_t last = min(k + 256u, len) - 1u + (c_lo - S_lo);
      const uint32_t need = last / kTmaTile + 1;
      while (landed < need) { mbar_wait(bar_u32 + (landed % kTmaTiles) * 8, (landed / kTmaTiles) & 1u); ++landed; }
      float2 xv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const uint32_t j = k + 32 * u + lane;
        xv[u] = j < len ? ring[(roff + k + 32 * u) & (kTmaRing - 1)] : make_float2(0.f, 0.f);
      }
      if (k + 256 <= t_lo) {
#pragma unroll
        for (int u = 0; u < 8; ++u) cfma(R[u], sA[((ph + u * inc32) & 0x7fffu) >> 8], xv[u]);
      } else {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const uint32_t js = k + 32 * u;
          if (js >= len) break;
          cfma(R[u], sA[((ph + u * inc32) & 0x7fffu) >> 8], xv[u]);
          if (js + 32 > t_lo) {
            const uint32_t j = js + lane;
            if (j >= t_lo && j < len) cfma(sent, cmul(Ab, __ldg(urow + (end_rel - j))), xv[u]);
          }
        }
      }
      // tiles that lie entirely before the next sample to be read are free: refill them
      const uint32_t next_rel = min(k + 256u, len) + (c_lo - S_lo);
      const uint32_t free_upto = next_rel / kTmaTile;       // tiles [0, free_upto) fully consumed
      __syncwarp();
      if (lane == 0) {
        while (issued < n_tiles && issued < free_upto + kTmaTiles) { issue(issued); ++issued; }
      } else {
        const uint32_t cap = min(n_tiles, free_upto + (uint32_t)kTmaTiles);
        if (issued < cap) issued = cap;
      }
      __syncwarp();
    }
    float2 tot = make_float2(base.x - sent.x, base.y - sent.y);
#pragma unroll
    for (int u = 0; u < 8; ++u) cfma(tot, H[u], R[u]);
    flush(acc_out, s, tot, lane);
    base = sent; base_slot = s + 1;
  }
  flush(acc_out, base_slot, base, lane);
}


// ---- bandwidth probes (SDRG_FOLD_PROBE=1..3; results are NOT the IQBaseBand output) ---------------
// Same persistent grid, chunk dealing and staging as iqbb_fold_f32_kernel with the arithmetic reduced
// to one complex add per sample: what the access pattern itself can reach.  MODE 1: batches of 8 steps
// (the production schedule); 2: the whole window (<= 16 steps) in one round trip; 3: the first batch of
// the NEXT chunk is issued before the current chunk's last batch is consumed.
template <int MODE>
__global__ void __launch_bounds__(kFoldThreads, MODE == 1 ? 4 : 3) iqbb_fold_probe_kernel(const IqbbFoldArgs a) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t total_warps = gridDim.x * kFoldWarps;
  const uint32_t wg = warp * gridDim.x + blockIdx.x;
  const float2 *__restrict__ x = (const float2 *)a.x;
  float *acc_out = (float *)a.acc_cur;
  WarpStage stage{(float2 *)dyn_smem + (size_t)warp * kStageRows * kStagePitch, 0u, 0u};
  const int L1 = (int)a.taps_len - 1;
  const int win_off = (int)a.first - (int)a.r0;
  if (MODE == 1) {
    for (uint32_t id = wg; id < a.n_chunks; id += total_warps) {
      Chunk c;
      if (!chunk_of(a, id, win_off, L1, c)) continue;
      const float2 *__restrict__ xc = x + c.c_lo + lane;
      float2 R[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) R[u] = make_float2(0.f, 0.f);
      int k = 0;
      for (; k + 256 <= c.len; k += 256) {
        float2 xv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) xv[u] = ld_stream(xc + k + 32 * u);
#pragma unroll
        for (int u = 0; u < 8; ++u) { R[u].x += xv[u].x; R[u].y += xv[u].y; }
      }
      if (k < c.len) {
        const int rem = c.len - k;
        float2 xv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) { xv[u] = make_float2(0.f, 0.f); if (32 * u + lane < rem) xv[u] = ld_stream(xc + k + 32 * u); }
#pragma unroll
        for (int u = 0; u < 8; ++u) { R[u].x += xv[u].x; R[u].y += xv[u].y; }
      }
      float2 tot = make_float2(0.f, 0.f);
#pragma unroll
      for (int u = 0; u < 8; ++u) { tot.x += R[u].x; tot.y += R[u].y; }
      stage.push(tot, c.s, lane, acc_out);
    }
  } else if (MODE == 2) {
    for (uint32_t id = wg; id < a.n_chunks; id += total_warps) {
      Chunk c;
      if (!chunk_of(a, id, win_off, L1, c)) continue;
      const float2 *__restrict__ xc = x + c.c_lo + lane;
      float2 tot = make_float2(0.f, 0.f);
      for (int k = 0; k < c.len; k += 512) {
        const int rem = c.len - k;
        float2 xv[16];
#pragma unroll
        for (int u = 0; u < 16; ++u) { xv[u] = make_float2(0.f, 0.f); if (32 * u + lane < rem) xv[u] = ld_stream(xc + k + 32 * u); }
#pragma unroll
        for (int u = 0; u < 16; ++u) { tot.x += xv[u].x; tot.y += xv[u].y; }
      }
      stage.push(tot, c.s, lane, acc_out);
    }
  } else {
    uint32_t id = wg;
    Chunk c; bool have = false;
    for (; id < a.n_chunks; id += total_warps) if (chunk_of(a, id, win_off, L1, c)) { have = true; break; }
    float2 xa[8];
    if (have) {
#pragma unroll
      for (int u = 0; u < 8; ++u) { xa[u] = make_float2(0.f, 0.f); if (32 * u + lane < c.len) xa[u] = ld_stream(x + c.c_lo + lane + 32 * u); }
    }
    while (have) {
      const float2 *__restrict__ xc = x + c.c_lo + lane;
      float2 xb[8];
      const int rem = c.len - 256;                         // second batch of this chunk (issued first)
#pragma unroll
      for (int u = 0; u < 8; ++u) { xb[u] = make_float2(0.f, 0.f); if (32 * u + lane < rem) xb[u] = ld_stream(xc + 256 + 32 * u); }
      float2 tot = make_float2(0.f, 0.f);
#pragma unroll
      for (int u = 0; u < 8; ++u) { tot.x += xa[u].x; tot.y += xa[u].y; }
      Chunk cn; bool haven = false;
      for (id += total_warps; id < a.n_chunks; id += total_warps) if (chunk_of(a, id, win_off, L1, cn)) { haven = true; break; }
      if (haven) {
#pragma unroll
        for (int u = 0; u < 8; ++u) { xa[u] = make_float2(0.f, 0.f); if (32 * u + lane < cn.len) xa[u] = ld_stream(x + cn.c_lo + lane + 32 * u); }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) { tot.x += xb[u].x; tot.y += xb[u].y; }
      for (int k = 512; k < c.len; k += 256) {             // longer pieces: plain batches
        const int r2 = c.len - k;
#pragma unroll
        for (int u = 0; u < 8; ++u) { xb[u] = make_float2(0.f, 0.f); if (32 * u + lane < r2) xb[u] = ld_stream(xc + k + 32 * u); }
#pragma unroll
        for (int u = 0; u < 8; ++u) { tot.x += xb[u].x; tot.y += xb[u].y; }
      }
      stage.push(tot, c.s, lane, acc_out);
      c = cn; have = haven;
    }
  }
  stage.drain(lane, acc_out);
}

template <int MODE>
int launch_fold_probe_t(IqbbFoldArgs a, cudaStream_t st) {
  const size_t smem = (size_t)kFoldWarps * kStageRows * kStagePitch * sizeof(float2);
  int resident = 0;
  const int rc = kernel_setup((const void *)iqbb_fold_probe_kernel<MODE>, kFoldThreads, smem, &resident);
  if (rc) return rc;
  static const int cap = [] { const char *e = getenv("SDRG_FOLD_PROBE_CTAS"); return e ? atoi(e) : 0; }();   // CTAs per SM
  if (cap > 0) {
    int dev = 0, sms = 0;
    SDRG_CUDA(cudaGetDevice(&dev));
    SDRG_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    resident = std::min(resident, sms * cap);
  }
  const uint64_t want = ((uint64_t)a.n_chunks + kFoldWarps - 1) / kFoldWarps;
  return launch("iqbb_fold_probe_kernel", iqbb_fold_probe_kernel<MODE>, (unsigned)std::min<uint64_t>(want, resident), kFoldThreads, smem, st, a);
}

}  // namespace

int launch_fold_tma(IqbbFoldArgs a, cudaStream_t st) {
  // one contiguous 2 KB-aligned segment per warp; ~2 waves of 148 x 3 CTAs
  const uint64_t target_warps = 148ull * 3 * kFoldWarps * 2;
  uint64_t seg = (a.n + target_warps - 1) / target_warps;
  seg = ((seg + kTmaTile - 1) / kTmaTile) * kTmaTile;
  if (seg < (uint64_t)kTmaTile) seg = kTmaTile;
  a.seg = (uint32_t)seg;
  const uint64_t per_block = seg * kFoldWarps;
  return launch("iqbb_fold_f32_tma_kernel", iqbb_fold_f32_tma_kernel, (unsigned)((a.n + per_block - 1) / per_block), kFoldThreads,
                (size_t)kFoldWarps * kTmaRing * sizeof(float2), st, a);
}


int launch_fold_probe(int mode, IqbbFoldArgs a, cudaStream_t st) {
  switch (mode) {
    case 1: return launch_fold_probe_t<1>(a, st);
    case 2: return launch_fold_probe_t<2>(a, st);
    default: return launch_fold_probe_t<3>(a, st);
  }
}

}  // namespace sdrg

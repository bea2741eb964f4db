// api.cu -- the C ABI of libsdrg (include/sdrg.h): handles, stream state, buffer residency.
//
// Host-side bookkeeping only; all sample arithmetic happens in the kernels.  The carried stream
// state of IQBaseBand (src/baseband.hh:278-296: _ring, _ring_offset, _sample_count, _last; and
// src/freqshift.hh:97-99: _lut_count) becomes
//   device: the last L-1 input samples (double buffered), the open window's partial sum
//           (slot 0 of the double-buffered accumulator array)
//   host  : consumed = samples since config() (fixes the window grid), phase0 = NCO phase
// all of which advance in closed form with the number of samples consumed.
#include "iqbb_kernels.cuh"

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cmath>
#include <cstring>
#include <map>
#include <mutex>
#include <vector>

namespace sdrg {

static thread_local char g_err[512] = "";
static thread_local int g_device = 0;
static std::atomic<uint64_t> g_launches{0};

int set_error(int code, const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
void count_launch(unsigned n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- optional per-kernel timing (CUDA events on the launching stream) -----------------------------
struct ProfSpan { cudaEvent_t a, b; int kind; };
static std::mutex g_prof_mu;
static bool g_prof_on = false;
static std::vector<ProfSpan> g_prof_spans;
static std::vector<cudaEvent_t> g_prof_pool;

static cudaEvent_t prof_event() {
  if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}
struct ProfScope {   // records [begin, end) around one kernel launch when profiling is on
  cudaStream_t st; int idx = -1;
  ProfScope(int kind, cudaStream_t s) : st(s) {
    if (!g_prof_on) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    ProfSpan sp{prof_event(), prof_event(), kind};
    cudaEventRecord(sp.a, st);
    g_prof_spans.push_back(sp);
    idx = (int)g_prof_spans.size() - 1;
  }
  ~ProfScope() {
    if (idx < 0) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    cudaEventRecord(g_prof_spans[idx].b, st);
  }
};

// ---- managed buffers ---------------------------------------------------------------------------
struct ManagedBuffer {
  char  *host = nullptr;
  char  *dev = nullptr;
  size_t bytes = 0;
  int    device = 0;
  size_t valid_lo = 0, valid_hi = 0;   // device-valid byte range (what a GPU node produced last)
  bool   host_synced = true;           // that range has been copied back already
  cudaEvent_t ready = nullptr;         // recorded after the producing kernels
  cudaEvent_t uploaded = nullptr;      // recorded after the last asynchronous host -> device copy out of `host`
  bool   upload_pending = false;       // ... which the producer must not overtake by refilling `host`
};
static std::mutex g_buf_mu;
static std::map<uintptr_t, ManagedBuffer> g_bufs;   // keyed by host base address

static ManagedBuffer *find_buffer(const void *p) {   // caller holds g_buf_mu
  if (g_bufs.empty()) return nullptr;
  auto it = g_bufs.upper_bound((uintptr_t)p);
  if (it == g_bufs.begin()) return nullptr;
  --it;
  ManagedBuffer &b = it->second;
  if ((uintptr_t)p < (uintptr_t)b.host + (b.bytes ? b.bytes : 1)) return &b;
  return nullptr;
}

}  // namespace sdrg

using namespace sdrg;

// ---- IQBaseBand handle -------------------------------------------------------------------------
struct sdrg_iqbb {
  IqbbDesign d;
  int device = 0;
  bool configured = false;
  double nco_Fs = 0;
  // device tables / state
  void *d_taps = nullptr, *d_lut = nullptr;
  void *d_hist[2] = {nullptr, nullptr};
  void *d_acc[2] = {nullptr, nullptr};
  size_t acc_cap = 0;
  uint32_t acc_dirty[2] = {0, 0};
  uint32_t taps_len = 1, hist_len = 0;
  std::vector<int32_t> host_taps;      // int paths: the Gauss-form taps as uploaded
  // folded float path (iqbb_fold_kernels.cu)
  int in_fmt = 0;                      // int16 only: 0 native, 2 complex uint8, 3 complex int8 (fused AutoCast), 4 real int16
  bool real_input = false;             // BaseBand<int16_t> (src/baseband.hh:304-529): real stream, plain windows, 2^16 FIR gain
  double r_Ff = 0, r_width = 0, r_Fs = 0;   // its double members _Ff, _width and FreqShiftBase::_Fs
  int float_path = 0;                  // 0 auto, 1 direct, 2 folded
  bool fold = false;
  void *d_tab_a = nullptr, *d_tab_u = nullptr;
  void *d_tab_v = nullptr, *d_tab_cls = nullptr;   // per-window kernel (iqbb_fold_perwin.cu): V(class, j) and phase byte -> class
  uint32_t v_rows = 0, v_pitch = 0;
  int last_float_kernel = 0;           // sdrg_iqbb_last_float_kernel
  uint32_t *d_work = nullptr;          // work counter of the window-pipelined kernel (0 between calls)
  // stream position
  uint32_t phase0 = 0;
  int parity = 0;
  uint64_t consumed = 0, produced = 0;
  // staging for the host-pointer entry points
  cudaStream_t stream = nullptr;
  void *d_in = nullptr, *d_out = nullptr;
  size_t in_cap = 0, out_cap = 0;
};

struct sdrg_fmdemod {
  int scalar = SDRG_T_S16, device = 0;
  void *d_alias = nullptr; size_t alias_cap = 0;   // result staging for aliased (in-place) device calls
  void *d_last[2] = {nullptr, nullptr};
  int parity = 0;
  cudaStream_t stream = nullptr;
  void *d_in = nullptr, *d_out = nullptr;
  size_t in_cap = 0, out_cap = 0;
};

struct sdrg_rxchain {
  sdrg_iqbb *bb = nullptr;
  int demod = SDRG_DEMOD_NONE;
  void *d_last[2] = {nullptr, nullptr};
  int parity = 0;
  void *d_in = nullptr, *d_bb = nullptr, *d_audio = nullptr;
  size_t in_cap = 0, bb_cap = 0, audio_cap = 0;
  // host-pointer entry point: the upload is cut into chunks on two copy streams so that the kernels of
  // chunk i run while chunk i+1 is still on the wire
  cudaStream_t copy_st[2] = {nullptr, nullptr};
  std::vector<cudaEvent_t> copy_ev;
};

namespace {

size_t sample_bytes(int scalar) { return 2 * scalar_bytes(scalar); }
size_t in_sample_bytes(const sdrg_iqbb *h);   // bytes per INPUT sample (2 when AutoCast is fused into the load)
size_t acc_bytes() { return 8; }   // int2 / float2

size_t audio_bytes(int scalar, int demod) {
  if (demod == SDRG_DEMOD_FM) return scalar == SDRG_T_F32 ? 4 : 2;
  return scalar_bytes(scalar);
}

size_t in_sample_bytes(const sdrg_iqbb *h) { return h->in_fmt == 5 ? 1 : (h->in_fmt ? 2 : sample_bytes(h->d.scalar)); }
int input_type_of(const sdrg_iqbb *h) {
  if (h->real_input) return h->d.scalar;
  return h->in_fmt == 2 ? SDRG_T_CU8 : (h->in_fmt == 3 ? SDRG_T_CS8 : complex_type_of(h->d.scalar));
}
const char *node_name(const sdrg_iqbb *h) { return h->real_input ? "BaseBand" : "IQBaseBand"; }
void design_filter(sdrg_iqbb *h) {
  if (h->real_input) design_kernel_real(h->d, h->r_Ff, h->r_width, h->r_Fs);
  else design_kernel(h->d);
}

int grow(void **p, size_t *cap, size_t need) {
  if (*cap >= need && *p) return SDRG_OK;
  if (*p) SDRG_CUDA(cudaFree(*p));
  *p = nullptr; *cap = 0;
  size_t want = need < 4096 ? 4096 : need;
  SDRG_CUDA(cudaMalloc(p, want));
  *cap = want;
  return SDRG_OK;
}

void free_dev(void **p) { if (*p) { cudaFree(*p); *p = nullptr; } }

typedef WindowAdvance Advance;
Advance advance(const sdrg_iqbb *h, uint64_t n) {
  return h->real_input ? window_advance_plain(h->consumed, h->d.sub_sample, n) : window_advance(h->consumed, h->d.sub_sample, n);
}

// Folded float path: A(a) and U(r,e) in double on the host (see iqbb_fold_kernels.cu).
int upload_fold_tables(sdrg_iqbb *h) {
  const IqbbDesign &d = h->d;
  free_dev(&h->d_tab_a); free_dev(&h->d_tab_u); free_dev(&h->d_tab_v); free_dev(&h->d_tab_cls);
  h->v_rows = h->v_pitch = 0;
  if (!h->d_work) SDRG_CUDA(cudaMalloc((void **)&h->d_work, sizeof(uint32_t)));
  SDRG_CUDA(cudaMemset(h->d_work, 0, sizeof(uint32_t)));
  const size_t L = d.order, ss = d.sub_sample;
  const bool eligible = d.scalar == SDRG_T_F32 && ss >= 2 && ss + 1 >= L;
  if (h->float_path >= 2 && !eligible && d.scalar == SDRG_T_F32)
    return set_error(SDRG_ERR_CONFIG, "IQBaseBand<float>: folded path needs sub_sample >= max(2, order-1) (ss=%zu, order=%zu)", ss, L);
  h->fold = eligible && h->float_path != 1;
  if (!h->fold) return SDRG_OK;
  const bool nco = d.lut_inc != 0, neg = d.negative;
  const uint64_t inc = d.lut_inc & 0x7fffu;
  std::vector<float> A(2 * 128), U(2 * 256 * L);
  fold_table_a(d, nco, neg, A.data());
  fold_table_u(d, L, U.data());
  SDRG_CUDA(cudaMalloc(&h->d_tab_a, A.size() * sizeof(float)));
  SDRG_CUDA(cudaMemcpy(h->d_tab_a, A.data(), A.size() * sizeof(float), cudaMemcpyHostToDevice));
  SDRG_CUDA(cudaMalloc(&h->d_tab_u, U.size() * sizeof(float)));
  SDRG_CUDA(cudaMemcpy(h->d_tab_u, U.data(), U.size() * sizeof(float), cudaMemcpyHostToDevice));
  // Window-direct kernel (short windows): V(r, j) = sum_{d = max(0, j-L+1)}^{min(j, ss-1)} B(r, d) k[j-d], j < ss+L-1.
  // B(r, d) depends on r only through the carry [r + (d inc & 255) >= 256], which is monotone in r: equal carry
  // patterns give equal rows, so rows are stored once per pattern (<= ss + 1 of them) and cls[r] names the row.
  if (ss <= 256) {
    const size_t len = ss + L - 1, pitch = len | 1;
    std::vector<uint16_t> cls(256);
    std::vector<float> V;
    std::vector<uint64_t> sig(ss), prev(ss);
    std::vector<double> dr(ss), di(ss);
    size_t rows = 0;
    for (size_t r = 0; r < 256; ++r) {
      for (size_t dd = 0; dd < ss; ++dd) sig[dd] = nco ? ((r + dd * inc) >> 8) : 0;
      if (r == 0 || sig != prev) {
        if ((rows + 1) * pitch * 8 > 160 * 1024) { rows = 0; break; }      // would not fit next to a tile: no direct kernel
        for (size_t dd = 0; dd < ss; ++dd) {
          if (!nco) { dr[dd] = 1.0; di[dd] = 0.0; continue; }
          const size_t idx = neg ? (size_t)((127 + 128 - (sig[dd] % 128)) % 128) : (size_t)(sig[dd] % 128);
          dr[dd] = d.lutd_re[idx]; di[dd] = d.lutd_im[idx];
        }
        V.resize(2 * (rows + 1) * pitch, 0.0f);
        for (size_t j = 0; j < len; ++j) {
          double sr = 0, si = 0;
          const size_t d_lo = j + 1 > L ? j + 1 - L : 0, d_hi = j < ss - 1 ? j : ss - 1;
          for (size_t dd = d_lo; dd <= d_hi; ++dd) {
            const double kr = d.kd_re[j - dd], ki = d.kd_im[j - dd];
            sr += dr[dd] * kr - di[dd] * ki;
            si += dr[dd] * ki + di[dd] * kr;
          }
          V[2 * (rows * pitch + j)] = (float)sr; V[2 * (rows * pitch + j) + 1] = (float)si;
        }
        ++rows;
        prev = sig;
      }
      cls[r] = (uint16_t)(rows - 1);
    }
    if (rows) {
      SDRG_CUDA(cudaMalloc(&h->d_tab_v, V.size() * sizeof(float)));
      SDRG_CUDA(cudaMemcpy(h->d_tab_v, V.data(), V.size() * sizeof(float), cudaMemcpyHostToDevice));
      SDRG_CUDA(cudaMalloc(&h->d_tab_cls, cls.size() * sizeof(uint16_t)));
      SDRG_CUDA(cudaMemcpy(h->d_tab_cls, cls.data(), cls.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
      h->v_rows = (uint32_t)rows; h->v_pitch = (uint32_t)pitch;
    }
  }
  return SDRG_OK;
}

int upload_design(sdrg_iqbb *h) {
  const IqbbDesign &d = h->d;
  const size_t L = d.order;
  SDRG_CUDA(cudaSetDevice(h->device));
  free_dev(&h->d_taps); free_dev(&h->d_lut);
  free_dev(&h->d_hist[0]); free_dev(&h->d_hist[1]);
  if (d.scalar == SDRG_T_F32) {
    std::vector<float> taps(2 * L), lut(256);
    for (size_t i = 0; i < L; ++i) { taps[2 * i] = (float)d.kd_re[i]; taps[2 * i + 1] = (float)d.kd_im[i]; }
    for (size_t j = 0; j < 128; ++j) { lut[2 * j] = (float)d.lutd_re[j]; lut[2 * j + 1] = (float)d.lutd_im[j]; }
    h->taps_len = (uint32_t)L;
    SDRG_CUDA(cudaMalloc(&h->d_taps, taps.size() * sizeof(float)));
    SDRG_CUDA(cudaMemcpy(h->d_taps, taps.data(), taps.size() * sizeof(float), cudaMemcpyHostToDevice));
    SDRG_CUDA(cudaMalloc(&h->d_lut, lut.size() * sizeof(float)));
    SDRG_CUDA(cudaMemcpy(h->d_lut, lut.data(), lut.size() * sizeof(float), cudaMemcpyHostToDevice));
  } else {
    // leading zero taps multiply x[n-(L-1)+t] by 0: dropping them is exact and shortens the halo
    size_t lead = 0;
    while (lead + 1 < L && d.k_re[lead] == 0 && d.k_im[lead] == 0) ++lead;
    const size_t Lp = L - lead;
    std::vector<int32_t> taps(4 * Lp), lut(256);
    h->host_taps.assign(4 * Lp, 0);
    for (size_t i = 0; i < Lp; ++i) {
      const uint32_t kr = (uint32_t)d.k_re[lead + i], ki = (uint32_t)d.k_im[lead + i];
      taps[4 * i] = (int32_t)kr; taps[4 * i + 1] = (int32_t)(ki - kr); taps[4 * i + 2] = (int32_t)(kr + ki);
      taps[4 * i + 3] = 0;
    }
    h->host_taps = taps;
    for (size_t j = 0; j < 128; ++j) { lut[2 * j] = d.lut_re[j]; lut[2 * j + 1] = d.lut_im[j]; }
    h->taps_len = (uint32_t)Lp;
    SDRG_CUDA(cudaMalloc(&h->d_taps, taps.size() * sizeof(int32_t)));
    SDRG_CUDA(cudaMemcpy(h->d_taps, taps.data(), taps.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    SDRG_CUDA(cudaMalloc(&h->d_lut, lut.size() * sizeof(int32_t)));
    SDRG_CUDA(cudaMemcpy(h->d_lut, lut.data(), lut.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  }
  int rc_fold = upload_fold_tables(h);
  if (rc_fold) return rc_fold;
  h->hist_len = h->taps_len - 1;
  const size_t hb = (h->hist_len ? h->hist_len : 1) * sample_bytes(d.scalar);   // >= the fused-AutoCast element size
  for (int k = 0; k < 2; ++k) {
    SDRG_CUDA(cudaMalloc(&h->d_hist[k], hb));
    // ring zeroed in the ctor (baseband.hh:42-43); a zero sample in cu8 form is the byte 127
    SDRG_CUDA(cudaMemset(h->d_hist[k], h->in_fmt == 2 ? 127 : 0, hb));
  }
  return SDRG_OK;
}

int ensure_acc(sdrg_iqbb *h, size_t slots) {
  if (h->acc_cap >= slots) return SDRG_OK;
  const size_t cap = slots + slots / 2 + 64;
  void *n0 = nullptr, *n1 = nullptr;
  SDRG_CUDA(cudaMalloc(&n0, cap * acc_bytes()));
  SDRG_CUDA(cudaMalloc(&n1, cap * acc_bytes()));
  SDRG_CUDA(cudaMemset(n0, 0, cap * acc_bytes()));
  SDRG_CUDA(cudaMemset(n1, 0, cap * acc_bytes()));
  if (h->d_acc[0]) {   // keep the open window (slot 0 of the current parity)
    SDRG_CUDA(cudaDeviceSynchronize());
    SDRG_CUDA(cudaMemcpy(h->parity == 0 ? n0 : n1, h->d_acc[h->parity], 2 * acc_bytes(), cudaMemcpyDeviceToDevice));
    cudaFree(h->d_acc[0]); cudaFree(h->d_acc[1]);
  }
  h->d_acc[0] = n0; h->d_acc[1] = n1;
  h->acc_dirty[0] = h->acc_dirty[1] = 0;
  h->acc_cap = cap;
  return SDRG_OK;
}

void reset_stream_state(sdrg_iqbb *h) {
  h->phase0 = 0; h->consumed = 0; h->produced = 0;
}

// config()-time recomputation (baseband.hh:156-194): host part
int design_only(sdrg_iqbb *h) {
  IqbbDesign &d = h->d;
  if (d.oFs > 0 && !h->real_input) {
    d.sub_sample = size_t(d.Fs / d.oFs);
    if (d.sub_sample < 1) d.sub_sample = 1;
  }
  if (d.sub_sample < 1) d.sub_sample = 1;    // the reference would divide by zero
  if (d.sub_sample > (1u << 30)) return set_error(SDRG_ERR_CONFIG, "%s: sub-sampling %zu too large", node_name(h), d.sub_sample);
  if (h->real_input && d.scalar == SDRG_T_S8 && (short)((int)(short)d.sub_sample * (int)(short)d.sub_sample) == 0)
    return set_error(SDRG_ERR_CONFIG, "BaseBand<int8_t>: sub-sampling %zu makes int16(ss*ss) zero -- the reference divides by zero "
                     "(complex<int16_t>::operator/=, src/baseband.hh:434)", d.sub_sample);
  design_filter(h);
  h->nco_Fs = h->real_input ? h->r_Fs : double(d.Fs);       // BaseBand keeps the double rate (baseband.hh:371)
  design_lut_increment(d, h->nco_Fs);
  d.out_bs = d.source_bs / d.sub_sample;
  if (d.source_bs % d.sub_sample) d.out_bs += 1;
  d.out_rate = h->real_input ? h->r_Fs / double(d.sub_sample) : double(size_t(d.Fs) / d.sub_sample);
  return SDRG_OK;
}

// ... and the device part: upload tables, reset the stream state
int reconfigure(sdrg_iqbb *h) {
  int rc = design_only(h);
  if (rc) return rc;
  IqbbDesign &d = h->d;
  rc = upload_design(h);
  if (rc) return rc;
  rc = ensure_acc(h, d.out_bs + 3);
  if (rc) return rc;
  SDRG_CUDA(cudaMemset(h->d_acc[0], 0, h->acc_cap * acc_bytes()));
  SDRG_CUDA(cudaMemset(h->d_acc[1], 0, h->acc_cap * acc_bytes()));
  h->acc_dirty[0] = h->acc_dirty[1] = 0;
  h->parity = 0;
  reset_stream_state(h);
  h->configured = true;
  return SDRG_OK;
}

// one launch pair; n <= 2^30
int run_call(sdrg_iqbb *h, const void *d_in, uint32_t n, void *d_bb, void *d_audio, int demod,
             uint64_t seg, int in_place, void *fm_last_in, void *fm_last_out, cudaStream_t st,
             uint64_t *n_out) {
  const Advance adv = advance(h, n);
  *n_out = adv.n_out;
  int rc = ensure_acc(h, adv.n_out + 3);
  if (rc) return rc;
  const int p = h->parity, q = p ^ 1;
  IqbbAccumArgs a{};
  a.x = d_in; a.hist_in = h->d_hist[p]; a.hist_out = h->d_hist[q];
  a.taps = h->d_taps; a.lut = h->d_lut;
  a.host_taps = (h->d.scalar != SDRG_T_F32 && !h->host_taps.empty()) ? h->host_taps.data() : nullptr;
  a.acc_cur = h->d_acc[p]; a.acc_next = h->d_acc[q];
  a.n = n; a.taps_len = h->taps_len; a.hist_len = h->hist_len;
  a.ss = (uint32_t)h->d.sub_sample; a.r0 = adv.r0; a.first = adv.first;
  a.phase0 = h->phase0; a.inc = (uint32_t)(h->d.lut_inc & 0x7fffu); a.nco = h->d.lut_inc != 0 ? 1u : 0u;
  a.neg = h->d.negative ? 1u : 0u;
  a.zero_next = h->acc_dirty[q];
  a.in_fmt = (uint32_t)h->in_fmt;
  a.fir_shift = h->real_input ? (h->d.scalar == SDRG_T_S8 ? 8u : 16u) : 14u;     // BaseBand: >> Traits<Scalar>::shift
  IqbbFinalizeArgs f{};
  f.acc_cur = h->d_acc[p]; f.acc_next = h->d_acc[q];
  f.bb_out = d_bb; f.audio_out = d_audio;
  f.fm_last_in = fm_last_in; f.fm_last_out = fm_last_out;
  f.n_out = (uint32_t)adv.n_out; f.ss = a.ss; f.demod = (uint32_t)demod; f.e0 = adv.e0;
  f.seg = seg; f.in_place = (uint32_t)in_place;
  f.narrow16 = (h->real_input && h->d.scalar == SDRG_T_S8) ? 1u : 0u;
  if (h->fold) {
    IqbbFoldArgs fa{};
    fa.x = d_in; fa.acc_cur = a.acc_cur; fa.acc_next = a.acc_next;
    fa.tab_a = (const float2 *)h->d_tab_a; fa.tab_u = (const float2 *)h->d_tab_u;
    fa.tab_v = (const float2 *)h->d_tab_v; fa.tab_cls = (const uint16_t *)h->d_tab_cls;
    fa.v_rows = h->v_rows; fa.v_pitch = h->v_pitch;
    fa.n = n; fa.taps_len = (uint32_t)h->d.order; fa.ss = a.ss; fa.r0 = a.r0; fa.first = a.first;
    fa.phase0 = a.nco ? a.phase0 : 0u; fa.inc = a.nco ? a.inc : 0u;
    fa.zero_next = a.zero_next;
    fa.work = h->d_work; f.work_reset = h->d_work;
    ProfScope ps(SDRG_KERNEL_IQBB_ACCUM, st);
    rc = launch_iqbb_fold(fa, st, &h->last_float_kernel);
  } else {
    ProfScope ps(SDRG_KERNEL_IQBB_ACCUM, st);
    if (h->d.scalar == SDRG_T_F32) h->last_float_kernel = 1;
    rc = launch_iqbb_accum(h->d.scalar, a, st);
  }
  if (rc) return rc;
  {
    ProfScope ps(SDRG_KERNEL_IQBB_FINALIZE, st);
    rc = launch_iqbb_finalize(h->d.scalar, f, st);
  }
  if (rc) return rc;
  h->acc_dirty[p] = (uint32_t)adv.n_out + 2;   // slots this call touched
  h->acc_dirty[q] = 2;                         // the carry
  h->parity = q;
  h->phase0 = (uint32_t)((h->phase0 + (uint64_t)n * (h->d.lut_inc & 0x7fffu)) & 0x7fffu);
  h->consumed += n; h->produced += adv.n_out;
  return SDRG_OK;
}

int check_handle(const sdrg_iqbb *h) {
  if (!h) return set_error(SDRG_ERR_ARG, "IQBaseBand: null handle");
  if (!h->configured) return set_error(SDRG_ERR_RUNTIME, "IQBaseBand: process() before config()");
  return SDRG_OK;
}

int config_common(const char *who, int expect_type, const sdrg_config *src, bool need_rate, bool *skip) {
  *skip = false;
  if (!src) return set_error(SDRG_ERR_ARG, "%s: null config", who);
  if (src->type == SDRG_T_UNDEFINED || src->buffer_size == 0 || (need_rate && src->sample_rate == 0)) {
    *skip = true;
    return SDRG_OK;
  }
  if (src->type != expect_type)
    return set_error(SDRG_ERR_CONFIG, "Can not configure %s: Invalid type %s (%d), expected %s (%d)", who,
                     type_name(src->type), src->type, type_name(expect_type), expect_type);
  return SDRG_OK;
}

}  // namespace

extern "C" {

int sdrg_abi_version(void) { return SDRG_ABI_VERSION; }
int sdrg_build_has_experiments(void) { return 0; }
const char *sdrg_last_error(void) { return g_err; }

int sdrg_device_count(int *count) {
  if (!count) return set_error(SDRG_ERR_ARG, "null argument");
  SDRG_CUDA(cudaGetDeviceCount(count));
  return SDRG_OK;
}
int sdrg_set_device(int device) {
  SDRG_CUDA(cudaSetDevice(device));
  g_device = device;
  return SDRG_OK;
}
int sdrg_get_device(int *device) {
  if (!device) return set_error(SDRG_ERR_ARG, "null argument");
  *device = g_device;
  return SDRG_OK;
}
int sdrg_device_synchronize(void) { SDRG_CUDA(cudaDeviceSynchronize()); return SDRG_OK; }
int sdrg_kernel_launch_count(uint64_t *count) {
  if (!count) return set_error(SDRG_ERR_ARG, "null argument");
  *count = g_launches.load();
  return SDRG_OK;
}

int sdrg_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_on = on != 0;
  return SDRG_OK;
}
int sdrg_profile_read(int kind, double *total_ms, uint64_t *launches) {
  if (!total_ms || !launches) return set_error(SDRG_ERR_ARG, "null argument");
  std::lock_guard<std::mutex> lk(g_prof_mu);
  *total_ms = 0; *launches = 0;
  std::vector<ProfSpan> keep;
  for (const ProfSpan &sp : g_prof_spans) {
    if (sp.kind != kind) { keep.push_back(sp); continue; }
    SDRG_CUDA(cudaEventSynchronize(sp.b));
    float ms = 0;
    SDRG_CUDA(cudaEventElapsedTime(&ms, sp.a, sp.b));
    *total_ms += ms; *launches += 1;
    g_prof_pool.push_back(sp.a); g_prof_pool.push_back(sp.b);
  }
  g_prof_spans.swap(keep);
  return SDRG_OK;
}

// ---- buffers -----------------------------------------------------------------------------------
int sdrg_buffer_alloc(size_t bytes, void **host_ptr) {
  if (!host_ptr) return set_error(SDRG_ERR_ARG, "null argument");
  *host_ptr = nullptr;
  ManagedBuffer b;
  b.bytes = bytes; b.device = g_device;
  SDRG_CUDA(cudaSetDevice(g_device));
  SDRG_CUDA(cudaHostAlloc((void **)&b.host, bytes ? bytes : 1, cudaHostAllocPortable));
  cudaError_t e = cudaMalloc((void **)&b.dev, bytes ? bytes : 1);
  if (e != cudaSuccess) { cudaFreeHost(b.host); return set_error(SDRG_ERR_CUDA, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e)); }
  e = cudaEventCreateWithFlags(&b.ready, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b.uploaded, cudaEventDisableTiming);
  if (e != cudaSuccess) {
    if (b.ready) cudaEventDestroy(b.ready);
    cudaFreeHost(b.host); cudaFree(b.dev);
    return set_error(SDRG_ERR_CUDA, "cudaEventCreate: %s", cudaGetErrorString(e));
  }
  std::lock_guard<std::mutex> lk(g_buf_mu);
  g_bufs[(uintptr_t)b.host] = b;
  *host_ptr = b.host;
  return SDRG_OK;
}

int sdrg_buffer_free(void *host_ptr) {
  if (!host_ptr) return SDRG_OK;
  ManagedBuffer b;
  {
    std::lock_guard<std::mutex> lk(g_buf_mu);
    auto it = g_bufs.find((uintptr_t)host_ptr);
    if (it == g_bufs.end()) return set_error(SDRG_ERR_ARG, "sdrg_buffer_free: %p is not a managed buffer", host_ptr);
    b = it->second;
    g_bufs.erase(it);
  }
  cudaSetDevice(b.device);
  cudaEventSynchronize(b.ready);
  if (b.upload_pending) cudaEventSynchronize(b.uploaded);
  cudaEventDestroy(b.ready);
  cudaEventDestroy(b.uploaded);
  cudaFree(b.dev);
  cudaFreeHost(b.host);
  return SDRG_OK;
}

int sdrg_buffer_is_managed(const void *host_ptr, int *managed) {
  if (!managed) return set_error(SDRG_ERR_ARG, "null argument");
  std::lock_guard<std::mutex> lk(g_buf_mu);
  *managed = find_buffer(host_ptr) ? 1 : 0;
  return SDRG_OK;
}

int sdrg_buffer_device_ptr(const void *host_ptr, void **dev_ptr) {
  if (!dev_ptr) return set_error(SDRG_ERR_ARG, "null argument");
  std::lock_guard<std::mutex> lk(g_buf_mu);
  ManagedBuffer *b = find_buffer(host_ptr);
  *dev_ptr = b ? (void *)(b->dev + ((const char *)host_ptr - b->host)) : nullptr;
  return SDRG_OK;
}

int sdrg_buffer_mark_device_valid(const void *host_ptr, size_t bytes, void *stream) {
  std::lock_guard<std::mutex> lk(g_buf_mu);
  ManagedBuffer *b = find_buffer(host_ptr);
  if (!b) return set_error(SDRG_ERR_ARG, "not a managed buffer");
  b->valid_lo = (const char *)host_ptr - b->host;
  b->valid_hi = b->valid_lo + bytes;
  b->host_synced = false;
  SDRG_CUDA(cudaEventRecord(b->ready, (cudaStream_t)stream));
  return SDRG_OK;
}

int sdrg_buffer_device_valid(const void *host_ptr, size_t bytes, int *valid) {
  if (!valid) return set_error(SDRG_ERR_ARG, "null argument");
  std::lock_guard<std::mutex> lk(g_buf_mu);
  ManagedBuffer *b = find_buffer(host_ptr);
  *valid = 0;
  if (b && b->valid_hi > b->valid_lo) {
    const size_t lo = (const char *)host_ptr - b->host;
    if (lo >= b->valid_lo && lo + bytes <= b->valid_hi) *valid = 1;
  }
  return SDRG_OK;
}

// The host copy becomes authoritative again, i.e. the buffer goes back to whoever fills it on the host.
// The reference's process() is synchronous with respect to its input buffer; here an upload out of the pinned
// host memory may still be in flight (sdrg_buffer_to_device), so it is waited for before the producer may
// overwrite the bytes.
int sdrg_buffer_invalidate_device(const void *host_ptr) {
  cudaEvent_t wait = nullptr;
  int device = 0;
  {
    std::lock_guard<std::mutex> lk(g_buf_mu);
    ManagedBuffer *b = find_buffer(host_ptr);
    if (!b) return SDRG_OK;
    b->valid_lo = b->valid_hi = 0; b->host_synced = true;
    if (b->upload_pending) { wait = b->uploaded; device = b->device; b->upload_pending = false; }
  }
  if (wait) {
    SDRG_CUDA(cudaSetDevice(device));
    SDRG_CUDA(cudaEventSynchronize(wait));
  }
  return SDRG_OK;
}

int sdrg_buffer_sync_to_host(const void *host_ptr, size_t bytes) {
  ManagedBuffer snap;
  {
    std::lock_guard<std::mutex> lk(g_buf_mu);
    ManagedBuffer *b = find_buffer(host_ptr);
    if (!b || b->host_synced || b->valid_hi <= b->valid_lo) return SDRG_OK;
    const size_t lo = (const char *)host_ptr - b->host, hi = lo + bytes;
    if (hi <= b->valid_lo || lo >= b->valid_hi) return SDRG_OK;     // disjoint: host copy is current
    snap = *b;
    b->host_synced = true;
  }
  SDRG_CUDA(cudaSetDevice(snap.device));
  SDRG_CUDA(cudaEventSynchronize(snap.ready));
  SDRG_CUDA(cudaMemcpy(snap.host + snap.valid_lo, snap.dev + snap.valid_lo, snap.valid_hi - snap.valid_lo,
                       cudaMemcpyDeviceToHost));
  return SDRG_OK;
}

int sdrg_buffer_to_device(const void *host_ptr, size_t bytes, void *stream, void **dev_ptr) {
  if (!dev_ptr) return set_error(SDRG_ERR_ARG, "null argument");
  *dev_ptr = nullptr;
  char *dev = nullptr; bool copy = true; int device = 0;
  cudaEvent_t uploaded = nullptr;
  {
    std::lock_guard<std::mutex> lk(g_buf_mu);
    ManagedBuffer *b = find_buffer(host_ptr);
    if (!b) return SDRG_OK;
    const size_t lo = (const char *)host_ptr - b->host;
    if (lo + bytes > b->bytes) return set_error(SDRG_ERR_ARG, "sdrg_buffer_to_device: range exceeds the buffer");
    dev = b->dev + lo; device = b->device;
    if (b->valid_hi > b->valid_lo && lo >= b->valid_lo && lo + bytes <= b->valid_hi) copy = false;
    else { b->valid_lo = b->valid_hi = 0; b->host_synced = true; }     // the host copy is authoritative
    if (copy && bytes) { uploaded = b->uploaded; b->upload_pending = true; }
  }
  if (copy && bytes) {
    SDRG_CUDA(cudaSetDevice(device));
    SDRG_CUDA(cudaMemcpyAsync(dev, host_ptr, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    SDRG_CUDA(cudaEventRecord(uploaded, (cudaStream_t)stream));       // waited for in sdrg_buffer_invalidate_device / _free
  }
  *dev_ptr = dev;
  return SDRG_OK;
}

static std::mutex g_stream_mu;
static std::map<int, cudaStream_t> g_streams;
int sdrg_stream_default(void **stream) {
  if (!stream) return set_error(SDRG_ERR_ARG, "null argument");
  std::lock_guard<std::mutex> lk(g_stream_mu);
  auto it = g_streams.find(g_device);
  if (it == g_streams.end()) {
    cudaStream_t s = nullptr;
    SDRG_CUDA(cudaSetDevice(g_device));
    SDRG_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    it = g_streams.emplace(g_device, s).first;
  }
  *stream = (void *)it->second;
  return SDRG_OK;
}
int sdrg_stream_synchronize(void *stream) { SDRG_CUDA(cudaStreamSynchronize((cudaStream_t)stream)); return SDRG_OK; }

struct ThreadScratch { void *p = nullptr; size_t cap = 0; int device = -1; ~ThreadScratch() { if (p) cudaFree(p); } };
// slot 0: the caller's scratch (sdrg_scratch); slot 1: the library's own staging of aliased
// (in-place) results -- kept apart so that an input staged in slot 0 is never overwritten by it
static thread_local ThreadScratch g_scratch[3];   // slot 2: staging of outputs for foreign (unmanaged) host memory
static int scratch_slot(int slot, size_t bytes, void **dev_ptr) {
  ThreadScratch &sc = g_scratch[slot];
  if (sc.device != g_device || sc.cap < bytes) {
    SDRG_CUDA(cudaSetDevice(g_device));
    if (sc.p) { SDRG_CUDA(cudaDeviceSynchronize()); cudaFree(sc.p); sc.p = nullptr; sc.cap = 0; }
    const size_t want = bytes < 65536 ? 65536 : bytes + bytes / 2;
    SDRG_CUDA(cudaMalloc(&sc.p, want));
    sc.cap = want; sc.device = g_device;
  }
  *dev_ptr = sc.p;
  return SDRG_OK;
}
int sdrg_scratch(size_t bytes, void **dev_ptr) {
  if (!dev_ptr) return set_error(SDRG_ERR_ARG, "null argument");
  return scratch_slot(0, bytes, dev_ptr);
}
int sdrg_scratch_out(size_t bytes, void **dev_ptr) {
  if (!dev_ptr) return set_error(SDRG_ERR_ARG, "null argument");
  return scratch_slot(2, bytes, dev_ptr);
}
int sdrg_memcpy_h2d_async(void *d_dst, const void *h_src, size_t bytes, void *stream) {
  if (bytes) SDRG_CUDA(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
  return SDRG_OK;
}
int sdrg_memcpy_d2h_async(void *h_dst, const void *d_src, size_t bytes, void *stream) {
  if (bytes) SDRG_CUDA(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  return SDRG_OK;
}

// ---- IQBaseBand ---------------------------------------------------------------------------------
int sdrg_iqbb_create(int scalar, double Fc, double Ff, double width, size_t order, size_t sub_sample,
                     double oFs, sdrg_iqbb **out) {
  if (!out) return set_error(SDRG_ERR_ARG, "null argument");
  *out = nullptr;
  if (scalar != SDRG_T_S8 && scalar != SDRG_T_S16 && scalar != SDRG_T_F32)
    return set_error(SDRG_ERR_ARG, "IQBaseBand: unsupported scalar type %s (%d)", type_name(scalar), scalar);
  if (order > kMaxOrder) return set_error(SDRG_ERR_ARG, "IQBaseBand: order %zu exceeds %zu", order, kMaxOrder);
  sdrg_iqbb *h = new sdrg_iqbb();
  h->device = g_device;
  IqbbDesign &d = h->d;
  d.scalar = scalar;
  d.freq_shift = Fc;                       // FreqShiftBase<Scalar>(Fc, 0): the un-truncated double
  d.Fc = int32_t(Fc); d.Ff = int32_t(Ff); d.Fs = 0; d.width = int32_t(width);
  d.order = order < 1 ? 1 : order;
  d.sub_sample = sub_sample;
  d.oFs = oFs;
  design_lut(d);
  design_lut_increment(d, 0);
  *out = h;
  return SDRG_OK;
}

// BaseBand<Scalar>(Fc, Ff, width, order, sub_sample) on a REAL stream (src/baseband.hh:339-350), Scalar = int16_t or
// int8_t.  The int8 instantiation computes in 16 bits throughout (see iqbb_finalize.cuh::fin_value_s8_real).
int sdrg_iqbb_create_real(int scalar, double Fc, double Ff, double width, size_t order, size_t sub_sample,
                          sdrg_iqbb **out) {
  if (!out) return set_error(SDRG_ERR_ARG, "null argument");
  *out = nullptr;
  if (scalar != SDRG_T_S16 && scalar != SDRG_T_S8)
    return set_error(SDRG_ERR_ARG, "BaseBand: unsupported scalar type %s (%d), only int16 and int8", type_name(scalar), scalar);
  int rc = sdrg_iqbb_create(scalar, Fc, Ff, width, order, sub_sample, 0.0, out);
  if (rc) return rc;
  sdrg_iqbb *h = *out;
  h->real_input = true; h->in_fmt = scalar == SDRG_T_S8 ? 5 : 4;
  h->r_Ff = Ff; h->r_width = width;
  return SDRG_OK;
}

int sdrg_iqbb_destroy(sdrg_iqbb *h) {
  if (!h) return SDRG_OK;
  cudaSetDevice(h->device);
  if (h->stream) { cudaStreamSynchronize(h->stream); cudaStreamDestroy(h->stream); }
  else cudaDeviceSynchronize();
  free_dev(&h->d_taps); free_dev(&h->d_lut);
  free_dev(&h->d_hist[0]); free_dev(&h->d_hist[1]);
  free_dev(&h->d_acc[0]); free_dev(&h->d_acc[1]);
  free_dev(&h->d_tab_a); free_dev(&h->d_tab_u); free_dev(&h->d_tab_v); free_dev(&h->d_tab_cls);
  if (h->d_work) { cudaFree(h->d_work); h->d_work = nullptr; }
  free_dev(&h->d_in); free_dev(&h->d_out);
  delete h;
  return SDRG_OK;
}

// The setters mirror the reference: the filter setters only recompute the kernel (no state reset),
// setCenterFrequency restarts the NCO phase (freqshift.hh:86), the rate setters reconfigure.
static int refresh_kernel(sdrg_iqbb *h) {
  if (!h->configured) return SDRG_OK;
  SDRG_CUDA(cudaSetDevice(h->device));
  SDRG_CUDA(cudaDeviceSynchronize());
  const uint32_t old_hist = h->hist_len;
  design_filter(h);
  // the history buffers depend on the stripped tap count; keep them when it is unchanged
  std::vector<char> keep;
  const size_t sb = in_sample_bytes(h);
  if (old_hist) { keep.resize(old_hist * sb); SDRG_CUDA(cudaMemcpy(keep.data(), h->d_hist[h->parity], keep.size(), cudaMemcpyDeviceToHost)); }
  int rc = upload_design(h);
  if (rc) return rc;
  if (h->hist_len && old_hist) {   // newest samples are at the end of the history
    const size_t m = h->hist_len < old_hist ? h->hist_len : old_hist;
    SDRG_CUDA(cudaMemcpy((char *)h->d_hist[h->parity] + (h->hist_len - m) * sb, keep.data() + (old_hist - m) * sb,
                         m * sb, cudaMemcpyHostToDevice));
  }
  return SDRG_OK;
}

int sdrg_iqbb_set_center_frequency(sdrg_iqbb *h, double Fc) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  h->d.Fc = int32_t(Fc);
  h->d.freq_shift = h->real_input ? Fc     // FreqShiftBase::setFrequencyShift(double), freqshift.hh:62-65
                                  : double(h->d.Fc);   // IQBaseBand: setFrequencyShift(_Fc) receives the int32 member
  design_lut_increment(h->d, h->nco_Fs);
  h->phase0 = 0;                           // _lut_count = 0
  if (h->configured && h->d.scalar == SDRG_T_F32) {   // the folded tables embed the NCO increment
    SDRG_CUDA(cudaSetDevice(h->device));
    SDRG_CUDA(cudaDeviceSynchronize());
    return upload_fold_tables(h);
  }
  return SDRG_OK;
}
int sdrg_iqbb_set_filter_frequency(sdrg_iqbb *h, double Ff) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  h->d.Ff = int32_t(Ff); h->r_Ff = Ff;
  return refresh_kernel(h);
}
int sdrg_iqbb_set_filter_width(sdrg_iqbb *h, double width) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  h->d.width = int32_t(width); h->r_width = width;
  return refresh_kernel(h);
}
int sdrg_iqbb_set_order(sdrg_iqbb *h, size_t order) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (order > kMaxOrder) return set_error(SDRG_ERR_ARG, "IQBaseBand: order %zu exceeds %zu", order, kMaxOrder);
  h->d.order = order < 1 ? 1 : order;
  if (!h->configured) return SDRG_OK;
  SDRG_CUDA(cudaSetDevice(h->device));
  SDRG_CUDA(cudaDeviceSynchronize());
  design_filter(h);
  return upload_design(h);                 // fresh, zeroed history (the reference leaves it uninitialised)
}
int sdrg_iqbb_set_subsample(sdrg_iqbb *h, size_t sub_sample) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  h->d.sub_sample = sub_sample < 1 ? 1 : sub_sample;
  if (h->d.Fs == 0 || h->d.source_bs == 0) return SDRG_OK;
  SDRG_CUDA(cudaSetDevice(h->device));
  SDRG_CUDA(cudaDeviceSynchronize());
  return reconfigure(h);
}
int sdrg_iqbb_set_output_sample_rate(sdrg_iqbb *h, double oFs) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (h->real_input) return set_error(SDRG_ERR_CONFIG, "BaseBand: no output-rate setter (src/baseband.hh:304-529), use the sub-sampling");
  h->d.oFs = oFs;
  if (h->d.Fs == 0 || h->d.source_bs == 0) return SDRG_OK;
  SDRG_CUDA(cudaSetDevice(h->device));
  SDRG_CUDA(cudaDeviceSynchronize());
  return reconfigure(h);
}

int sdrg_iqbb_set_input_type(sdrg_iqbb *h, int type) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (h->configured) return set_error(SDRG_ERR_RUNTIME, "IQBaseBand: select the input type before config()");
  if (h->real_input) {
    if (type == h->d.scalar) return SDRG_OK;
    return set_error(SDRG_ERR_CONFIG, "Can not configure BaseBand: Invalid type %s (%d), expected %s (%d)", type_name(type), type,
                     type_name(h->d.scalar), h->d.scalar);
  }
  if (type == complex_type_of(h->d.scalar)) { h->in_fmt = 0; return SDRG_OK; }
  if (h->d.scalar != SDRG_T_S16 || (type != SDRG_T_CU8 && type != SDRG_T_CS8))
    return set_error(SDRG_ERR_CONFIG, "AutoCast: Can not cast from type %s (%d) to %s (%d)", type_name(type), type,
                     type_name(complex_type_of(h->d.scalar)), complex_type_of(h->d.scalar));
  h->in_fmt = type == SDRG_T_CU8 ? 2 : 3;
  return SDRG_OK;
}

int sdrg_iqbb_set_float_path(sdrg_iqbb *h, int mode) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (mode == 3) return set_error(SDRG_ERR_CONFIG, "IQBaseBand: there is no float path 3 (the TMA staging variant was removed)");
  if (mode < 0 || mode > 2) return set_error(SDRG_ERR_ARG, "IQBaseBand: float path must be 0 (auto), 1 (direct) or 2 (folded)");
  if (h->configured) return set_error(SDRG_ERR_RUNTIME, "IQBaseBand: select the float path before config()");
  h->float_path = mode;
  return SDRG_OK;
}

int sdrg_iqbb_last_float_kernel(const sdrg_iqbb *h, int *which) {
  if (!h || !which) return set_error(SDRG_ERR_ARG, "null argument");
  *which = h->last_float_kernel;
  return SDRG_OK;
}

int sdrg_iqbb_configure(sdrg_iqbb *h, const sdrg_config *src, sdrg_config *out) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (out) { out->type = SDRG_T_UNDEFINED; out->sample_rate = 0; out->buffer_size = 0; out->num_buffers = 0; }
  bool skip = false;
  int rc = config_common(node_name(h), input_type_of(h), src, true, &skip);
  if (rc || skip) return rc;
  SDRG_CUDA(cudaSetDevice(h->device));
  SDRG_CUDA(cudaDeviceSynchronize());
  h->d.Fs = int32_t(src->sample_rate); h->r_Fs = src->sample_rate;
  h->d.source_bs = src->buffer_size;
  rc = reconfigure(h);
  if (rc) return rc;
  if (out) {
    out->type = complex_type_of(h->d.scalar);
    out->sample_rate = h->d.out_rate;
    out->buffer_size = h->d.out_bs;
    out->num_buffers = 1;
  }
  return SDRG_OK;
}

int sdrg_iqbb_design(sdrg_iqbb *h, const sdrg_config *src, sdrg_config *out) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (out) { out->type = SDRG_T_UNDEFINED; out->sample_rate = 0; out->buffer_size = 0; out->num_buffers = 0; }
  bool skip = false;
  int rc = config_common(node_name(h), input_type_of(h), src, true, &skip);
  if (rc || skip) return rc;
  h->d.Fs = int32_t(src->sample_rate); h->r_Fs = src->sample_rate;
  h->d.source_bs = src->buffer_size;
  h->configured = false;                    // tables are not on the device
  rc = design_only(h);
  if (rc) return rc;
  if (out) {
    out->type = complex_type_of(h->d.scalar);
    out->sample_rate = h->d.out_rate; out->buffer_size = h->d.out_bs; out->num_buffers = 1;
  }
  return SDRG_OK;
}

int sdrg_iqbb_get_info(const sdrg_iqbb *h, sdrg_iqbb_info *info, void *kernel, void *lut) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  const IqbbDesign &d = h->d;
  if (info) {
    info->order = d.order; info->sub_sample = d.sub_sample; info->lut_inc = d.lut_inc;
    info->negative_shift = d.negative ? 1 : 0;
    info->samples_consumed = h->consumed; info->outputs_produced = h->produced;
  }
  if (kernel) {
    for (size_t i = 0; i < d.order; ++i) {
      if (d.scalar == SDRG_T_F32) { ((float *)kernel)[2 * i] = (float)d.kd_re[i]; ((float *)kernel)[2 * i + 1] = (float)d.kd_im[i]; }
      else { ((int32_t *)kernel)[2 * i] = d.k_re[i]; ((int32_t *)kernel)[2 * i + 1] = d.k_im[i]; }
    }
  }
  if (lut) {
    for (size_t j = 0; j < 128; ++j) {
      if (d.scalar == SDRG_T_F32) { ((float *)lut)[2 * j] = (float)d.lutd_re[j]; ((float *)lut)[2 * j + 1] = (float)d.lutd_im[j]; }
      else { ((int32_t *)lut)[2 * j] = d.lut_re[j]; ((int32_t *)lut)[2 * j + 1] = d.lut_im[j]; }
    }
  }
  return SDRG_OK;
}

int sdrg_iqbb_outputs_for(const sdrg_iqbb *h, size_t n_in, size_t *n_out) {
  if (!h || !n_out) return set_error(SDRG_ERR_ARG, "null argument");
  if (!h->configured) return set_error(SDRG_ERR_RUNTIME, "IQBaseBand: not configured");
  *n_out = (size_t)advance(h, n_in).n_out;
  return SDRG_OK;
}

int sdrg_iqbb_process_dev(sdrg_iqbb *h, const void *d_in, size_t n_in, void *d_out, size_t out_cap,
                          size_t *n_out, void *stream) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (n_out) *n_out = 0;
  const size_t total = (size_t)advance(h, n_in).n_out;
  if (total > out_cap) return set_error(SDRG_ERR_RUNTIME, "IQBaseBand: output buffer too small (%zu < %zu)", out_cap, total);
  SDRG_CUDA(cudaSetDevice(h->device));
  const size_t sb = sample_bytes(h->d.scalar), isb = in_sample_bytes(h);
  size_t done = 0, produced = 0;
  while (done < n_in) {
    const uint32_t n = (uint32_t)((n_in - done) > (1u << 30) ? (1u << 30) : (n_in - done));
    uint64_t got = 0;
    rc = run_call(h, (const char *)d_in + done * isb, n, (char *)d_out + produced * sb, nullptr, SDRG_DEMOD_NONE, 0, 0,
                  nullptr, nullptr, (cudaStream_t)stream, &got);
    if (rc) return rc;
    done += n; produced += got;
  }
  if (n_out) *n_out = produced;
  return SDRG_OK;
}

static int own_stream(cudaStream_t *s) {
  if (!*s) SDRG_CUDA(cudaStreamCreateWithFlags(s, cudaStreamNonBlocking));
  return SDRG_OK;
}

int sdrg_iqbb_process(sdrg_iqbb *h, const void *in, size_t n_in, void *out, size_t out_cap, size_t *n_out) {
  int rc = check_handle(h);
  if (rc) return rc;
  if (n_out) *n_out = 0;
  if (n_in == 0) return SDRG_OK;
  SDRG_CUDA(cudaSetDevice(h->device));
  if ((rc = own_stream(&h->stream))) return rc;
  const size_t sb = sample_bytes(h->d.scalar);
  const size_t total = (size_t)advance(h, n_in).n_out;
  if (total > out_cap) return set_error(SDRG_ERR_RUNTIME, "IQBaseBand: output buffer too small (%zu < %zu)", out_cap, total);
  const size_t isb = in_sample_bytes(h);
  if ((rc = grow(&h->d_in, &h->in_cap, n_in * isb))) return rc;
  if ((rc = grow(&h->d_out, &h->out_cap, (total + 1) * sb))) return rc;
  SDRG_CUDA(cudaMemcpyAsync(h->d_in, in, n_in * isb, cudaMemcpyHostToDevice, h->stream));
  size_t got = 0;
  rc = sdrg_iqbb_process_dev(h, h->d_in, n_in, h->d_out, total, &got, h->stream);
  if (rc) return rc;
  if (got) SDRG_CUDA(cudaMemcpyAsync(out, h->d_out, got * sb, cudaMemcpyDeviceToHost, h->stream));
  SDRG_CUDA(cudaStreamSynchronize(h->stream));
  if (n_out) *n_out = got;
  return SDRG_OK;
}

// ---- FMDemod ------------------------------------------------------------------------------------
int sdrg_fmdemod_create(int in_scalar, sdrg_fmdemod **out) {
  if (!out) return set_error(SDRG_ERR_ARG, "null argument");
  *out = nullptr;
  if (in_scalar != SDRG_T_S8 && in_scalar != SDRG_T_S16 && in_scalar != SDRG_T_F32)
    return set_error(SDRG_ERR_ARG, "FMDemod: unsupported scalar type %d", in_scalar);
  sdrg_fmdemod *h = new sdrg_fmdemod();
  h->scalar = in_scalar; h->device = g_device;
  cudaError_t e = cudaSetDevice(h->device);
  for (int k = 0; k < 2 && e == cudaSuccess; ++k) {
    e = cudaMalloc(&h->d_last[k], 8);
    if (e == cudaSuccess) e = cudaMemset(h->d_last[k], 0, 8);
  }
  if (e != cudaSuccess) { delete h; return set_error(SDRG_ERR_CUDA, "FMDemod: %s", cudaGetErrorString(e)); }
  *out = h;
  return SDRG_OK;
}
int sdrg_fmdemod_destroy(sdrg_fmdemod *h) {
  if (!h) return SDRG_OK;
  cudaSetDevice(h->device);
  if (h->stream) { cudaStreamSynchronize(h->stream); cudaStreamDestroy(h->stream); }
  else cudaDeviceSynchronize();
  free_dev(&h->d_last[0]); free_dev(&h->d_last[1]); free_dev(&h->d_in); free_dev(&h->d_out); free_dev(&h->d_alias);
  delete h;
  return SDRG_OK;
}
int sdrg_fmdemod_configure(sdrg_fmdemod *h, const sdrg_config *src, sdrg_config *out) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (out) { out->type = SDRG_T_UNDEFINED; out->sample_rate = 0; out->buffer_size = 0; out->num_buffers = 0; }
  bool skip = false;
  int rc = config_common("FMDemod", complex_type_of(h->scalar), src, false, &skip);
  if (rc || skip) return rc;
  SDRG_CUDA(cudaSetDevice(h->device));
  SDRG_CUDA(cudaDeviceSynchronize());
  SDRG_CUDA(cudaMemset(h->d_last[0], 0, 8));     // _last_value = 0 (demod.hh:210)
  SDRG_CUDA(cudaMemset(h->d_last[1], 0, 8));
  if (out) {
    out->type = h->scalar == SDRG_T_F32 ? SDRG_T_F32 : SDRG_T_S16;
    out->sample_rate = src->sample_rate; out->buffer_size = src->buffer_size; out->num_buffers = 1;
  }
  return SDRG_OK;
}
int sdrg_fmdemod_process_dev(sdrg_fmdemod *h, const void *d_in, size_t n, void *d_out, int in_place, void *stream) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (n == 0) return SDRG_OK;                    // demod.hh:231
  SDRG_CUDA(cudaSetDevice(h->device));
  const size_t ob = audio_bytes(h->scalar, SDRG_DEMOD_FM);
  void *dst = d_out;
  if (d_in == d_out) {            // true in-place use: form the result aside, then copy it over the input
    int rc = grow(&h->d_alias, &h->alias_cap, n * ob);
    if (rc) return rc;
    dst = h->d_alias; in_place = 1;
  }
  int rc = launch_fmdemod(h->scalar, d_in, n, dst, h->d_last[h->parity], h->d_last[h->parity ^ 1], in_place, (cudaStream_t)stream);
  if (rc) return rc;
  if (dst != d_out) SDRG_CUDA(cudaMemcpyAsync(d_out, dst, n * ob, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  h->parity ^= 1;
  return SDRG_OK;
}
int sdrg_fmdemod_process(sdrg_fmdemod *h, const void *in, size_t n, void *out, int in_place) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (n == 0) return SDRG_OK;
  SDRG_CUDA(cudaSetDevice(h->device));
  int rc = own_stream(&h->stream);
  if (rc) return rc;
  const size_t ib = sample_bytes(h->scalar), ob = audio_bytes(h->scalar, SDRG_DEMOD_FM);
  if ((rc = grow(&h->d_in, &h->in_cap, n * ib))) return rc;
  if ((rc = grow(&h->d_out, &h->out_cap, n * ob))) return rc;
  SDRG_CUDA(cudaMemcpyAsync(h->d_in, in, n * ib, cudaMemcpyHostToDevice, h->stream));
  // out of place: element 0 keeps whatever the caller's buffer holds
  if (!in_place) SDRG_CUDA(cudaMemcpyAsync(h->d_out, out, ob, cudaMemcpyHostToDevice, h->stream));
  rc = sdrg_fmdemod_process_dev(h, h->d_in, n, h->d_out, in_place, h->stream);
  if (rc) return rc;
  SDRG_CUDA(cudaMemcpyAsync(out, h->d_out, n * ob, cudaMemcpyDeviceToHost, h->stream));
  SDRG_CUDA(cudaStreamSynchronize(h->stream));
  return SDRG_OK;
}

// ---- AM / USB ----------------------------------------------------------------------------------
static int envelope_configure(const char *who, int scalar, const sdrg_config *src, sdrg_config *out, bool keep_num) {
  if (out) { out->type = SDRG_T_UNDEFINED; out->sample_rate = 0; out->buffer_size = 0; out->num_buffers = 0; }
  if (scalar != SDRG_T_S8 && scalar != SDRG_T_S16 && scalar != SDRG_T_F32)
    return set_error(SDRG_ERR_ARG, "%s: unsupported scalar type %d", who, scalar);
  bool skip = false;
  int rc = config_common(who, complex_type_of(scalar), src, false, &skip);
  if (rc || skip) return rc;
  if (out) {
    out->type = scalar; out->sample_rate = src->sample_rate; out->buffer_size = src->buffer_size;
    out->num_buffers = keep_num ? src->num_buffers : 1;
  }
  return SDRG_OK;
}
int sdrg_amdemod_configure(int scalar, const sdrg_config *src, sdrg_config *out) {
  return envelope_configure("AMDemod", scalar, src, out, true);      // demod.hh:60-61 keeps numBuffers
}
int sdrg_usbdemod_configure(int scalar, const sdrg_config *src, sdrg_config *out) {
  return envelope_configure("USBDemod", scalar, src, out, false);    // demod.hh:140-141 sets 1
}
static int envelope_dev(bool usb, int scalar, const void *d_in, size_t n, void *d_out, void *stream) {
  void *dst = d_out;
  const size_t ob = scalar_bytes(scalar);
  if (d_in == d_out && n) {       // in-place use (demod.hh:68, 145-147): result aside, then over the input
    int rc = scratch_slot(1, n * ob, &dst);
    if (rc) return rc;
  }
  int rc = usb ? launch_usbdemod(scalar, d_in, n, dst, (cudaStream_t)stream) : launch_amdemod(scalar, d_in, n, dst, (cudaStream_t)stream);
  if (rc) return rc;
  if (dst != d_out) SDRG_CUDA(cudaMemcpyAsync(d_out, dst, n * ob, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return SDRG_OK;
}
int sdrg_amdemod_process_dev(int scalar, const void *d_in, size_t n, void *d_out, void *stream) {
  return envelope_dev(false, scalar, d_in, n, d_out, stream);
}
int sdrg_usbdemod_process_dev(int scalar, const void *d_in, size_t n, void *d_out, void *stream) {
  return envelope_dev(true, scalar, d_in, n, d_out, stream);
}
static int envelope_host(bool usb, int scalar, const void *in, size_t n, void *out) {
  if (n == 0) return SDRG_OK;
  const size_t ib = sample_bytes(scalar), ob = scalar_bytes(scalar);
  if (!ob) return set_error(SDRG_ERR_ARG, "demod: unsupported scalar type %d", scalar);
  SDRG_CUDA(cudaSetDevice(g_device));
  void *d_in = nullptr, *d_out = nullptr;
  SDRG_CUDA(cudaMalloc(&d_in, n * ib));
  cudaError_t e = cudaMalloc(&d_out, n * ob);
  if (e != cudaSuccess) { cudaFree(d_in); return set_error(SDRG_ERR_CUDA, "cudaMalloc: %s", cudaGetErrorString(e)); }
  int rc = SDRG_OK;
  e = cudaMemcpy(d_in, in, n * ib, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) rc = usb ? launch_usbdemod(scalar, d_in, n, d_out, 0) : launch_amdemod(scalar, d_in, n, d_out, 0);
  if (e == cudaSuccess && rc == SDRG_OK) e = cudaMemcpy(out, d_out, n * ob, cudaMemcpyDeviceToHost);
  cudaFree(d_in); cudaFree(d_out);
  if (e != cudaSuccess) return set_error(SDRG_ERR_CUDA, "demod: %s", cudaGetErrorString(e));
  return rc;
}
int sdrg_amdemod_process(int scalar, const void *in, size_t n, void *out) { return envelope_host(false, scalar, in, n, out); }
int sdrg_usbdemod_process(int scalar, const void *in, size_t n, void *out) { return envelope_host(true, scalar, in, n, out); }

// ---- AutoCast / FMDeemph ----------------------------------------------------------------------------
// (in_type, out_type) -> cast kind of demod_kernels.cu (0 = identity, -1 = the reference refuses the pair), bytes per
// input element, output bytes per input element  (src/autocast.hh:30-69)
static int cast_kind(int in_type, int out_type, size_t *in_elem, size_t *out_per_in, size_t *scalars_per_elem) {
  static const size_t elem[] = {0, 1, 1, 2, 2, 4, 8, 2, 2, 4, 4, 8, 16};
  if (in_type < SDRG_T_U8 || in_type > SDRG_T_CF64) return -1;
  *in_elem = elem[in_type];
  const bool cin = in_type >= SDRG_T_CU8;
  *scalars_per_elem = cin ? 2 : 1;
  int k = -1;
  switch (out_type) {
    case SDRG_T_S8:
      k = in_type == SDRG_T_U8 ? 1 : in_type == SDRG_T_S8 ? 0 : in_type == SDRG_T_U16 ? 2 : in_type == SDRG_T_S16 ? 3 : -1; break;
    case SDRG_T_CS8:
      k = in_type == SDRG_T_U8 ? 4 : in_type == SDRG_T_S8 ? 5 : in_type == SDRG_T_CU8 ? 1 : in_type == SDRG_T_CS8 ? 0 :
          in_type == SDRG_T_U16 ? 6 : in_type == SDRG_T_S16 ? 7 : in_type == SDRG_T_CU16 ? 2 : in_type == SDRG_T_CS16 ? 3 : -1; break;
    case SDRG_T_S16:
      k = in_type == SDRG_T_U8 ? 8 : in_type == SDRG_T_S8 ? 9 : in_type == SDRG_T_U16 ? 10 : in_type == SDRG_T_S16 ? 0 : -1; break;
    case SDRG_T_CS16:
      k = in_type == SDRG_T_U8 ? 11 : in_type == SDRG_T_S8 ? 12 : in_type == SDRG_T_CU8 ? 8 : in_type == SDRG_T_CS8 ? 9 :
          in_type == SDRG_T_U16 ? 13 : in_type == SDRG_T_S16 ? 14 : in_type == SDRG_T_CU16 ? 10 : in_type == SDRG_T_CS16 ? 0 : -1; break;
    default: break;
  }
  if (k < 0) return -1;
  const size_t out_scalar = (out_type == SDRG_T_S8 || out_type == SDRG_T_CS8) ? 1 : 2;
  const bool complexify = (k >= 4 && k <= 7) || k >= 11;          // real scalar in, complex value out
  *out_per_in = k == 0 ? *in_elem : (*scalars_per_elem) * out_scalar * (complexify ? 2 : 1);
  return k;
}

int sdrg_autocast_out_bytes(int in_type, int out_type, size_t n, size_t *bytes) {
  size_t ie = 0, opi = 0, spe = 0;
  if (!bytes) return set_error(SDRG_ERR_ARG, "null argument");
  if (cast_kind(in_type, out_type, &ie, &opi, &spe) < 0)
    return set_error(SDRG_ERR_CONFIG, "AutoCast: Can not cast from type %s (%d) to %s (%d)", type_name(in_type), in_type,
                     type_name(out_type), out_type);
  *bytes = n * opi;
  return SDRG_OK;
}
int sdrg_autocast_process_dev(int in_type, int out_type, const void *d_in, size_t n, void *d_out, void *stream) {
  size_t ie = 0, opi = 0, spe = 0;
  const int k = cast_kind(in_type, out_type, &ie, &opi, &spe);
  if (k < 0)
    return set_error(SDRG_ERR_CONFIG, "AutoCast: Can not cast from type %s (%d) to %s (%d)", type_name(in_type), in_type,
                     type_name(out_type), out_type);
  if (k == 0) {                   // _identity: the bytes as they are
    if (n && d_in != d_out) SDRG_CUDA(cudaMemcpyAsync(d_out, d_in, n * ie, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return SDRG_OK;
  }
  return launch_autocast(k, d_in, n * spe, d_out, (cudaStream_t)stream);
}
int sdrg_autocast_process(int in_type, int out_type, const void *in, size_t n, void *out) {
  if (!n) return SDRG_OK;
  size_t ie = 0, opi = 0, spe = 0;
  if (cast_kind(in_type, out_type, &ie, &opi, &spe) < 0)
    return set_error(SDRG_ERR_CONFIG, "AutoCast: Can not cast from type %s (%d) to %s (%d)", type_name(in_type), in_type,
                     type_name(out_type), out_type);
  SDRG_CUDA(cudaSetDevice(g_device));
  const size_t ib = n * ie, ob = n * opi, off = (ib + 15) & ~(size_t)15;
  void *d = nullptr;
  int rc = sdrg_scratch(off + ob, &d);
  if (rc) return rc;
  SDRG_CUDA(cudaMemcpy(d, in, ib, cudaMemcpyHostToDevice));
  rc = sdrg_autocast_process_dev(in_type, out_type, d, n, (char *)d + off, 0);
  if (rc) return rc;
  SDRG_CUDA(cudaMemcpy(out, (char *)d + off, ob, cudaMemcpyDeviceToHost));
  return SDRG_OK;
}

struct sdrg_fmdeemph_impl { int device; size_t streams; int alpha; bool enabled; void *d_avg; };
int sdrg_fmdeemph_create(size_t streams, sdrg_fmdeemph **out) {
  if (!out || !streams) return set_error(SDRG_ERR_ARG, "FMDeemph: bad argument");
  sdrg_fmdeemph_impl *h = new sdrg_fmdeemph_impl{g_device, streams, 0, true, nullptr};
  *out = (sdrg_fmdeemph *)h;
  return SDRG_OK;
}
int sdrg_fmdeemph_destroy(sdrg_fmdeemph *hh) {
  sdrg_fmdeemph_impl *h = (sdrg_fmdeemph_impl *)hh;
  if (!h) return SDRG_OK;
  cudaSetDevice(h->device); cudaDeviceSynchronize();
  if (h->d_avg) cudaFree(h->d_avg);
  delete h;
  return SDRG_OK;
}
int sdrg_fmdeemph_configure(sdrg_fmdeemph *hh, const sdrg_config *src, sdrg_config *out) {
  sdrg_fmdeemph_impl *h = (sdrg_fmdeemph_impl *)hh;
  if (!h || !src) return set_error(SDRG_ERR_ARG, "null argument");
  if (out) { out->type = SDRG_T_UNDEFINED; out->sample_rate = 0; out->buffer_size = 0; out->num_buffers = 0; }
  if (src->type == SDRG_T_UNDEFINED || src->sample_rate == 0 || src->buffer_size == 0) return SDRG_OK;   // demod.hh:300
  if (src->type != SDRG_T_S16)
    return set_error(SDRG_ERR_CONFIG, "Can not configure FMDeemph: Invalid type %s (%d), expected %s (%d)",
                     type_name(src->type), src->type, type_name(SDRG_T_S16), SDRG_T_S16);
  h->alpha = (int)round(1.0 / ((1.0 - exp(-1.0 / (src->sample_rate * 75e-6)))));   // demod.hh:309-310
  SDRG_CUDA(cudaSetDevice(h->device));
  if (!h->d_avg) SDRG_CUDA(cudaMalloc(&h->d_avg, h->streams * 2));
  SDRG_CUDA(cudaDeviceSynchronize());
  SDRG_CUDA(cudaMemset(h->d_avg, 0, h->streams * 2));                              // _avg = 0
  if (out) { out->type = SDRG_T_S16; out->sample_rate = src->sample_rate; out->buffer_size = src->buffer_size; out->num_buffers = 1; }
  return SDRG_OK;
}
int sdrg_fmdeemph_process_dev(sdrg_fmdeemph *hh, const void *d_in, size_t n, size_t stride, void *d_out, void *stream) {
  sdrg_fmdeemph_impl *h = (sdrg_fmdeemph_impl *)hh;
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (!h->alpha) return set_error(SDRG_ERR_RUNTIME, "FMDeemph: process() before config()");
  SDRG_CUDA(cudaSetDevice(h->device));
  return launch_fmdeemph(d_in, d_out, n, h->streams, stride, h->alpha, h->d_avg, (cudaStream_t)stream);
}
int sdrg_fmdeemph_process(sdrg_fmdeemph *hh, const void *in, size_t n, size_t stride, void *out) {
  sdrg_fmdeemph_impl *h = (sdrg_fmdeemph_impl *)hh;
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (!n) return SDRG_OK;
  SDRG_CUDA(cudaSetDevice(h->device));
  const size_t bytes = ((h->streams - 1) * stride + n) * 2;
  void *d = nullptr;
  int rc = sdrg_scratch(bytes, &d);
  if (rc) return rc;
  SDRG_CUDA(cudaMemcpy(d, in, bytes, cudaMemcpyHostToDevice));
  rc = sdrg_fmdeemph_process_dev(hh, d, n, stride, d, 0);        // in place is safe: one thread per stream
  if (rc) return rc;
  SDRG_CUDA(cudaMemcpy(out, d, bytes, cudaMemcpyDeviceToHost));
  return SDRG_OK;
}

// ---- receive chain -------------------------------------------------------------------------------
int sdrg_rxchain_create(sdrg_iqbb *bb, int demod, sdrg_rxchain **out) {
  if (!bb || !out) return set_error(SDRG_ERR_ARG, "null argument");
  *out = nullptr;
  if (demod < SDRG_DEMOD_NONE || demod > SDRG_DEMOD_USB) return set_error(SDRG_ERR_ARG, "rxchain: unknown demodulator %d", demod);
  sdrg_rxchain *h = new sdrg_rxchain();
  h->bb = bb; h->demod = demod;
  cudaError_t e = cudaSetDevice(bb->device);
  for (int k = 0; k < 2 && e == cudaSuccess; ++k) {
    e = cudaMalloc(&h->d_last[k], 8);
    if (e == cudaSuccess) e = cudaMemset(h->d_last[k], 0, 8);
  }
  if (e != cudaSuccess) { delete h; return set_error(SDRG_ERR_CUDA, "rxchain: %s", cudaGetErrorString(e)); }
  *out = h;
  return SDRG_OK;
}
int sdrg_rxchain_destroy(sdrg_rxchain *h) {
  if (!h) return SDRG_OK;
  cudaSetDevice(h->bb->device);
  cudaDeviceSynchronize();
  free_dev(&h->d_last[0]); free_dev(&h->d_last[1]);
  free_dev(&h->d_in); free_dev(&h->d_bb); free_dev(&h->d_audio);
  for (int k = 0; k < 2; ++k) if (h->copy_st[k]) cudaStreamDestroy(h->copy_st[k]);
  for (cudaEvent_t e : h->copy_ev) cudaEventDestroy(e);
  delete h;
  return SDRG_OK;
}
int sdrg_rxchain_reset(sdrg_rxchain *h) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  SDRG_CUDA(cudaSetDevice(h->bb->device));
  SDRG_CUDA(cudaDeviceSynchronize());
  SDRG_CUDA(cudaMemset(h->d_last[0], 0, 8));
  SDRG_CUDA(cudaMemset(h->d_last[1], 0, 8));
  return SDRG_OK;
}

int sdrg_rxchain_process_dev(sdrg_rxchain *h, const void *d_in, size_t buffer_size, size_t n_buffers,
                             void *d_bb, void *d_audio, size_t out_cap, size_t *n_out, size_t *counts,
                             void *stream) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  sdrg_iqbb *bb = h->bb;
  int rc = check_handle(bb);
  if (rc) return rc;
  if (n_out) *n_out = 0;
  if (buffer_size == 0 || n_buffers == 0) return SDRG_OK;
  if (buffer_size > (1u << 30)) return set_error(SDRG_ERR_ARG, "rxchain: buffer_size %zu exceeds 2^30", buffer_size);
  const size_t n_in = buffer_size * n_buffers;
  const size_t total = (size_t)advance(bb, n_in).n_out;
  if (total > out_cap) return set_error(SDRG_ERR_RUNTIME, "rxchain: output buffers too small (%zu < %zu)", out_cap, total);
  if (counts) {    // per-buffer output counts, closed form
    size_t prev = 0;
    for (size_t b = 0; b < n_buffers; ++b) {
      const size_t upto = (size_t)advance(bb, (b + 1) * buffer_size).n_out;
      counts[b] = upto - prev; prev = upto;
    }
  }
  SDRG_CUDA(cudaSetDevice(bb->device));
  const size_t sb = sample_bytes(bb->d.scalar), ab = audio_bytes(bb->d.scalar, h->demod);
  const size_t per_call = ((size_t)1 << 30) / buffer_size;     // whole buffers per launch
  size_t done_b = 0, produced = 0;
  while (done_b < n_buffers) {
    const size_t nb = (n_buffers - done_b) < per_call ? (n_buffers - done_b) : per_call;
    uint64_t got = 0;
    rc = run_call(bb, (const char *)d_in + done_b * buffer_size * in_sample_bytes(bb), (uint32_t)(nb * buffer_size),
                  d_bb ? (char *)d_bb + produced * sb : nullptr,
                  (d_audio && h->demod != SDRG_DEMOD_NONE) ? (char *)d_audio + produced * ab : nullptr,
                  h->demod, buffer_size, 1, h->d_last[h->parity], h->d_last[h->parity ^ 1],
                  (cudaStream_t)stream, &got);
    if (rc) return rc;
    if (h->demod == SDRG_DEMOD_FM) h->parity ^= 1;
    done_b += nb; produced += got;
  }
  if (n_out) *n_out = produced;
  return SDRG_OK;
}

int sdrg_rxchain_process(sdrg_rxchain *h, const void *in, size_t buffer_size, size_t n_buffers,
                         void *bb_out, void *audio, size_t out_cap, size_t *n_out, size_t *counts) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  sdrg_iqbb *bb = h->bb;
  int rc = check_handle(bb);
  if (rc) return rc;
  if (n_out) *n_out = 0;
  if (buffer_size == 0 || n_buffers == 0) return SDRG_OK;
  SDRG_CUDA(cudaSetDevice(bb->device));
  if ((rc = own_stream(&bb->stream))) return rc;
  const size_t n_in = buffer_size * n_buffers;
  const size_t total = (size_t)advance(bb, n_in).n_out;
  if (total > out_cap) return set_error(SDRG_ERR_RUNTIME, "rxchain: output buffers too small (%zu < %zu)", out_cap, total);
  const size_t sb = sample_bytes(bb->d.scalar), ab = audio_bytes(bb->d.scalar, h->demod);
  const size_t isb = in_sample_bytes(bb);
  if ((rc = grow(&h->d_in, &h->in_cap, n_in * isb))) return rc;
  if ((rc = grow(&h->d_bb, &h->bb_cap, (total + 1) * sb))) return rc;
  if ((rc = grow(&h->d_audio, &h->audio_cap, (total + 1) * (ab ? ab : 1)))) return rc;
  // Upload in chunks of whole buffers (>= 64 MiB each, at most 16 chunks) on two alternating copy streams;
  // the compute stream waits for chunk i only, so its kernels overlap the upload of chunk i+1.
  const size_t buf_bytes = buffer_size * isb;
  size_t per_chunk = ((size_t)64 << 20) / (buf_bytes ? buf_bytes : 1);
  if (per_chunk < 1) per_chunk = 1;
  if ((n_buffers + per_chunk - 1) / per_chunk > 16) per_chunk = (n_buffers + 15) / 16;
  const size_t n_chunks = (n_buffers + per_chunk - 1) / per_chunk;
  for (int k = 0; k < 2; ++k)
    if (!h->copy_st[k]) SDRG_CUDA(cudaStreamCreateWithFlags(&h->copy_st[k], cudaStreamNonBlocking));
  while (h->copy_ev.size() < n_chunks) {
    cudaEvent_t e = nullptr;
    SDRG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    h->copy_ev.push_back(e);
  }
  size_t got = 0;
  for (size_t c = 0; c < n_chunks; ++c) {
    const size_t b0 = c * per_chunk, nb = (n_buffers - b0) < per_chunk ? (n_buffers - b0) : per_chunk;
    cudaStream_t cs = n_chunks > 1 ? h->copy_st[c & 1] : bb->stream;
    SDRG_CUDA(cudaMemcpyAsync((char *)h->d_in + b0 * buf_bytes, (const char *)in + b0 * buf_bytes, nb * buf_bytes,
                              cudaMemcpyHostToDevice, cs));
    if (n_chunks > 1) {
      SDRG_CUDA(cudaEventRecord(h->copy_ev[c], cs));
      SDRG_CUDA(cudaStreamWaitEvent(bb->stream, h->copy_ev[c], 0));
    }
    size_t g = 0;
    rc = sdrg_rxchain_process_dev(h, (char *)h->d_in + b0 * buf_bytes, buffer_size, nb, (char *)h->d_bb + got * sb,
                                  (char *)h->d_audio + got * ab, total - got, &g, counts ? counts + b0 : nullptr, bb->stream);
    if (rc) { cudaStreamSynchronize(h->copy_st[0]); cudaStreamSynchronize(h->copy_st[1]); return rc; }
    got += g;
  }
  if (got && bb_out) SDRG_CUDA(cudaMemcpyAsync(bb_out, h->d_bb, got * sb, cudaMemcpyDeviceToHost, bb->stream));
  if (got && audio && h->demod != SDRG_DEMOD_NONE)
    SDRG_CUDA(cudaMemcpyAsync(audio, h->d_audio, got * ab, cudaMemcpyDeviceToHost, bb->stream));
  SDRG_CUDA(cudaStreamSynchronize(bb->stream));
  if (n_out) *n_out = got;
  return SDRG_OK;
}

}  // extern "C"

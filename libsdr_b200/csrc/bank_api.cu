// bank_api.cu -- C ABI of the channel bank: C independent IQBaseBand<Scalar> chains on one input
// stream, each followed by FM / AM / USB demodulators connected out of place (several sinks on one
// source, src/node.cc:75), i.e. BASELINE configs 4 and 5.  Per channel the results are bit-identical
// to an IQBaseBand<Scalar>(Fc_k, Ff_k, width, order, sub_sample, oFs) node fed the same buffers (int8 / int16);
// float channels match the float node to rounding (folded weights, bank_fold_f32_kernel).
#include "iqbb_kernels.cuh"

#include <vector>

using namespace sdrg;

struct sdrg_bank {
  int scalar = SDRG_T_S16, device = 0;
  size_t channels = 0;
  std::vector<IqbbDesign> d;
  bool configured = false;
  uint32_t taps_len = 1, hist_len = 0;
  void *d_taps = nullptr, *d_lut = nullptr, *d_inc = nullptr, *d_neg = nullptr, *d_tab_u = nullptr;
  void *d_hist[2] = {nullptr, nullptr};
  void *d_acc[2] = {nullptr, nullptr};
  size_t acc_stride = 0; uint32_t acc_dirty[2] = {0, 0};
  void *d_fm_last[2] = {nullptr, nullptr};
  int parity = 0, fm_parity = 0;
  uint64_t consumed = 0;
  size_t source_bs = 0, out_bs = 0; double out_rate = 0;
  cudaStream_t stream = nullptr;
  void *d_in = nullptr; size_t in_cap = 0;
  void *d_out[4] = {nullptr, nullptr, nullptr, nullptr}; size_t out_cap[4] = {0, 0, 0, 0};
};

namespace {
size_t sample_bytes(int scalar) { return 2 * scalar_bytes(scalar); }
size_t fm_bytes(int scalar) { return scalar == SDRG_T_F32 ? 4 : 2; }
void free_dev(void **p) { if (*p) { cudaFree(*p); *p = nullptr; } }

int ensure_acc(sdrg_bank *h, size_t slots) {
  if (h->acc_stride >= slots) return SDRG_OK;
  const size_t stride = slots + slots / 2 + 64;
  void *n0 = nullptr, *n1 = nullptr;
  const size_t bytes = stride * h->channels * 8;
  SDRG_CUDA(cudaMalloc(&n0, bytes)); SDRG_CUDA(cudaMalloc(&n1, bytes));
  SDRG_CUDA(cudaMemset(n0, 0, bytes)); SDRG_CUDA(cudaMemset(n1, 0, bytes));
  if (h->d_acc[0]) {      // keep the open windows: 2 slots per channel of the current parity
    SDRG_CUDA(cudaDeviceSynchronize());
    SDRG_CUDA(cudaMemcpy2D(h->parity == 0 ? n0 : n1, stride * 8, h->d_acc[h->parity], h->acc_stride * 8, 16, h->channels, cudaMemcpyDeviceToDevice));
    cudaFree(h->d_acc[0]); cudaFree(h->d_acc[1]);
  }
  h->d_acc[0] = n0; h->d_acc[1] = n1; h->acc_stride = stride;
  h->acc_dirty[0] = h->acc_dirty[1] = 0;
  return SDRG_OK;
}

int grow(void **p, size_t *cap, size_t need) {
  if (*cap >= need && *p) return SDRG_OK;
  if (*p) { SDRG_CUDA(cudaDeviceSynchronize()); SDRG_CUDA(cudaFree(*p)); }
  *p = nullptr; *cap = 0;
  SDRG_CUDA(cudaMalloc(p, need ? need : 16));
  *cap = need;
  return SDRG_OK;
}
}  // namespace

extern "C" {

int sdrg_bank_create(int scalar, size_t n_channels, const double *Fc, const double *Ff, double width, size_t order,
                     size_t sub_sample, double oFs, sdrg_bank **out) {
  if (!out || !Fc) return set_error(SDRG_ERR_ARG, "null argument");
  *out = nullptr;
  if (scalar != SDRG_T_S8 && scalar != SDRG_T_S16 && scalar != SDRG_T_F32) return set_error(SDRG_ERR_ARG, "bank: scalar must be int8, int16 or float");
  if (n_channels == 0) return set_error(SDRG_ERR_ARG, "bank: no channels");
  if (order > 256) return set_error(SDRG_ERR_ARG, "bank: order %zu exceeds 256", order);
  sdrg_bank *h = new sdrg_bank();
  cudaGetDevice(&h->device);
  h->scalar = scalar; h->channels = n_channels;
  h->d.resize(n_channels);
  for (size_t c = 0; c < n_channels; ++c) {
    IqbbDesign &d = h->d[c];
    d.scalar = scalar;
    d.freq_shift = Fc[c];
    d.Fc = int32_t(Fc[c]); d.Ff = int32_t(Ff ? Ff[c] : Fc[c]); d.Fs = 0; d.width = int32_t(width);
    d.order = order < 1 ? 1 : order;
    d.sub_sample = sub_sample; d.oFs = oFs;
    design_lut(d);
  }
  *out = h;
  return SDRG_OK;
}

int sdrg_bank_destroy(sdrg_bank *h) {
  if (!h) return SDRG_OK;
  cudaSetDevice(h->device); cudaDeviceSynchronize();
  if (h->stream) cudaStreamDestroy(h->stream);
  free_dev(&h->d_taps); free_dev(&h->d_lut); free_dev(&h->d_inc); free_dev(&h->d_neg); free_dev(&h->d_tab_u);
  free_dev(&h->d_hist[0]); free_dev(&h->d_hist[1]); free_dev(&h->d_acc[0]); free_dev(&h->d_acc[1]);
  free_dev(&h->d_fm_last[0]); free_dev(&h->d_fm_last[1]); free_dev(&h->d_in);
  for (int k = 0; k < 4; ++k) free_dev(&h->d_out[k]);
  delete h;
  return SDRG_OK;
}

int sdrg_bank_configure(sdrg_bank *h, const sdrg_config *src, sdrg_config *out) {
  if (!h || !src) return set_error(SDRG_ERR_ARG, "null argument");
  if (out) { out->type = SDRG_T_UNDEFINED; out->sample_rate = 0; out->buffer_size = 0; out->num_buffers = 0; }
  if (src->type == SDRG_T_UNDEFINED || src->sample_rate == 0 || src->buffer_size == 0) return SDRG_OK;
  const int want = complex_type_of(h->scalar);
  if (src->type != want)
    return set_error(SDRG_ERR_CONFIG, "Can not configure IQBaseBand: Invalid type %s (%d), expected %s (%d)",
                     type_name(src->type), src->type, type_name(want), want);
  SDRG_CUDA(cudaSetDevice(h->device));
  SDRG_CUDA(cudaDeviceSynchronize());
  const size_t C = h->channels;
  size_t ss = 0, lead = (size_t)-1, L = h->d[0].order;
  std::vector<uint32_t> inc(C), neg(C);
  for (size_t c = 0; c < C; ++c) {
    IqbbDesign &d = h->d[c];
    d.Fs = int32_t(src->sample_rate); d.source_bs = src->buffer_size;
    if (d.oFs > 0) { d.sub_sample = size_t(d.Fs / d.oFs); if (d.sub_sample < 1) d.sub_sample = 1; }
    if (d.sub_sample < 1) d.sub_sample = 1;
    design_kernel(d);
    design_lut_increment(d, double(d.Fs));
    inc[c] = (uint32_t)d.lut_inc; neg[c] = d.negative ? 1u : 0u;
    if (d.lut_inc > 0xffffffffull) return set_error(SDRG_ERR_CONFIG, "bank: NCO increment out of range");
    ss = d.sub_sample;
    size_t l = 0;
    if (h->scalar != SDRG_T_F32) while (l + 1 < L && d.k_re[l] == 0 && d.k_im[l] == 0) ++l;
    if (l < lead) lead = l;
  }
  if (ss < 256) return set_error(SDRG_ERR_CONFIG, "bank: the bank kernel needs sub-sampling >= 256 (got %zu); use IQBaseBand nodes", ss);
  if (ss > (1u << 30)) return set_error(SDRG_ERR_CONFIG, "bank: sub-sampling %zu too large", ss);
  const size_t Lp = L - lead;      // common leading zero taps are dropped (exact; integer taps only)
  free_dev(&h->d_taps); free_dev(&h->d_lut); free_dev(&h->d_inc); free_dev(&h->d_neg); free_dev(&h->d_tab_u);
  free_dev(&h->d_hist[0]); free_dev(&h->d_hist[1]);
  if (h->scalar == SDRG_T_F32) {
    // bank_fold_f32_kernel: taps [t][channel] and U_c(r, 0) [group][r][channel in group], channels padded to 32 with zeros
    const size_t Cp = (C + 31) / 32 * 32;
    std::vector<float> taps(2 * L * Cp, 0.0f), tab_u(2 * 256 * Cp, 0.0f), u(2 * 256), lut(256);
    for (size_t c = 0; c < C; ++c) {
      const IqbbDesign &d = h->d[c];
      for (size_t t = 0; t < L; ++t) { taps[2 * (t * Cp + c)] = (float)d.kd_re[t]; taps[2 * (t * Cp + c) + 1] = (float)d.kd_im[t]; }
      fold_table_u(d, 1, u.data());
      for (size_t r = 0; r < 256; ++r) {
        const size_t k = ((c / 32) * 256 + r) * 32 + c % 32;
        tab_u[2 * k] = u[2 * r]; tab_u[2 * k + 1] = u[2 * r + 1];
      }
    }
    for (size_t j = 0; j < 128; ++j) { lut[2 * j] = (float)h->d[0].lutd_re[j]; lut[2 * j + 1] = (float)h->d[0].lutd_im[j]; }
    SDRG_CUDA(cudaMalloc(&h->d_taps, taps.size() * 4)); SDRG_CUDA(cudaMemcpy(h->d_taps, taps.data(), taps.size() * 4, cudaMemcpyHostToDevice));
    SDRG_CUDA(cudaMalloc(&h->d_tab_u, tab_u.size() * 4)); SDRG_CUDA(cudaMemcpy(h->d_tab_u, tab_u.data(), tab_u.size() * 4, cudaMemcpyHostToDevice));
    SDRG_CUDA(cudaMalloc(&h->d_lut, 1024)); SDRG_CUDA(cudaMemcpy(h->d_lut, lut.data(), 1024, cudaMemcpyHostToDevice));
  } else {
    std::vector<int32_t> taps(4 * Lp * C), lut(256);
    for (size_t c = 0; c < C; ++c)
      for (size_t i = 0; i < Lp; ++i) {
        const uint32_t kr = (uint32_t)h->d[c].k_re[lead + i], ki = (uint32_t)h->d[c].k_im[lead + i];
        int32_t *t = &taps[4 * (c * Lp + i)];
        t[0] = (int32_t)kr; t[1] = (int32_t)(ki - kr); t[2] = (int32_t)(kr + ki); t[3] = 0;
      }
    for (size_t j = 0; j < 128; ++j) { lut[2 * j] = h->d[0].lut_re[j]; lut[2 * j + 1] = h->d[0].lut_im[j]; }
    SDRG_CUDA(cudaMalloc(&h->d_taps, taps.size() * 4)); SDRG_CUDA(cudaMemcpy(h->d_taps, taps.data(), taps.size() * 4, cudaMemcpyHostToDevice));
    SDRG_CUDA(cudaMalloc(&h->d_lut, 1024)); SDRG_CUDA(cudaMemcpy(h->d_lut, lut.data(), 1024, cudaMemcpyHostToDevice));
  }
  SDRG_CUDA(cudaMalloc(&h->d_inc, C * 4)); SDRG_CUDA(cudaMemcpy(h->d_inc, inc.data(), C * 4, cudaMemcpyHostToDevice));
  SDRG_CUDA(cudaMalloc(&h->d_neg, C * 4)); SDRG_CUDA(cudaMemcpy(h->d_neg, neg.data(), C * 4, cudaMemcpyHostToDevice));
  h->taps_len = (uint32_t)Lp; h->hist_len = (uint32_t)Lp - 1;
  const size_t hb = (h->hist_len ? h->hist_len : 1) * sample_bytes(h->scalar);
  for (int k = 0; k < 2; ++k) {
    SDRG_CUDA(cudaMalloc(&h->d_hist[k], hb)); SDRG_CUDA(cudaMemset(h->d_hist[k], 0, hb));
    if (!h->d_fm_last[k]) SDRG_CUDA(cudaMalloc(&h->d_fm_last[k], C * 8));
    SDRG_CUDA(cudaMemset(h->d_fm_last[k], 0, C * 8));
  }
  h->source_bs = src->buffer_size;
  h->out_bs = src->buffer_size / ss + (src->buffer_size % ss ? 1 : 0);
  h->out_rate = double(size_t(h->d[0].Fs) / ss);
  int rc = ensure_acc(h, h->out_bs + 3);
  if (rc) return rc;
  SDRG_CUDA(cudaMemset(h->d_acc[0], 0, h->acc_stride * C * 8));
  SDRG_CUDA(cudaMemset(h->d_acc[1], 0, h->acc_stride * C * 8));
  h->acc_dirty[0] = h->acc_dirty[1] = 0;
  h->parity = 0; h->fm_parity = 0; h->consumed = 0;
  h->configured = true;
  if (out) { out->type = want; out->sample_rate = h->out_rate; out->buffer_size = h->out_bs; out->num_buffers = 1; }
  return SDRG_OK;
}

int sdrg_bank_get_info(const sdrg_bank *h, size_t *channels, size_t *sub_sample, size_t channel, sdrg_iqbb_info *info, void *kernel) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (channels) *channels = h->channels;
  if (sub_sample) *sub_sample = h->d[0].sub_sample;
  if (channel >= h->channels) return set_error(SDRG_ERR_ARG, "bank: no channel %zu", channel);
  const IqbbDesign &d = h->d[channel];
  if (info) {
    info->order = d.order; info->sub_sample = d.sub_sample; info->lut_inc = d.lut_inc; info->negative_shift = d.negative ? 1 : 0;
    info->samples_consumed = h->consumed; info->outputs_produced = windows_done(h->consumed, d.sub_sample);
  }
  if (kernel) {
    for (size_t i = 0; i < d.order; ++i) {
      if (h->scalar == SDRG_T_F32) { ((float *)kernel)[2 * i] = (float)d.kd_re[i]; ((float *)kernel)[2 * i + 1] = (float)d.kd_im[i]; }
      else { ((int32_t *)kernel)[2 * i] = d.k_re[i]; ((int32_t *)kernel)[2 * i + 1] = d.k_im[i]; }
    }
  }
  return SDRG_OK;
}

int sdrg_bank_outputs_for(const sdrg_bank *h, size_t n_in, size_t *n_out) {
  if (!h || !n_out) return set_error(SDRG_ERR_ARG, "null argument");
  if (!h->configured) return set_error(SDRG_ERR_RUNTIME, "bank: not configured");
  *n_out = (size_t)window_advance(h->consumed, h->d[0].sub_sample, n_in).n_out;
  return SDRG_OK;
}

// n_buffers buffers of buffer_size samples; per channel c the outputs land at <ptr> + c*out_stride
// (elements).  Any of d_bb/d_fm/d_am/d_usb may be NULL.  FM: out of place, element 0 of every
// buffer is left untouched (demod.hh:245).
int sdrg_bank_process_dev(sdrg_bank *h, const void *d_in, size_t buffer_size, size_t n_buffers, void *d_bb, void *d_fm,
                          void *d_am, void *d_usb, size_t out_stride, size_t *n_out, void *stream) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (!h->configured) return set_error(SDRG_ERR_RUNTIME, "bank: process() before config()");
  if (n_out) *n_out = 0;
  if (!buffer_size || !n_buffers) return SDRG_OK;
  const size_t n_in = buffer_size * n_buffers;
  if (n_in > (1u << 30)) return set_error(SDRG_ERR_ARG, "bank: at most 2^30 samples per call");
  SDRG_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t ss = h->d[0].sub_sample;
  const WindowAdvance adv = window_advance(h->consumed, ss, n_in);
  if (adv.n_out > out_stride) return set_error(SDRG_ERR_RUNTIME, "bank: out_stride (%zu) smaller than the output (%zu)", out_stride, (size_t)adv.n_out);
  int rc = ensure_acc(h, adv.n_out + 3);
  if (rc) return rc;
  const int p = h->parity, q = p ^ 1;
  BankAccumArgs a{};
  a.x = d_in; a.hist_in = h->d_hist[p]; a.hist_out = h->d_hist[q];
  a.taps = h->d_taps; a.lut = h->d_lut; a.tab_u = h->d_tab_u; a.inc = (const uint32_t *)h->d_inc; a.neg = (const uint32_t *)h->d_neg;
  a.acc_cur = h->d_acc[p]; a.acc_next = h->d_acc[q]; a.acc_stride = h->acc_stride;
  a.n = (uint32_t)n_in; a.channels = (uint32_t)h->channels; a.group = 32;
  a.taps_len = h->taps_len; a.hist_len = h->hist_len; a.ss = (uint32_t)ss; a.r0 = adv.r0; a.first = adv.first;
  a.consumed15 = (uint32_t)(h->consumed & 0x7fffu); a.zero_next = h->acc_dirty[q];
  rc = launch_bank_accum(h->scalar, a, st);
  if (rc) return rc;
  IqbbFinalizeArgs f{};
  f.acc_cur = h->d_acc[p]; f.acc_next = h->d_acc[q];
  f.n_out = (uint32_t)adv.n_out; f.ss = (uint32_t)ss; f.e0 = adv.e0; f.seg = buffer_size; f.in_place = 0;
  f.fm_last_in = h->d_fm_last[h->fm_parity]; f.fm_last_out = h->d_fm_last[h->fm_parity ^ 1];
  BankFinalizeStrides s{h->acc_stride, out_stride, (uint32_t)sample_bytes(h->scalar), 0};
  bool bb_done = false, any = false;
  struct { void *ptr; int demod; uint32_t bytes; } outs[3] = {{d_fm, SDRG_DEMOD_FM, (uint32_t)fm_bytes(h->scalar)}, {d_am, SDRG_DEMOD_AM, (uint32_t)scalar_bytes(h->scalar)},
                                                             {d_usb, SDRG_DEMOD_USB, (uint32_t)scalar_bytes(h->scalar)}};
  for (int k = 0; k < 3; ++k) {
    if (!outs[k].ptr) continue;
    f.bb_out = bb_done ? nullptr : d_bb; bb_done = true; any = true;
    f.audio_out = outs[k].ptr; f.demod = (uint32_t)outs[k].demod; s.audio_bytes = outs[k].bytes;
    rc = launch_bank_finalize(h->scalar, f, s, (uint32_t)h->channels, st);
    if (rc) return rc;
  }
  if (!any) {
    f.bb_out = d_bb; f.audio_out = nullptr; f.demod = SDRG_DEMOD_NONE;
    rc = launch_bank_finalize(h->scalar, f, s, (uint32_t)h->channels, st);
    if (rc) return rc;
  }
  if (d_fm) h->fm_parity ^= 1;
  h->acc_dirty[p] = (uint32_t)adv.n_out + 2; h->acc_dirty[q] = 2;
  h->parity = q;
  h->consumed += n_in;
  if (n_out) *n_out = (size_t)adv.n_out;
  return SDRG_OK;
}

int sdrg_bank_process(sdrg_bank *h, const void *in, size_t buffer_size, size_t n_buffers, void *bb, void *fm, void *am,
                      void *usb, size_t out_stride, size_t *n_out) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (!h->configured) return set_error(SDRG_ERR_RUNTIME, "bank: process() before config()");
  SDRG_CUDA(cudaSetDevice(h->device));
  if (!h->stream) SDRG_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  const size_t n_in = buffer_size * n_buffers, sb = sample_bytes(h->scalar), C = h->channels;
  int rc = grow(&h->d_in, &h->in_cap, n_in * sb);
  if (rc) return rc;
  void *host[4] = {bb, fm, am, usb};
  const size_t eb[4] = {sb, fm_bytes(h->scalar), scalar_bytes(h->scalar), scalar_bytes(h->scalar)};
  void *dev[4] = {nullptr, nullptr, nullptr, nullptr};
  for (int k = 0; k < 4; ++k) {
    if (!host[k]) continue;
    if ((rc = grow(&h->d_out[k], &h->out_cap[k], C * out_stride * eb[k]))) return rc;
    dev[k] = h->d_out[k];
    // out-of-place FM leaves element 0 of each buffer untouched: start from the caller's bytes
    if (k == 1) SDRG_CUDA(cudaMemcpyAsync(dev[k], host[k], C * out_stride * eb[k], cudaMemcpyHostToDevice, h->stream));
  }
  SDRG_CUDA(cudaMemcpyAsync(h->d_in, in, n_in * sb, cudaMemcpyHostToDevice, h->stream));
  size_t got = 0;
  rc = sdrg_bank_process_dev(h, h->d_in, buffer_size, n_buffers, dev[0], dev[1], dev[2], dev[3], out_stride, &got, h->stream);
  if (rc) return rc;
  for (int k = 0; k < 4; ++k)
    if (host[k]) SDRG_CUDA(cudaMemcpyAsync(host[k], dev[k], C * out_stride * eb[k], cudaMemcpyDeviceToHost, h->stream));
  SDRG_CUDA(cudaStreamSynchronize(h->stream));
  if (n_out) *n_out = got;
  return SDRG_OK;
}

}  // extern "C"

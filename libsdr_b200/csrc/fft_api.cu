// fft_api.cu -- C ABI of FFTPlan<float> and of the FFT-convolution filter bank (FilterNode).
// Host-side design follows src/filternode.hh:17-28 (sinc_flt_kernel<float>, including its float
// precision choreography) and :186-203 (_updateFilter: zero-pad to 2N, forward DFT, divide by the
// l2 norm of the spectrum); the DFT of the taps is evaluated in double on the host.
#include "fft_kernels.cuh"

#include <cmath>
#include <complex>
#include <cstring>
#include <vector>

using namespace sdrg;

namespace {

int ilog2(size_t n) { int l = 0; while (((size_t)1 << l) < n) ++l; return l; }
bool pow2(size_t n) { return n && !(n & (n - 1)); }

int upload_twiddles(size_t n, void **d_tw) {
  std::vector<float> tw(2 * n);
  for (size_t k = 0; k < n; ++k) {
    const double a = -2.0 * M_PI * (double)k / (double)n;
    tw[2 * k] = (float)std::cos(a); tw[2 * k + 1] = (float)std::sin(a);
  }
  SDRG_CUDA(cudaMalloc(d_tw, tw.size() * sizeof(float)));
  SDRG_CUDA(cudaMemcpy(*d_tw, tw.data(), tw.size() * sizeof(float), cudaMemcpyHostToDevice));
  return SDRG_OK;
}

// in-place iterative radix-2 DFT in double (config-time only)
void host_fft(std::vector<std::complex<double> > &a) {
  const size_t n = a.size();
  for (size_t i = 1, j = 0; i < n; ++i) {
    size_t bit = n >> 1;
    for (; j & bit; bit >>= 1) j ^= bit;
    j ^= bit;
    if (i < j) std::swap(a[i], a[j]);
  }
  for (size_t len = 2; len <= n; len <<= 1) {
    for (size_t k = 0; k < len / 2; ++k) {
      const std::complex<double> w = std::polar(1.0, -2.0 * M_PI * (double)k / (double)len);
      for (size_t s = 0; s < n; s += len) {
        const std::complex<double> u = a[s + k], t = a[s + k + len / 2] * w;
        a[s + k] = u + t; a[s + k + len / 2] = u - t;
      }
    }
  }
}

// sinc_flt_kernel<float>(i, N, Fc, bw, Fs), src/filternode.hh:17-28
std::complex<float> sinc_tap(int i, int N, double Fc, double bw, double Fs) {
  std::complex<float> v;
  if ((N / 2) == i) v = M_PI * (bw / Fs);
  else v = std::sin(M_PI * (bw / Fs) * (i - N / 2)) / (i - N / 2);
  v *= std::exp(std::complex<float>(0.0, (2 * M_PI * Fc * i) / Fs));
  v *= (0.42 - 0.5 * cos((2 * M_PI * i) / N) + 0.08 * cos((4 * M_PI * i) / N));
  return v;
}

int upload_tab8k(void **d_tab) {
  std::vector<float> tab;
  fft8k_tables(tab);
  SDRG_CUDA(cudaMalloc(d_tab, tab.size() * sizeof(float)));
  SDRG_CUDA(cudaMemcpy(*d_tab, tab.data(), tab.size() * sizeof(float), cudaMemcpyHostToDevice));
  return SDRG_OK;
}

}  // namespace

struct sdrg_fft {
  int device = 0;
  size_t n = 0; int inverse = 0;
  AnyFft *plan = nullptr;                // shared-memory kernels (2..8192), four-step, or Bluestein (fft_general.cu)
  cudaStream_t stream = nullptr;
  void *d_in = nullptr, *d_out = nullptr; size_t cap = 0;
};

struct FilterBand { double fmin, fmax; std::vector<float> taps, kern, kern_m; };   // kern: 2B-point spectrum; kern_m: M-point (general path)

struct sdrg_filter {
  int device = 0;
  size_t block = 0; int log2n = 0;
  double Fs = 0;
  bool configured = false;
  std::vector<FilterBand> bands;
  void *d_tw = nullptr, *d_kern = nullptr; bool kern_dirty = true;
  void *d_kperm = nullptr, *d_tab8k = nullptr;         // block 4096: permuted spectra + tables of fft8k_kernels.cu
  GeneralOla *gen = nullptr;                           // blocks that are not a power of two <= 4096 (fft_general.cu)
  void *d_hist[2] = {nullptr, nullptr}; int parity = 0;
  void *d_pend = nullptr; size_t pending = 0;          // re-chunking (BufferNode): < block samples waiting
  void *d_stage = nullptr; size_t stage_cap = 0;
  void *d_spec = nullptr; size_t spec_cap = 0;         // filter banks: block spectra shared by the filters
  cudaStream_t stream = nullptr;
  void *d_in = nullptr, *d_out = nullptr; size_t in_cap = 0, out_cap = 0;
};

namespace {

// O(n^2) DFT in double with exact phase reduction (config time, sizes that are not a power of two)
void host_dft(std::vector<std::complex<double> > &a) {
  const size_t n = a.size();
  std::vector<std::complex<double> > w(n), out(n);
  for (size_t k = 0; k < n; ++k) w[k] = std::polar(1.0, -2.0 * M_PI * (double)k / (double)n);
  for (size_t k = 0; k < n; ++k) {
    std::complex<double> acc(0, 0);
    size_t idx = 0;
    for (size_t j = 0; j < n; ++j) { acc += a[j] * w[idx]; idx += k; if (idx >= n) idx -= n; }
    out[k] = acc;
  }
  a.swap(out);
}

int design_band(sdrg_filter *h, FilterBand &b) {
  const size_t N = h->block;
  const double Fs = h->Fs;
  const double fmin = std::max(b.fmin, -Fs / 2), fmax = std::min(b.fmax, Fs / 2);
  const double bw = fmax - fmin, Fc = fmin + bw / 2;
  b.taps.assign(2 * N, 0.f);
  b.kern.clear(); b.kern_m.clear();
  double e2 = 0;
  std::vector<std::complex<double> > z(2 * N, std::complex<double>(0, 0));
  for (size_t i = 0; i < N; ++i) {
    const std::complex<float> v = sinc_tap((int)i, (int)N, Fc, bw, Fs);
    b.taps[2 * i] = v.real(); b.taps[2 * i + 1] = v.imag();
    z[i] = std::complex<double>(v.real(), v.imag());
    e2 += std::norm(z[i]);
  }
  // l2 norm of the 2N-point spectrum (Buffer::norm2, src/buffer.hh:182-188) = sqrt(2N) |h|_2 by Parseval
  const double nrm = std::sqrt(2.0 * (double)N * e2);
  if (h->gen) {                 // general path: the same taps on the M-point grid
    const size_t M = h->gen->M;
    std::vector<std::complex<double> > zm(M, std::complex<double>(0, 0));
    for (size_t i = 0; i < N; ++i) zm[i] = z[i];
    host_fft(zm);
    b.kern_m.resize(2 * M);
    for (size_t i = 0; i < M; ++i) { b.kern_m[2 * i] = (float)(zm[i].real() / nrm); b.kern_m[2 * i + 1] = (float)(zm[i].imag() / nrm); }
  }
  if (pow2(2 * N)) host_fft(z);
  else if (2 * N <= 16384) host_dft(z);
  else z.clear();                // the reference-shaped 2N-point spectrum is for inspection only; too slow to form here
  if (!z.empty()) {
    b.kern.resize(4 * N);
    for (size_t i = 0; i < 2 * N; ++i) { b.kern[2 * i] = (float)(z[i].real() / nrm); b.kern[2 * i + 1] = (float)(z[i].imag() / nrm); }
  }
  h->kern_dirty = true;
  return SDRG_OK;
}

int upload_kernels(sdrg_filter *h) {
  if (!h->kern_dirty) return SDRG_OK;
  const size_t n2 = 2 * h->block, F = h->bands.size();
  if (h->d_kern) { SDRG_CUDA(cudaDeviceSynchronize()); cudaFree(h->d_kern); h->d_kern = nullptr; }
  if (h->d_kperm) { cudaFree(h->d_kperm); h->d_kperm = nullptr; }
  if (F && h->gen) {            // general path: M-point spectra
    const size_t M = h->gen->M;
    SDRG_CUDA(cudaMalloc(&h->d_kern, F * M * 2 * sizeof(float)));
    for (size_t f = 0; f < F; ++f)
      SDRG_CUDA(cudaMemcpy((float *)h->d_kern + f * M * 2, h->bands[f].kern_m.data(), M * 2 * sizeof(float), cudaMemcpyHostToDevice));
  } else if (F) {
    SDRG_CUDA(cudaMalloc(&h->d_kern, F * n2 * 2 * sizeof(float)));
    for (size_t f = 0; f < F; ++f)
      SDRG_CUDA(cudaMemcpy((float *)h->d_kern + f * n2 * 2, h->bands[f].kern.data(), n2 * 2 * sizeof(float), cudaMemcpyHostToDevice));
    if (n2 == 8192) {
      std::vector<float> kp(n2 * 2);
      SDRG_CUDA(cudaMalloc(&h->d_kperm, F * n2 * 2 * sizeof(float)));
      for (size_t f = 0; f < F; ++f) {
        fft8k_permute_kernel(h->bands[f].kern.data(), kp.data());
        SDRG_CUDA(cudaMemcpy((float *)h->d_kperm + f * n2 * 2, kp.data(), n2 * 2 * sizeof(float), cudaMemcpyHostToDevice));
      }
      if (!h->d_tab8k) { int rc = upload_tab8k(&h->d_tab8k); if (rc) return rc; }
    }
  }
  h->kern_dirty = false;
  return SDRG_OK;
}

int grow_dev(void **p, size_t *cap, size_t need) {
  if (*cap >= need && *p) return SDRG_OK;
  if (*p) { SDRG_CUDA(cudaDeviceSynchronize()); SDRG_CUDA(cudaFree(*p)); }
  *p = nullptr; *cap = 0;
  SDRG_CUDA(cudaMalloc(p, need ? need : 16));
  *cap = need;
  return SDRG_OK;
}

int own_stream(cudaStream_t *s) {
  if (!*s) SDRG_CUDA(cudaStreamCreateWithFlags(s, cudaStreamNonBlocking));
  return SDRG_OK;
}

}  // namespace

extern "C" {

// ---- FFTPlan<float> -------------------------------------------------------------------------------
int sdrg_fft_create(size_t n, int direction, sdrg_fft **out) {
  if (!out) return set_error(SDRG_ERR_ARG, "null argument");
  *out = nullptr;
  if (n == 0) return set_error(SDRG_ERR_CONFIG, "Can not construct FFT plan: Buffer is empty!");      // fftplan_fftw3.hh:93-97
  sdrg_fft *h = new sdrg_fft();
  int dev = 0; cudaGetDevice(&dev);
  h->device = dev; h->n = n; h->inverse = direction ? 1 : 0;
  h->plan = new AnyFft();
  const int rc = h->plan->init(n);
  if (rc) { delete h->plan; delete h; return rc; }
  *out = h;
  return SDRG_OK;
}
int sdrg_fft_destroy(sdrg_fft *h) {
  if (!h) return SDRG_OK;
  cudaSetDevice(h->device); cudaDeviceSynchronize();
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h->plan;
  cudaFree(h->d_in); cudaFree(h->d_out);
  delete h;
  return SDRG_OK;
}
int sdrg_fft_exec_dev(sdrg_fft *h, const void *d_in, void *d_out, size_t batch, void *stream) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  SDRG_CUDA(cudaSetDevice(h->device));
  return h->plan->exec(d_in, d_out, batch, h->inverse, (cudaStream_t)stream);
}
int sdrg_fft_exec(sdrg_fft *h, const void *in, void *out, size_t batch) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (!batch) return SDRG_OK;
  SDRG_CUDA(cudaSetDevice(h->device));
  int rc = own_stream(&h->stream);
  if (rc) return rc;
  const size_t bytes = batch * h->n * 2 * sizeof(float);
  if (h->cap < bytes) {
    if (h->d_in) { cudaFree(h->d_in); cudaFree(h->d_out); h->d_in = h->d_out = nullptr; }
    SDRG_CUDA(cudaMalloc(&h->d_in, bytes)); SDRG_CUDA(cudaMalloc(&h->d_out, bytes)); h->cap = bytes;
  }
  SDRG_CUDA(cudaMemcpyAsync(h->d_in, in, bytes, cudaMemcpyHostToDevice, h->stream));
  rc = sdrg_fft_exec_dev(h, h->d_in, h->d_out, batch, h->stream);
  if (rc) return rc;
  SDRG_CUDA(cudaMemcpyAsync(out, h->d_out, bytes, cudaMemcpyDeviceToHost, h->stream));
  SDRG_CUDA(cudaStreamSynchronize(h->stream));
  return SDRG_OK;
}

// ---- FFTPlan<double> ------------------------------------------------------------------------------
struct sdrg_fft64_impl { int device; int inverse; Fft64 plan; cudaStream_t stream; void *d_in, *d_out; size_t cap; };
int sdrg_fft64_create(size_t n, int direction, sdrg_fft64 **out) {
  if (!out) return set_error(SDRG_ERR_ARG, "null argument");
  *out = nullptr;
  if (n == 0) return set_error(SDRG_ERR_CONFIG, "Can not construct FFT plan: Buffer is empty!");      // fftplan_fftw3.hh:27-31
  sdrg_fft64_impl *h = new sdrg_fft64_impl();
  h->device = 0; cudaGetDevice(&h->device);
  h->inverse = direction ? 1 : 0; h->stream = nullptr; h->d_in = h->d_out = nullptr; h->cap = 0;
  const int rc = h->plan.init(n);
  if (rc) { delete h; return rc; }
  *out = (sdrg_fft64 *)h;
  return SDRG_OK;
}
int sdrg_fft64_destroy(sdrg_fft64 *hh) {
  sdrg_fft64_impl *h = (sdrg_fft64_impl *)hh;
  if (!h) return SDRG_OK;
  cudaSetDevice(h->device); cudaDeviceSynchronize();
  if (h->stream) cudaStreamDestroy(h->stream);
  cudaFree(h->d_in); cudaFree(h->d_out);
  delete h;
  return SDRG_OK;
}
int sdrg_fft64_exec_dev(sdrg_fft64 *hh, const void *d_in, void *d_out, size_t batch, void *stream) {
  sdrg_fft64_impl *h = (sdrg_fft64_impl *)hh;
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  SDRG_CUDA(cudaSetDevice(h->device));
  return h->plan.exec(d_in, d_out, batch, h->inverse, (cudaStream_t)stream);
}
int sdrg_fft64_exec(sdrg_fft64 *hh, const void *in, void *out, size_t batch) {
  sdrg_fft64_impl *h = (sdrg_fft64_impl *)hh;
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (!batch) return SDRG_OK;
  SDRG_CUDA(cudaSetDevice(h->device));
  int rc = own_stream(&h->stream);
  if (rc) return rc;
  const size_t bytes = batch * h->plan.n * 2 * sizeof(double);
  if (h->cap < bytes) {
    if (h->d_in) { cudaFree(h->d_in); cudaFree(h->d_out); h->d_in = h->d_out = nullptr; }
    SDRG_CUDA(cudaMalloc(&h->d_in, bytes)); SDRG_CUDA(cudaMalloc(&h->d_out, bytes)); h->cap = bytes;
  }
  SDRG_CUDA(cudaMemcpyAsync(h->d_in, in, bytes, cudaMemcpyHostToDevice, h->stream));
  rc = sdrg_fft64_exec_dev(hh, h->d_in, h->d_out, batch, h->stream);
  if (rc) return rc;
  SDRG_CUDA(cudaMemcpyAsync(out, h->d_out, bytes, cudaMemcpyDeviceToHost, h->stream));
  SDRG_CUDA(cudaStreamSynchronize(h->stream));
  return SDRG_OK;
}

// ---- FilterNode -------------------------------------------------------------------------------------
int sdrg_filter_create(size_t block_size, sdrg_filter **out) {
  if (!out) return set_error(SDRG_ERR_ARG, "null argument");
  *out = nullptr;
  if (block_size < 1 || block_size > ((size_t)1 << 22))
    return set_error(SDRG_ERR_CONFIG, "FilterNode: block size %zu is not supported on the device (1..%d)", block_size, 1 << 22);
  sdrg_filter *h = new sdrg_filter();
  int dev = 0; cudaGetDevice(&dev);
  h->device = dev; h->block = block_size; h->log2n = ilog2(2 * block_size);
  if (!pow2(block_size) || 2 * block_size > ((size_t)1 << kFftMaxLog2)) {      // not a fused-kernel size
    h->gen = new GeneralOla();
    const int rc = h->gen->init(block_size);
    if (rc) { delete h->gen; delete h; return rc; }
  }
  *out = h;
  return SDRG_OK;
}
int sdrg_filter_destroy(sdrg_filter *h) {
  if (!h) return SDRG_OK;
  cudaSetDevice(h->device); cudaDeviceSynchronize();
  if (h->stream) cudaStreamDestroy(h->stream);
  cudaFree(h->d_tw); cudaFree(h->d_kern); cudaFree(h->d_kperm); cudaFree(h->d_tab8k); cudaFree(h->d_hist[0]); cudaFree(h->d_hist[1]);
  cudaFree(h->d_pend); cudaFree(h->d_stage); cudaFree(h->d_spec); cudaFree(h->d_in); cudaFree(h->d_out);
  delete h->gen;
  delete h;
  return SDRG_OK;
}
int sdrg_filter_add(sdrg_filter *h, double fmin, double fmax, size_t *index) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (fmax < fmin) std::swap(fmin, fmax);                       // FilterNode::addFilter, filternode.hh:264
  FilterBand b; b.fmin = fmin; b.fmax = fmax;
  h->bands.push_back(b);
  if (index) *index = h->bands.size() - 1;
  if (h->configured) return design_band(h, h->bands.back());
  h->kern_dirty = true;
  return SDRG_OK;
}
int sdrg_filter_set_freq(sdrg_filter *h, size_t index, double fmin, double fmax) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (index >= h->bands.size()) return set_error(SDRG_ERR_ARG, "FilterNode: no filter %zu", index);
  h->bands[index].fmin = fmin; h->bands[index].fmax = fmax;     // FilterSource::setFreq, filternode.hh:128-130
  if (h->configured) return design_band(h, h->bands[index]);
  return SDRG_OK;
}
int sdrg_filter_count(const sdrg_filter *h, size_t *n) {
  if (!h || !n) return set_error(SDRG_ERR_ARG, "null argument");
  *n = h->bands.size();
  return SDRG_OK;
}
int sdrg_filter_configure(sdrg_filter *h, const sdrg_config *src, sdrg_config *out) {
  if (!h || !src) return set_error(SDRG_ERR_ARG, "null argument");
  if (out) { out->type = SDRG_T_UNDEFINED; out->sample_rate = 0; out->buffer_size = 0; out->num_buffers = 0; }
  if (src->type == SDRG_T_UNDEFINED || src->sample_rate == 0 || src->buffer_size == 0) return SDRG_OK;   // filternode.hh:58-60
  if (src->type != SDRG_T_CF32)
    return set_error(SDRG_ERR_CONFIG, "Can not configure filter-sink: Invalid type %s (%d), expected %s (%d)",
                     type_name(src->type), src->type, type_name(SDRG_T_CF32), SDRG_T_CF32);
  SDRG_CUDA(cudaSetDevice(h->device));
  SDRG_CUDA(cudaDeviceSynchronize());
  h->Fs = src->sample_rate;
  for (size_t f = 0; f < h->bands.size(); ++f) design_band(h, h->bands[f]);
  if (!h->d_tw && !h->gen) { int rc = upload_twiddles(2 * h->block, &h->d_tw); if (rc) return rc; }
  const size_t hb = h->block * 2 * sizeof(float);
  const size_t hist_b = (h->gen ? h->gen->M - h->block : h->block) * 2 * sizeof(float);   // general path: M - B samples of history
  for (int k = 0; k < 2; ++k) {
    if (!h->d_hist[k]) SDRG_CUDA(cudaMalloc(&h->d_hist[k], hist_b));
    SDRG_CUDA(cudaMemset(h->d_hist[k], 0, hist_b));             // _last_trafo zeroed, filternode.hh:117-119
  }
  if (!h->d_pend) SDRG_CUDA(cudaMalloc(&h->d_pend, hb));
  h->pending = 0; h->parity = 0;
  h->configured = true;
  if (out) { out->type = SDRG_T_CF32; out->sample_rate = src->sample_rate; out->buffer_size = h->block; out->num_buffers = src->num_buffers; }
  return SDRG_OK;
}
int sdrg_filter_get_design(const sdrg_filter *h, size_t index, void *kern_2n, void *taps_n) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (index >= h->bands.size() || h->bands[index].taps.empty()) return set_error(SDRG_ERR_RUNTIME, "FilterNode: filter %zu not designed yet", index);
  if (kern_2n && h->bands[index].kern.empty())
    return set_error(SDRG_ERR_RUNTIME, "FilterNode: the 2N-point spectrum is not formed for block sizes that are neither a power of two nor <= 8192");
  if (kern_2n) memcpy(kern_2n, h->bands[index].kern.data(), h->bands[index].kern.size() * sizeof(float));
  if (taps_n) memcpy(taps_n, h->bands[index].taps.data(), h->block * 2 * sizeof(float));
  return SDRG_OK;
}
int sdrg_filter_outputs_for(const sdrg_filter *h, size_t n_in, size_t *n_out) {
  if (!h || !n_out) return set_error(SDRG_ERR_ARG, "null argument");
  *n_out = ((h->pending + n_in) / h->block) * h->block;
  return SDRG_OK;
}

// n_in complex samples in; every filter f gets the completed blocks at d_out + f*out_stride.
// Input that does not fill a block waits for the next call (BufferNode, src/buffernode.hh:61-91).
int sdrg_filter_process_dev(sdrg_filter *h, const void *d_in, size_t n_in, void *d_out, size_t out_stride,
                            size_t *n_out, void *stream) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (!h->configured) return set_error(SDRG_ERR_RUNTIME, "FilterNode: process() before config()");
  if (n_out) *n_out = 0;
  SDRG_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  int rc = upload_kernels(h);
  if (rc) return rc;
  const size_t N = h->block, sb = 2 * sizeof(float);
  const size_t total = h->pending + n_in, nblk = total / N, rem = total - nblk * N;
  if (nblk * N > out_stride && h->bands.size() > 1) return set_error(SDRG_ERR_ARG, "FilterNode: out_stride smaller than the output");
  const char *src = (const char *)d_in;
  if (h->pending) {             // stitch the waiting samples in front of the new ones
    rc = grow_dev(&h->d_stage, &h->stage_cap, (nblk ? nblk * N : 1) * sb);
    if (rc) return rc;
    if (nblk) {
      SDRG_CUDA(cudaMemcpyAsync(h->d_stage, h->d_pend, h->pending * sb, cudaMemcpyDeviceToDevice, st));
      SDRG_CUDA(cudaMemcpyAsync((char *)h->d_stage + h->pending * sb, d_in, (nblk * N - h->pending) * sb, cudaMemcpyDeviceToDevice, st));
      src = (const char *)h->d_stage;
    }
  }
  if (nblk && h->gen) {
    rc = h->gen->run(src, nblk, h->d_hist[h->parity], h->d_hist[h->parity ^ 1], h->d_kern, (int)h->bands.size(), d_out, out_stride, st);
    if (rc) return rc;
    h->parity ^= 1;
  } else if (nblk) {
    FilterArgs a{};
    a.x = src; a.hist_in = h->d_hist[h->parity]; a.hist_out = h->d_hist[h->parity ^ 1];
    a.kern = h->d_kern; a.out = d_out; a.out_stride = out_stride; a.tw = h->d_tw;
    a.block = (int)N; a.log2n = h->log2n; a.n_filters = (int)h->bands.size();
    a.spec = nullptr; a.kperm = h->d_kperm; a.tab8k = h->d_tab8k;
    size_t spec_bytes = nblk * 2 * N * sb;
    if (a.n_filters > 1 && 2 * N == 8192 && a.kperm) {      // one 64 KB line per CTA
      int grid = 0;
      rc = conv8k_grid(nblk, &grid);
      if (rc) return rc;
      spec_bytes = (size_t)grid * 8192 * sb;
    }
    if (a.n_filters > 1 && 2 * N >= 512 && spec_bytes <= ((size_t)2 << 30)) {
      rc = grow_dev(&h->d_spec, &h->spec_cap, spec_bytes);
      if (rc) return rc;
      a.spec = h->d_spec;
    }
    rc = launch_filter_ola(a, nblk, st);
    if (rc) return rc;
    h->parity ^= 1;
  }
  // keep what does not fill a block
  if (rem) {
    if (nblk || !h->pending) {
      const size_t consumed_new = nblk * N - (nblk ? h->pending : 0);
      SDRG_CUDA(cudaMemcpyAsync(h->d_pend, (const char *)d_in + (nblk ? consumed_new : 0) * sb, rem * sb, cudaMemcpyDeviceToDevice, st));
    } else {
      SDRG_CUDA(cudaMemcpyAsync((char *)h->d_pend + h->pending * sb, d_in, n_in * sb, cudaMemcpyDeviceToDevice, st));
    }
  }
  h->pending = rem;
  if (n_out) *n_out = nblk * N;
  return SDRG_OK;
}

int sdrg_filter_process(sdrg_filter *h, const void *in, size_t n_in, void *out, size_t out_stride, size_t *n_out) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (!h->configured) return set_error(SDRG_ERR_RUNTIME, "FilterNode: process() before config()");
  SDRG_CUDA(cudaSetDevice(h->device));
  int rc = own_stream(&h->stream);
  if (rc) return rc;
  const size_t sb = 2 * sizeof(float), F = h->bands.size();
  size_t expect = 0;
  sdrg_filter_outputs_for(h, n_in, &expect);
  if ((rc = grow_dev(&h->d_in, &h->in_cap, (n_in ? n_in : 1) * sb))) return rc;
  if ((rc = grow_dev(&h->d_out, &h->out_cap, (F ? F : 1) * (expect ? expect : 1) * sb))) return rc;
  SDRG_CUDA(cudaMemcpyAsync(h->d_in, in, n_in * sb, cudaMemcpyHostToDevice, h->stream));
  size_t got = 0;
  rc = sdrg_filter_process_dev(h, h->d_in, n_in, h->d_out, expect, &got, h->stream);
  if (rc) return rc;
  for (size_t f = 0; f < F && got; ++f)
    SDRG_CUDA(cudaMemcpyAsync((char *)out + f * out_stride * sb, (char *)h->d_out + f * expect * sb, got * sb, cudaMemcpyDeviceToHost, h->stream));
  SDRG_CUDA(cudaStreamSynchronize(h->stream));
  if (n_out) *n_out = got;
  return SDRG_OK;
}

}  // extern "C"

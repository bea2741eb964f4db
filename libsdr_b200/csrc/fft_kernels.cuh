// fft_kernels.cuh -- launch wrappers of the shared-memory FFT and the fused FFT-convolution filter.
#pragma once
#include "common.cuh"

namespace sdrg {

constexpr int kFftMaxLog2 = 13;          // one CTA holds up to 8192 points (3 x 64 KB for the filter)

struct FilterArgs {
  const void *x;          // n_blocks x block complex floats
  const void *hist_in;    // the previous call's last block
  void       *hist_out;
  const void *kern;       // n_filters x 2*block spectra (already divided by their l2 norm)
  void       *out;        // filter f writes block b to out + f*out_stride + b*block
  size_t      out_stride; // in samples
  const void *tw;         // 2*block-th roots of unity, exp(-2 pi i k / (2 block))
  int         block;
  int         log2n;      // log2(2*block)
  int         n_filters;
  void       *spec;       // multi-filter radix-16 path: spectra of the blocks, n_blocks x 2*block (null: fused 3-buffer kernel)
  const void *kperm;      // block 4096 only (fft8k_kernels.cu): the spectra in the kernel's digit-reversed order, pre-scaled by 1/8192
  const void *tab8k;      // ... and its twiddle tables
};

int launch_fft_batch(const void *in, void *out, int n, int log2n, int inverse, size_t batch, const void *tw, cudaStream_t st);
int launch_filter_ola(const FilterArgs &a, size_t n_blocks, cudaStream_t st);

// fft8k_kernels.cu: n = 8192 / 4096 transforms and the block-4096 convolution (in-place radix-16 stages, table twiddles)
}  // namespace sdrg
#include <vector>
namespace sdrg {
void fft8k_tables(std::vector<float> &tab);                           // host: the twiddle tables (interleaved re, im)
void fft8k_permute_kernel(const float *kern_8192, float *kperm_8192); // host: spectrum -> kernel order, x 1/8192
int launch_fft8k(const void *in, void *out, int n, int inverse, size_t batch, const void *tab, cudaStream_t st);
int launch_conv8k(const FilterArgs &a, size_t n_blocks, cudaStream_t st);
int conv8k_grid(size_t n_blocks, int *grid);   // CTAs that launch will use: a filter bank needs 64 KB of FilterArgs::spec per CTA


// fft_general.cu: every other size, composed from the kernels above (see its header comment)
struct Pow2Fft {          // n = 2^L >= 2: shared-memory kernels up to 8192, four-step above (up to 2^26)
  size_t n = 0; int log2n = 0;
  void *d_tw = nullptr, *d_tab8k = nullptr;
  size_t n1 = 0, n2 = 0; Pow2Fft *sub1 = nullptr, *sub2 = nullptr;
  void *d_tw_hi = nullptr, *d_tw_lo = nullptr, *d_s0 = nullptr, *d_s1 = nullptr; size_t cap0 = 0, cap1 = 0;
  ~Pow2Fft();
  int init(size_t n);
  int exec(const void *in, void *out, size_t batch, int inverse, cudaStream_t st);   // in == out allowed
};
struct AnyFft {           // any n >= 1: Pow2Fft directly or through Bluestein's convolution of length M
  size_t n = 0, M = 0; Pow2Fft *p2 = nullptr;
  void *d_chirp = nullptr, *d_ghat = nullptr, *d_a = nullptr; size_t cap_a = 0;
  ~AnyFft();
  int init(size_t n);
  int exec(const void *in, void *out, size_t batch, int inverse, cudaStream_t st);
};
struct GeneralOla {       // FilterNode block B (any), FFT size M = 2^ceil(log2 2B), history M - B samples
  size_t B = 0, M = 0; Pow2Fft *p2 = nullptr;
  void *d_seg = nullptr, *d_work = nullptr; size_t cap_seg = 0, cap_work = 0;
  ~GeneralOla();
  int init(size_t block);
  int run(const void *x, size_t n_blocks, const void *hist_in, void *hist_out, const void *kern_M, int n_filters,
          void *out, size_t out_stride, cudaStream_t st);
};

struct Fft64 {            // FFTPlan<double>: any n <= 2^22, radix-2 global-memory passes (+ Bluestein), double arithmetic
  size_t n = 0, M = 0;
  void *d_tw = nullptr, *d_chirp = nullptr, *d_ghat = nullptr, *d_a = nullptr, *d_b = nullptr; size_t cap_a = 0, cap_b = 0;
  ~Fft64();
  int init(size_t n);
  int exec(const void *in, void *out, size_t batch, int inverse, cudaStream_t st);
  int pow2_inplace(size_t batch, int inverse, cudaStream_t st);
};

}  // namespace sdrg

// common.cuh -- shared declarations of the libsdrg implementation (not part of the public ABI).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <string>

#include "../../include/sdrg.h"

namespace sdrg {

// ---- error plumbing ---------------------------------------------------------------------------
int set_error(int code, const char *fmt, ...);          // stores the thread-local message, returns code
void count_launch(unsigned n = 1);                      // kernel launch counter (sdrg_kernel_launch_count)

#define SDRG_CUDA(expr)                                                                         \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess)                                                                      \
      return ::sdrg::set_error(SDRG_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,                   \
                               cudaGetErrorString(_e), __FILE__, __LINE__);                     \
  } while (0)

#define SDRG_CHECK_LAUNCH(name)                                                                 \
  do {                                                                                          \
    cudaError_t _e = cudaGetLastError();                                                        \
    if (_e != cudaSuccess)                                                                      \
      return ::sdrg::set_error(SDRG_ERR_CUDA, "launch of %s failed: %s", name,                  \
                               cudaGetErrorString(_e));                                         \
    ::sdrg::count_launch();                                                                     \
  } while (0)

// Tuning / diagnostic switches read from the environment exist only in builds made with -DSDRG_EXPERIMENTS
// (python -m libsdr_b200.build with SDRG_EXPERIMENTS=1).  The shipped library always takes the default:
// no environment variable can change what it computes or which kernel it launches.
#ifdef SDRG_EXPERIMENTS
#include <cstdlib>
static inline int env_int(const char *name, int dflt) { const char *e = getenv(name); return e ? atoi(e) : dflt; }
#else
static inline int env_int(const char *, int dflt) { return dflt; }
#endif

// Per-device one-time launch setup.  Function attributes (dynamic shared memory opt-in) and
// occupancy are properties of (kernel, device): cache them per device, not per process.
constexpr int kMaxDevices = 64;
static inline int current_device() { int d = 0; cudaGetDevice(&d); return (d >= 0 && d < kMaxDevices) ? d : 0; }

// ---- scalar helpers ---------------------------------------------------------------------------
static inline size_t scalar_bytes(int scalar) {
  switch (scalar) {
    case SDRG_T_S8: return 1; case SDRG_T_S16: return 2; case SDRG_T_F32: return 4; default: return 0;
  }
}
static inline int complex_type_of(int scalar) {
  switch (scalar) {
    case SDRG_T_S8: return SDRG_T_CS8; case SDRG_T_S16: return SDRG_T_CS16;
    case SDRG_T_F32: return SDRG_T_CF32; default: return SDRG_T_UNDEFINED;
  }
}
const char *type_name(int type);   // sdr::typeName(), src/node.hh:141-158

// ---- IQBaseBand design (host, double precision; design.cc) ------------------------------------
struct IqbbDesign {
  // constructor / setter state (reference members, src/baseband.hh:264-296, src/freqshift.hh:90-104)
  int      scalar = SDRG_T_S16;
  double   freq_shift = 0;           // FreqShiftBase::_freq_shift
  int32_t  Fc = 0, Ff = 0, Fs = 0, width = 0;
  size_t   order = 1, sub_sample = 1;
  double   oFs = 0;
  size_t   source_bs = 0;
  // derived
  size_t   lut_inc = 0;
  bool     negative = false;
  size_t   out_bs = 0;
  double   out_rate = 0;
  int32_t  k_re[1024], k_im[1024];   // 2^14-scaled integer kernel
  double   kd_re[1024], kd_im[1024]; // alpha/norm (float variant)
  int32_t  lut_re[128], lut_im[128]; // integer LUT (2^shift scaled, truncated; int16-wrapped for S8)
  double   lutd_re[128], lutd_im[128];
};
static const size_t kMaxOrder = 1024;
void design_lut(IqbbDesign &d);
void design_kernel(IqbbDesign &d);
void design_lut_increment(IqbbDesign &d, double nco_Fs);
void design_kernel_real(IqbbDesign &d, double Ff, double width, double Fs);   // BaseBand<int16_t>, 2^16 scaled
// folded float path, in double and rounded to float: A(a), 128 complex entries (1 when !nco, conjugated when neg),
// and U(r, e) = sum_{j=0}^{L-1-e} B(r, j) k[L-1-e-j] for e < n_e, 256 rows of n_e complex entries (design.cc)
void fold_table_a(const IqbbDesign &d, bool nco, bool neg, float *A);
void fold_table_u(const IqbbDesign &d, size_t n_e, float *U);

// Window grid in closed form (SURVEY.md 8 a1).  With c = samples consumed since config(), global
// sample n carries the window counter q(n) = max(n,1)-1 (window 0 holds ss+1 samples because
// _sample_count is incremented after the test, baseband.hh:200,212-217); a window completes at every
// n >= 1 with n % ss == 0.  ss == 1 degenerates to one output per sample (baseband.hh:218-219).
struct WindowAdvance { uint64_t n_out; uint32_t r0; uint32_t first; uint32_t e0; };
static inline uint64_t windows_done(uint64_t c, uint64_t ss) { return ss == 1 ? c : (c ? (c - 1) / ss : 0); }
static inline WindowAdvance window_advance(uint64_t c, uint64_t ss, uint64_t n) {
  WindowAdvance a{};
  a.n_out = windows_done(c + n, ss) - windows_done(c, ss);
  if (ss == 1) { a.r0 = 0; a.first = 0; a.e0 = 0; return a; }
  a.first = c == 0 ? 1u : 0u;
  a.r0 = c ? (uint32_t)((c - 1) % ss) : 0u;
  const uint64_t lo = c ? c : 1;                           // first global index that can complete
  a.e0 = (uint32_t)(((lo + ss - 1) / ss) * ss - c);
  return a;
}

// Real-input BaseBand (src/baseband.hh:425-436): the counter is incremented BEFORE the test, so every
// window holds exactly ss samples and global sample n completes one when (n+1) % ss == 0.
static inline WindowAdvance window_advance_plain(uint64_t c, uint64_t ss, uint64_t n) {
  WindowAdvance a{};
  a.n_out = (c + n) / ss - c / ss;
  a.first = 0;
  a.r0 = (uint32_t)(c % ss);
  a.e0 = (uint32_t)(ss - 1 - c % ss);
  return a;
}

}  // namespace sdrg

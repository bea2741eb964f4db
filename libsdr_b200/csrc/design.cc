// design.cc -- config-time (cold, host, double precision) coefficient design of IQBaseBand and
// FreqShiftBase.  The GPU kernels take these tables as data; they are never recomputed on the
// device because libm/device sin/cos would round differently and the integer paths must be
// bit-exact.  The arithmetic below follows, operation by operation, the expressions in
//   src/baseband.hh:239-262  (IQBaseBand::_update_filter_kernel)
//   src/freqshift.hh:26-36   (FreqShiftBase ctor: LUT)
//   src/freqshift.hh:78-87   (FreqShiftBase::_update_lut_incr)
// so that truncation to int32 lands on the same integers (checked against the reference's own
// tables: tests/test_abi_and_design.py on the golden vectors, tests/test_oracle_vs_live_reference.py on random
// parameter sets against the live reference harness).
#include "common.cuh"

#include <cmath>
#include <complex>
#include <vector>

namespace sdrg {

static inline int trait_shift(int scalar) {      // Traits<Scalar>::shift, src/traits.cc:11-29
  return scalar == SDRG_T_S16 ? 16 : (scalar == SDRG_T_S8 ? 8 : 0);
}

void design_lut(IqbbDesign &d) {
  const double gain = double(1 << trait_shift(d.scalar));
  for (size_t j = 0; j < 128; ++j) {
    const std::complex<double> e = std::exp(std::complex<double>(0, -(2 * M_PI * j) / 128));
    const std::complex<double> v = gain * e;
    d.lutd_re[j] = v.real();
    d.lutd_im[j] = v.imag();
    if (d.scalar == SDRG_T_S8) {           // LUT element type is complex<int16_t> for int8 input
      d.lut_re[j] = int16_t(v.real());
      d.lut_im[j] = int16_t(v.imag());
    } else {
      d.lut_re[j] = int32_t(v.real());
      d.lut_im[j] = int32_t(v.imag());
    }
  }
}

void design_lut_increment(IqbbDesign &d, double nco_Fs) {
  d.negative = (0 > d.freq_shift);
  if (nco_Fs == 0) { d.lut_inc = 0; return; }
  const size_t lut_size = 128;
  d.lut_inc = size_t((lut_size * (1 << 8) * std::abs(d.freq_shift)) / nco_Fs);
}

void design_kernel(IqbbDesign &d) {
  const size_t L = d.order;
  std::complex<double> a[kMaxOrder];
  const double w = (M_PI * d.width) / (d.Fs);
  const double M = double(L) / 2.;
  double norm = 0;
  for (size_t i = 0; i < L; ++i) {
    if (L == 2 * i) a[i] = 4 * (w / M_PI);
    else a[i] = std::sin(w * (i - M)) / (w * (i - M));
    a[i] *= std::exp(std::complex<double>(0.0, (-2 * M_PI * d.Ff * i) / d.Fs));
    a[i] *= (0.42 - 0.5 * cos((2 * M_PI * i) / L) + 0.08 * cos((4 * M_PI * i) / L));
    norm += std::abs(a[i]);
  }
  for (size_t i = 0; i < L; ++i) {
    const std::complex<double> q = (double(1 << 14) * a[i]) / norm;
    d.k_re[i] = int32_t(q.real());
    d.k_im[i] = int32_t(q.imag());
    d.kd_re[i] = a[i].real() / norm;
    d.kd_im[i] = a[i].imag() / norm;
  }
}

// Tables of the folded float path (iqbb_fold_kernels.cu): the 15-bit NCO phase phi = 256 a + r factorises the LUT
// value at phi + d*inc into A(a) B(r, d).
void fold_table_a(const IqbbDesign &d, bool nco, bool neg, float *A) {
  for (size_t a = 0; a < 128; ++a) {
    A[2 * a] = nco ? (float)d.lutd_re[a] : 1.0f;
    A[2 * a + 1] = nco ? (float)(neg ? -d.lutd_im[a] : d.lutd_im[a]) : 0.0f;
  }
}

void fold_table_u(const IqbbDesign &d, size_t n_e, float *U) {
  const size_t L = d.order;
  const bool nco = d.lut_inc != 0, neg = d.negative;
  const uint64_t inc = d.lut_inc & 0x7fffu;
  std::vector<double> br(L), bi(L);
  for (size_t r = 0; r < 256; ++r) {
    for (size_t j = 0; j < L; ++j) {           // B(r, j)
      if (!nco) { br[j] = 1.0; bi[j] = 0.0; continue; }
      const uint64_t s = (r + j * inc) >> 8;
      const size_t idx = neg ? (size_t)((127 + 128 - (s % 128)) % 128) : (size_t)(s % 128);
      br[j] = d.lutd_re[idx]; bi[j] = d.lutd_im[idx];
    }
    for (size_t e = 0; e < n_e; ++e) {
      double sr = 0, si = 0;
      for (size_t j = 0; j + e < L; ++j) {
        const double kr = d.kd_re[L - 1 - e - j], ki = d.kd_im[L - 1 - e - j];
        sr += br[j] * kr - bi[j] * ki;
        si += br[j] * ki + bi[j] * kr;
      }
      U[2 * (r * n_e + e)] = (float)sr; U[2 * (r * n_e + e) + 1] = (float)si;
    }
  }
}

// BaseBand<Scalar>::_update_filter_kernel (src/baseband.hh:462-487): centre tap 1, exp(+j..) shift,
// Blackman window over (i+1)/(order+2), gain 2^Traits<Scalar>::shift; Ff, width and Fs are doubles here.
void design_kernel_real(IqbbDesign &d, double Ff, double width, double Fs) {
  const size_t L = d.order;
  std::complex<double> a[kMaxOrder];
  const double w = (2 * M_PI * width) / (2 * Fs);
  const double M = double(L) / 2;
  double norm = 0;
  for (size_t i = 0; i < L; ++i) {
    if (L == 2 * i) a[i] = 1;
    else a[i] = std::sin(w * (i - M)) / (w * (i - M));
  }
  for (size_t i = 0; i < L; ++i) {
    a[i] = a[i] * std::exp(std::complex<double>(0, (2 * M_PI * Ff * i) / Fs));
    a[i] *= (0.42 - 0.5 * cos((2 * M_PI * (i + 1)) / (L + 2)) + 0.08 * cos((4 * M_PI * (i + 1)) / (L + 2)));
    norm += std::abs(a[i]);
  }
  for (size_t i = 0; i < L; ++i) {
    const std::complex<double> q = (double(1 << trait_shift(d.scalar)) * a[i]) / norm;
    d.k_re[i] = int32_t(q.real());
    d.k_im[i] = int32_t(q.imag());
    d.kd_re[i] = a[i].real() / norm;
    d.kd_im[i] = a[i].imag() / norm;
  }
}

const char *type_name(int type) {
  static const char *names[] = {"UNDEFINED", "uint8", "int8", "uint16", "int16", "float", "double",
                                "complex uint8", "complex int8", "complex uint16", "complex int16",
                                "complex float", "complex double"};
  return (type >= 0 && type <= SDRG_T_CF64) ? names[type] : "unknown";
}

}  // namespace sdrg

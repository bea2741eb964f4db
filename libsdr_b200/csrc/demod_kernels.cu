// demod_kernels.cu -- stand-alone FMDemod / AMDemod / USBDemod kernels (one buffer per launch).
// Reference semantics: src/demod.hh:65-81 (AM), 156-161 (USB), 242-254 (FM), src/math.hh:12-40.
// These are HBM-streaming elementwise kernels: 4 (2, 8) bytes in and 2 (1, 4) bytes out per
// sample, one sample per thread-iteration, grid-stride, coalesced.
#include "iqbb_kernels.cuh"
#include "launch.cuh"
#include "demod_math.cuh"

namespace sdrg {
namespace {

template <int SCALAR> struct In;
template <> struct In<SDRG_T_S16> {
  typedef short2 T; typedef short Fm; typedef short Au; typedef int Last;
  static __device__ __forceinline__ int2 get(const T v) { return make_int2(v.x, v.y); }
  static __device__ __forceinline__ Last phi(int2 v) { return fm_phi_int(v.x, v.y); }
  static __device__ __forceinline__ Fm fm(Last l, Last p) { return (short)(l - p); }
  static __device__ __forceinline__ Fm first(int2 v) { return (short)v.x; }
  static __device__ __forceinline__ Au am(int2 v) { return (short)am_int(v.x, v.y); }
  static __device__ __forceinline__ Au usb(int2 v) { return (short)usb_int(v.x, v.y); }
};
template <> struct In<SDRG_T_S8> {
  typedef char2 T; typedef short Fm; typedef signed char Au; typedef int Last;
  static __device__ __forceinline__ int2 get(const T v) { return make_int2(v.x, v.y); }
  static __device__ __forceinline__ Last phi(int2 v) { return fm_phi_int(v.x, v.y); }
  static __device__ __forceinline__ Fm fm(Last l, Last p) { return (short)(l - p); }
  static __device__ __forceinline__ Fm first(int2 v) {
    return (short)(((uint32_t)(uint8_t)v.x) | (((uint32_t)(uint8_t)v.y) << 8));
  }
  static __device__ __forceinline__ Au am(int2 v) { return (signed char)am_int(v.x, v.y); }
  static __device__ __forceinline__ Au usb(int2 v) { return (signed char)usb_int(v.x, v.y); }
};
template <> struct In<SDRG_T_F32> {
  typedef float2 T; typedef float Fm; typedef float Au; typedef double Last;
  static __device__ __forceinline__ float2 get(const T v) { return v; }
  static __device__ __forceinline__ Last phi(float2 v) { return fm_phi_f64((double)v.x, (double)v.y); }
  static __device__ __forceinline__ Fm fm(Last l, Last p) { return (float)(l - p); }
  static __device__ __forceinline__ Fm first(float2 v) { return v.x; }
  static __device__ __forceinline__ Au am(float2 v) { return sqrtf(v.x * v.x + v.y * v.y); }
  static __device__ __forceinline__ Au usb(float2 v) { return (v.x + v.y) / 2; }
};

// out[i] = phi(in[i-1]) - phi(in[i]) for i >= 2, out[1] = last - phi(in[1]); element 0 skipped.
template <int SCALAR>
__global__ void __launch_bounds__(256) fmdemod_kernel(const typename In<SCALAR>::T *in, size_t n,
                                                       typename In<SCALAR>::Fm *out,
                                                       const typename In<SCALAR>::Last *last_in,
                                                       typename In<SCALAR>::Last *last_out, int in_place) {
  typedef In<SCALAR> I;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const auto v = I::get(in[i]);
    if (i == 0) {
      if (in_place) out[0] = I::first(v);
      if (n == 1) *last_out = *last_in;
      continue;
    }
    const typename I::Last p = I::phi(v);
    const typename I::Last l = (i == 1) ? *last_in : I::phi(I::get(in[i - 1]));
    out[i] = I::fm(l, p);
    if (i == n - 1) *last_out = p;
  }
}

template <int SCALAR, bool USB>
__global__ void __launch_bounds__(256) envelope_kernel(const typename In<SCALAR>::T *in, size_t n,
                                                        typename In<SCALAR>::Au *out) {
  typedef In<SCALAR> I;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const auto v = I::get(in[i]);
    out[i] = USB ? I::usb(v) : I::am(v);
  }
}

// FMDeemph<int16_t> (src/demod.hh:345-352): a 1-pole integer IIR with rounding -- serial and not
// associative within a stream, so one thread walks one stream; banks give the parallelism.
__global__ void __launch_bounds__(128) fmdeemph_kernel(const short *in, short *out, size_t n, size_t streams, size_t stride,
                                                       int alpha, short *avg_state) {
  const size_t s = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= streams) return;
  const short *x = in + s * stride;
  short *y = out + s * stride;
  short avg = avg_state[s];
  const int half = alpha / 2;
  for (size_t i = 0; i < n; ++i) {
    const short diff = (short)(x[i] - avg);
    avg = (short)(avg + ((diff > 0) ? (diff + half) / alpha : (diff - half) / alpha));
    y[i] = avg;
  }
  avg_state[s] = avg;
}

unsigned grid_for(size_t n) {
  size_t g = (n + 255) / 256;
  const size_t cap = 148 * 16;          // 16 resident CTAs of 256 threads per SM, 148 SMs
  return (unsigned)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace

int launch_fmdemod(int scalar, const void *in, size_t n, void *out, const void *last_in, void *last_out,
                   int in_place, cudaStream_t st) {
  if (n == 0) return SDRG_OK;
  const unsigned g = grid_for(n);
  switch (scalar) {
    case SDRG_T_S16:
      fmdemod_kernel<SDRG_T_S16><<<g, 256, 0, st>>>((const short2 *)in, n, (short *)out, (const int *)last_in, (int *)last_out, in_place); break;
    case SDRG_T_S8:
      fmdemod_kernel<SDRG_T_S8><<<g, 256, 0, st>>>((const char2 *)in, n, (short *)out, (const int *)last_in, (int *)last_out, in_place); break;
    case SDRG_T_F32:
      fmdemod_kernel<SDRG_T_F32><<<g, 256, 0, st>>>((const float2 *)in, n, (float *)out, (const double *)last_in, (double *)last_out, in_place); break;
    default: return set_error(SDRG_ERR_ARG, "FMDemod: unsupported scalar %d", scalar);
  }
  SDRG_CHECK_LAUNCH("fmdemod_kernel");
  return SDRG_OK;
}

template <bool USB>
static int launch_envelope(int scalar, const void *in, size_t n, void *out, cudaStream_t st) {
  if (n == 0) return SDRG_OK;
  const unsigned g = grid_for(n);
  switch (scalar) {
    case SDRG_T_S16: envelope_kernel<SDRG_T_S16, USB><<<g, 256, 0, st>>>((const short2 *)in, n, (short *)out); break;
    case SDRG_T_S8: envelope_kernel<SDRG_T_S8, USB><<<g, 256, 0, st>>>((const char2 *)in, n, (signed char *)out); break;
    case SDRG_T_F32: envelope_kernel<SDRG_T_F32, USB><<<g, 256, 0, st>>>((const float2 *)in, n, (float *)out); break;
    default: return set_error(SDRG_ERR_ARG, "demod: unsupported scalar %d", scalar);
  }
  SDRG_CHECK_LAUNCH(USB ? "usbdemod_kernel" : "amdemod_kernel");
  return SDRG_OK;
}

// ---- the whole AutoCast table (src/autocast.hh:30-69; cast functions :120-262) -----------------------------------------
// One input SCALAR per thread-iteration; kinds 1-3 and 8-10 write one scalar, the others a complex value with a zero
// imaginary part.  The arithmetic restates the reference's expressions (their widths, the int8_t* reinterpretation in
// _uint8_int16, the constants (2<<15)-1 and 1<<15); every pair is checked against bytes the reference itself produced
// (tests/golden/cast_table.npz).
template <int KIND>
__global__ void __launch_bounds__(256) autocast_kernel(const void *__restrict__ in, size_t n, void *__restrict__ out) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    int v;
    if (KIND == 1 || KIND == 4 || KIND == 11) v = (int)((const unsigned char *)in)[i];
    else if (KIND == 5 || KIND == 8 || KIND == 9 || KIND == 12) v = (int)((const signed char *)in)[i];
    else if (KIND == 2 || KIND == 10 || KIND == 13) v = (int)((const unsigned short *)in)[i];
    else v = (int)((const short *)in)[i];                                   // 3, 6 (uint16 read as int16), 7, 14
    int r;
    switch (KIND) {
      case 1: case 4: r = v - 127; break;
      case 2: r = (v >> 8) - 127; break;
      case 3: case 7: r = v >> 8; break;
      case 5: case 14: r = v; break;
      case 6: r = (v >> 8) - 65535; break;
      case 8: case 11: r = (int)((unsigned)(v - 127) << 8); break;
      case 9: case 12: r = (int)((unsigned)v << 8); break;
      case 10: r = v - 65535; break;
      default: r = v - 32768; break;                                        // 13
    }
    if (KIND <= 3) ((signed char *)out)[i] = (signed char)r;
    else if (KIND <= 7) ((char2 *)out)[i] = make_char2((signed char)r, 0);
    else if (KIND <= 10) ((short *)out)[i] = (short)r;
    else ((short2 *)out)[i] = make_short2((short)r, 0);
  }
}

int launch_autocast(int kind, const void *in, size_t n_scalars, void *out, cudaStream_t st) {
  if (n_scalars == 0) return SDRG_OK;
  return dispatch(kind, int_range<1, 14>{}, [&](auto K) { return launch("autocast_kernel", autocast_kernel<K>, grid_for(n_scalars), 256, 0, st, in, n_scalars, out); },
                  [&] { return set_error(SDRG_ERR_ARG, "AutoCast: unknown cast kind %d", kind); });
}

int launch_fmdeemph(const void *in, void *out, size_t n, size_t streams, size_t stride, int alpha, void *avg, cudaStream_t st) {
  if (n == 0 || streams == 0) return SDRG_OK;
  fmdeemph_kernel<<<(unsigned)((streams + 127) / 128), 128, 0, st>>>((const short *)in, (short *)out, n, streams, stride, alpha, (short *)avg);
  SDRG_CHECK_LAUNCH("fmdeemph_kernel");
  return SDRG_OK;
}

int launch_amdemod(int scalar, const void *in, size_t n, void *out, cudaStream_t st) {
  return launch_envelope<false>(scalar, in, n, out, st);
}
int launch_usbdemod(int scalar, const void *in, size_t n, void *out, cudaStream_t st) {
  return launch_envelope<true>(scalar, in, n, out, st);
}

}  // namespace sdrg

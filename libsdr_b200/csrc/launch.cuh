// launch.cuh -- how every kernel of the library is set up and launched (launch.cu owns the per-device state).
#pragma once
#include "common.cuh"

#include <utility>

namespace sdrg {

// Prepares kernel `fn` for a launch with `threads` threads and `smem` bytes of dynamic shared memory on the current
// device: above the default (48 KB less the kernel's static shared memory) the kernel's shared-memory opt-in is
// raised to at least `smem`, and never lowered, so host threads that drive one device with different sizes cannot
// undo each other's opt-in.  When `resident` is not null it receives the CTAs of that shape that fit the device at
// once: SMs x CTAs per SM, at least one per SM.  Both are cached per (kernel, device).  Returns SDRG_OK or an error
// set through set_error.
int kernel_setup(const void *fn, int threads, size_t smem, int *resident);

// fn<<<grid, threads, smem, st>>>(args...) after kernel_setup; counts one launch.
template <typename... P, typename... A>
int launch(const char *name, void (*fn)(P...), dim3 grid, int threads, size_t smem, cudaStream_t st, const A &...args) {
  if (smem > 0) {
    const int rc = kernel_setup((const void *)fn, threads, smem, nullptr);
    if (rc) return rc;
  }
  fn<<<grid, threads, smem, st>>>(args...);
  SDRG_CHECK_LAUNCH(name);
  return SDRG_OK;
}

// A persistent grid: min(want, CTAs resident on the device at once).
template <typename... P, typename... A>
int launch_persistent(const char *name, void (*fn)(P...), uint64_t want, int threads, size_t smem, cudaStream_t st, const A &...args) {
  int resident = 0;
  const int rc = kernel_setup((const void *)fn, threads, smem, &resident);
  if (rc) return rc;
  fn<<<(unsigned)(want < (uint64_t)resident ? want : (uint64_t)resident), threads, smem, st>>>(args...);
  SDRG_CHECK_LAUNCH(name);
  return SDRG_OK;
}

// A runtime value as a template argument: f(std::integral_constant<int, V>{}) for the V of Vs equal to v, otherwise().
template <int... Vs, typename F, typename E>
int dispatch(int v, std::integer_sequence<int, Vs...>, F &&f, E &&otherwise) {
  int rc = 0;
  return ((v == Vs && ((rc = f(std::integral_constant<int, Vs>{})), true)) || ...) ? rc : otherwise();
}

template <int First, int Step, int... I>
constexpr std::integer_sequence<int, (First + Step * I)...> shift_seq(std::integer_sequence<int, I...>) { return {}; }
// First, First + Step, ..., Last
template <int First, int Last, int Step = 1>
using int_range = decltype(shift_seq<First, Step>(std::make_integer_sequence<int, (Last - First) / Step + 1>{}));

}  // namespace sdrg

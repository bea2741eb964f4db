// launch.cu -- the per-device launch state of every kernel: shared-memory opt-ins and resident-CTA counts (launch.cuh).
#include "launch.cuh"

#include <map>
#include <mutex>

namespace sdrg {

namespace {
struct KernelState {                                    // one kernel on one device
  size_t opt_in;                                        // dynamic shared memory the kernel may use
  std::map<std::pair<int, size_t>, int> resident;       // (threads, smem) -> CTAs that fit the device at once
};
std::mutex g_setup_mu;                                  // raising the opt-in and recording it are one step
std::map<std::pair<const void *, int>, KernelState> g_setup;
}  // namespace

int kernel_setup(const void *fn, int threads, size_t smem, int *resident) {
  int dev = 0;
  SDRG_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(g_setup_mu);
  auto it = g_setup.find({fn, dev});
  if (it == g_setup.end()) {                            // the default: 48 KB less the kernel's static shared memory
    cudaFuncAttributes fa{};
    SDRG_CUDA(cudaFuncGetAttributes(&fa, fn));
    it = g_setup.emplace(std::make_pair(fn, dev), KernelState{(size_t)fa.maxDynamicSharedSizeBytes, {}}).first;
  }
  KernelState &k = it->second;
  if (smem > k.opt_in) {
    SDRG_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k.opt_in = smem;
  }
  if (!resident) return SDRG_OK;
  int &r = k.resident[{threads, smem}];
  if (!r) {
    int sms = 0, per_sm = 0;
    SDRG_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    SDRG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, threads, smem));
    r = sms * (per_sm > 0 ? per_sm : 1);
  }
  *resident = r;
  return SDRG_OK;
}

}  // namespace sdrg

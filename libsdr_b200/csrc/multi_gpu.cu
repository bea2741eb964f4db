// multi_gpu.cu -- the parts of the C ABI that span more than one GPU (include/sdrg.h, "multi-GPU").
//
// The receive chain has no exchange step: a channel bank shards by contiguous channel ranges, every
// shard reads the whole input stream, and the only data that crosses GPUs is the demodulated output
// (SURVEY.md 8e; the reference itself is single-threaded, src/queue.cc:57-60 is its only thread).
// Two ways to use several GPUs, both built on plain peer memory so that the compute kernels never
// share SMs with a collective:
//   * sdrg_bank_sharded_*: ONE process drives G devices.  The input is broadcast with copy-engine
//     peer copies, every shard's finalize kernel stores its channel rows straight into the output
//     arrays on the primary device (NVLink peer stores), streams are joined with events.
//   * sdrg_peer_*: one process per GPU (torch.distributed / MPI style).  The consumer rank exports a
//     window of its HBM through CUDA IPC; producers map it and pass addresses inside it as the output
//     pointers of sdrg_rxchain_process_dev / sdrg_bank_process_dev, then publish progress with
//     sdrg_peer_signal(); the consumer orders its stream behind them with sdrg_peer_wait().
#include "common.cuh"

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <vector>

#include <sys/mman.h>
#include <sys/syscall.h>
#include <unistd.h>

using namespace sdrg;

namespace {

struct DeviceGuard {   // restores the calling thread's device
  int prev = 0;
  DeviceGuard() { cudaGetDevice(&prev); }
  ~DeviceGuard() { cudaSetDevice(prev); }
};

__global__ void peer_signal_kernel(unsigned long long *slot, unsigned long long value) {
  __threadfence_system();                                   // everything this stream wrote before is visible first
  *(volatile unsigned long long *)slot = value;
  __threadfence_system();
}

// one thread per slot; gives up after timeout_ns and raises *timed_out (host-mapped) instead of hanging
__global__ void peer_wait_kernel(const unsigned long long *slots, unsigned n, unsigned long long value,
                                 unsigned long long timeout_ns, int *timed_out) {
  unsigned long long t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  for (unsigned k = threadIdx.x; k < n; k += blockDim.x) {
    const volatile unsigned long long *p = slots + k;
    unsigned ns = 64;
    while (*p < value) {
      __nanosleep(ns);
      if (ns < 2048) ns <<= 1;
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      if (t - t0 > timeout_ns) { *timed_out = 1; break; }
    }
  }
  __threadfence_system();
}

int *g_timeout_flag_host = nullptr;     // pinned + mapped, one per process (sticky until read)
int ensure_timeout_flag() {
  if (g_timeout_flag_host) return SDRG_OK;
  SDRG_CUDA(cudaHostAlloc((void **)&g_timeout_flag_host, sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable));
  *g_timeout_flag_host = 0;
  return SDRG_OK;
}

size_t elem_bytes(int scalar, int k) {   // k: 0 bb, 1 fm, 2 am, 3 usb
  const size_t s = scalar_bytes(scalar);
  return k == 0 ? 2 * s : (k == 1 ? (scalar == SDRG_T_F32 ? 4 : 2) : s);   // FM: int16, or float for a float bank
}

int grow(void **p, size_t *cap, size_t need) {
  if (*cap >= need && *p) return SDRG_OK;
  if (*p) { SDRG_CUDA(cudaDeviceSynchronize()); SDRG_CUDA(cudaFree(*p)); }
  *p = nullptr; *cap = 0;
  SDRG_CUDA(cudaMalloc(p, need ? need : 16));
  *cap = need;
  return SDRG_OK;
}

// NUMA node of a CUDA device from sysfs (-1: unknown / single node)
int device_numa_node(int device) {
  char bus[32] = "";
  if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device) != cudaSuccess) { cudaGetLastError(); return -1; }
  for (char *c = bus; *c; ++c) if (*c >= 'A' && *c <= 'Z') *c = (char)(*c - 'A' + 'a');
  char path[128];
  snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bus);
  FILE *f = fopen(path, "r");
  if (!f) return -1;
  int node = -1;
  if (fscanf(f, "%d", &node) != 1) node = -1;
  fclose(f);
  return node;
}

struct HostBlock { size_t bytes; bool mapped; };
std::mutex g_host_mu;
std::map<void *, HostBlock> g_host_blocks;

}  // namespace

struct sdrg_bank_sharded {
  struct Shard {
    int device = 0;
    size_t lo = 0, hi = 0;               // channel range
    sdrg_bank *bank = nullptr;
    cudaStream_t st = nullptr;
    cudaEvent_t done = nullptr;
    bool direct = false;                 // its kernels may store into the primary device's memory
    void *d_in = nullptr; size_t in_cap = 0;
    void *d_out[4] = {nullptr, nullptr, nullptr, nullptr}; size_t out_cap[4] = {0, 0, 0, 0};
  };
  int scalar = SDRG_T_S16;
  size_t channels = 0;
  std::vector<Shard> shards;
  cudaEvent_t ev_in = nullptr;           // on the primary device
  bool configured = false;
};

extern "C" {

// ---- peer windows ------------------------------------------------------------------------------------
int sdrg_peer_window_create(size_t bytes, void **d_ptr, void *ipc_handle) {
  if (!d_ptr || !ipc_handle) return set_error(SDRG_ERR_ARG, "null argument");
  *d_ptr = nullptr;
  static_assert(sizeof(cudaIpcMemHandle_t) == SDRG_IPC_HANDLE_BYTES, "IPC handle size");
  void *p = nullptr;
  SDRG_CUDA(cudaMalloc(&p, bytes ? bytes : 16));
  cudaError_t e = cudaMemset(p, 0, bytes ? bytes : 16);
  cudaIpcMemHandle_t hd;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&hd, p);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { cudaFree(p); return set_error(SDRG_ERR_CUDA, "peer window: %s", cudaGetErrorString(e)); }
  memcpy(ipc_handle, &hd, sizeof(hd));
  *d_ptr = p;
  return SDRG_OK;
}
int sdrg_peer_window_open(const void *ipc_handle, void **d_ptr) {
  if (!d_ptr || !ipc_handle) return set_error(SDRG_ERR_ARG, "null argument");
  *d_ptr = nullptr;
  cudaIpcMemHandle_t hd;
  memcpy(&hd, ipc_handle, sizeof(hd));
  SDRG_CUDA(cudaIpcOpenMemHandle(d_ptr, hd, cudaIpcMemLazyEnablePeerAccess));
  return SDRG_OK;
}
int sdrg_peer_window_close(void *d_ptr) {
  if (d_ptr) SDRG_CUDA(cudaIpcCloseMemHandle(d_ptr));
  return SDRG_OK;
}
int sdrg_peer_window_destroy(void *d_ptr) {
  if (d_ptr) { SDRG_CUDA(cudaDeviceSynchronize()); SDRG_CUDA(cudaFree(d_ptr)); }
  return SDRG_OK;
}
int sdrg_peer_signal(void *d_slot, uint64_t value, void *stream) {
  if (!d_slot) return set_error(SDRG_ERR_ARG, "null argument");
  peer_signal_kernel<<<1, 1, 0, (cudaStream_t)stream>>>((unsigned long long *)d_slot, (unsigned long long)value);
  SDRG_CHECK_LAUNCH("peer_signal_kernel");
  return SDRG_OK;
}
int sdrg_peer_wait(const void *d_slots, size_t n_slots, uint64_t value, unsigned timeout_ms, void *stream) {
  if (!d_slots) return set_error(SDRG_ERR_ARG, "null argument");
  if (!n_slots) return SDRG_OK;
  int rc = ensure_timeout_flag();
  if (rc) return rc;
  int *d_flag = nullptr;
  SDRG_CUDA(cudaHostGetDevicePointer((void **)&d_flag, g_timeout_flag_host, 0));
  const unsigned threads = (unsigned)std::min<size_t>(n_slots, 64);
  peer_wait_kernel<<<1, threads, 0, (cudaStream_t)stream>>>((const unsigned long long *)d_slots, (unsigned)n_slots,
                                                           (unsigned long long)value,
                                                           (unsigned long long)(timeout_ms ? timeout_ms : 10000u) * 1000000ull, d_flag);
  SDRG_CHECK_LAUNCH("peer_wait_kernel");
  return SDRG_OK;
}
int sdrg_peer_wait_timed_out(int *timed_out) {
  if (!timed_out) return set_error(SDRG_ERR_ARG, "null argument");
  *timed_out = g_timeout_flag_host ? *(volatile int *)g_timeout_flag_host : 0;
  if (g_timeout_flag_host) *g_timeout_flag_host = 0;
  return SDRG_OK;
}
int sdrg_memcpy_d2d_async(void *d_dst, const void *d_src, size_t bytes, void *stream) {
  if (bytes) SDRG_CUDA(cudaMemcpyAsync(d_dst, d_src, bytes, cudaMemcpyDefault, (cudaStream_t)stream));
  return SDRG_OK;
}

// ---- pinned host memory next to a GPU --------------------------------------------------------------------
// Pages are bound (mbind, MPOL_BIND) to the NUMA node the device hangs off, touched, then registered with
// CUDA; on a single-node host, or when the node is unknown, this is cudaHostAlloc.
int sdrg_host_alloc(size_t bytes, int device, void **host_ptr, int *numa_node) {
  if (!host_ptr) return set_error(SDRG_ERR_ARG, "null argument");
  *host_ptr = nullptr;
  const int node = device_numa_node(device);
  if (numa_node) *numa_node = node;
  if (!bytes) bytes = 1;
  void *p = nullptr;
  bool mapped = false;
#ifdef SYS_mbind
  if (node >= 0 && node < 1024) {
    const size_t page = (size_t)sysconf(_SC_PAGESIZE);
    const size_t len = (bytes + page - 1) / page * page;
    void *m = mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (m != MAP_FAILED) {
      unsigned long mask[16] = {0};
      mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
      const long r = syscall(SYS_mbind, m, len, 2 /* MPOL_BIND */, mask, (unsigned long)(8 * sizeof(mask)), 0ul);
      if (r == 0) {
        for (size_t o = 0; o < len; o += page) ((volatile char *)m)[o] = 0;     // fault the pages in on that node
        if (cudaHostRegister(m, len, cudaHostRegisterPortable) == cudaSuccess) { p = m; mapped = true; bytes = len; }
        else cudaGetLastError();
      }
      if (!mapped) munmap(m, len);
    }
  }
#endif
  if (!p) SDRG_CUDA(cudaHostAlloc(&p, bytes, cudaHostAllocPortable));
  std::lock_guard<std::mutex> lk(g_host_mu);
  g_host_blocks[p] = HostBlock{bytes, mapped};
  *host_ptr = p;
  return SDRG_OK;
}
int sdrg_host_free(void *host_ptr) {
  if (!host_ptr) return SDRG_OK;
  HostBlock b;
  {
    std::lock_guard<std::mutex> lk(g_host_mu);
    auto it = g_host_blocks.find(host_ptr);
    if (it == g_host_blocks.end()) return set_error(SDRG_ERR_ARG, "sdrg_host_free: %p was not returned by sdrg_host_alloc", host_ptr);
    b = it->second;
    g_host_blocks.erase(it);
  }
  if (b.mapped) { cudaHostUnregister(host_ptr); munmap(host_ptr, b.bytes); }
  else cudaFreeHost(host_ptr);
  return SDRG_OK;
}

// ---- channel bank sharded over the devices of one process ---------------------------------------------
int sdrg_bank_sharded_create(int scalar, size_t n_channels, const double *Fc, const double *Ff, double width, size_t order,
                             size_t sub_sample, double oFs, const int *devices, size_t n_devices, sdrg_bank_sharded **out) {
  if (!out || !Fc || !devices) return set_error(SDRG_ERR_ARG, "null argument");
  *out = nullptr;
  if (n_devices == 0) return set_error(SDRG_ERR_ARG, "sharded bank: no devices");
  if (n_channels < n_devices) return set_error(SDRG_ERR_ARG, "sharded bank: %zu channels on %zu devices", n_channels, n_devices);
  int count = 0;
  SDRG_CUDA(cudaGetDeviceCount(&count));
  for (size_t g = 0; g < n_devices; ++g)
    if (devices[g] < 0 || devices[g] >= count) return set_error(SDRG_ERR_ARG, "sharded bank: no device %d (%d visible)", devices[g], count);
  DeviceGuard guard;
  sdrg_bank_sharded *h = new sdrg_bank_sharded();
  h->scalar = scalar; h->channels = n_channels;
  h->shards.resize(n_devices);
  const int primary = devices[0];
  const size_t base = n_channels / n_devices, extra = n_channels % n_devices;
  int rc = SDRG_OK;
  size_t lo = 0;
  for (size_t g = 0; g < n_devices && rc == SDRG_OK; ++g) {
    sdrg_bank_sharded::Shard &s = h->shards[g];
    s.device = devices[g]; s.lo = lo; s.hi = lo + base + (g < extra ? 1 : 0); lo = s.hi;
    cudaError_t e = cudaSetDevice(s.device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s.st, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming);
    if (e != cudaSuccess) { rc = set_error(SDRG_ERR_CUDA, "sharded bank: device %d: %s", s.device, cudaGetErrorString(e)); break; }
    if (s.device == primary) s.direct = true;
    else {
      int can = 0;
      cudaDeviceCanAccessPeer(&can, s.device, primary);
      if (can) {
        e = cudaDeviceEnablePeerAccess(primary, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
        s.direct = e == cudaSuccess;
        if (!s.direct) cudaGetLastError();
      }
    }
    // sdrg_bank_create binds the handle to the thread's current CUDA device
    rc = sdrg_bank_create(scalar, s.hi - s.lo, Fc + s.lo, Ff ? Ff + s.lo : nullptr, width, order, sub_sample, oFs, &s.bank);
  }
  if (rc == SDRG_OK) {
    cudaError_t e = cudaSetDevice(primary);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming);
    if (e != cudaSuccess) rc = set_error(SDRG_ERR_CUDA, "sharded bank: %s", cudaGetErrorString(e));
  }
  if (rc != SDRG_OK) {
    char msg[512];
    strncpy(msg, sdrg_last_error(), sizeof(msg) - 1); msg[sizeof(msg) - 1] = 0;
    sdrg_bank_sharded_destroy(h);
    return set_error(rc, "%s", msg);
  }
  *out = h;
  return SDRG_OK;
}

int sdrg_bank_sharded_destroy(sdrg_bank_sharded *h) {
  if (!h) return SDRG_OK;
  DeviceGuard guard;
  for (auto &s : h->shards) {
    cudaSetDevice(s.device);
    if (s.st) cudaStreamSynchronize(s.st);
    if (s.bank) sdrg_bank_destroy(s.bank);
    if (s.st) cudaStreamDestroy(s.st);
    if (s.done) cudaEventDestroy(s.done);
    if (s.d_in) cudaFree(s.d_in);
    for (int k = 0; k < 4; ++k) if (s.d_out[k]) cudaFree(s.d_out[k]);
  }
  if (h->ev_in) { cudaSetDevice(h->shards[0].device); cudaEventDestroy(h->ev_in); }
  delete h;
  return SDRG_OK;
}

int sdrg_bank_sharded_configure(sdrg_bank_sharded *h, const sdrg_config *src, sdrg_config *out) {
  if (!h || !src) return set_error(SDRG_ERR_ARG, "null argument");
  DeviceGuard guard;
  h->configured = false;
  sdrg_config o{};
  for (auto &s : h->shards) {
    SDRG_CUDA(cudaSetDevice(s.device));
    int rc = sdrg_bank_configure(s.bank, src, &o);
    if (rc) return rc;
  }
  h->configured = o.type != SDRG_T_UNDEFINED;
  if (out) *out = o;
  return SDRG_OK;
}

int sdrg_bank_sharded_info(const sdrg_bank_sharded *h, size_t *channels, size_t *n_shards, size_t shard, int *device,
                           size_t *first_channel, size_t *n_shard_channels, int *direct_peer_stores) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (channels) *channels = h->channels;
  if (n_shards) *n_shards = h->shards.size();
  if (shard >= h->shards.size()) return set_error(SDRG_ERR_ARG, "sharded bank: no shard %zu", shard);
  const auto &s = h->shards[shard];
  if (device) *device = s.device;
  if (first_channel) *first_channel = s.lo;
  if (n_shard_channels) *n_shard_channels = s.hi - s.lo;
  if (direct_peer_stores) *direct_peer_stores = s.direct ? 1 : 0;
  return SDRG_OK;
}

int sdrg_bank_sharded_outputs_for(const sdrg_bank_sharded *h, size_t n_in, size_t *n_out) {
  if (!h || !n_out) return set_error(SDRG_ERR_ARG, "null argument");
  return sdrg_bank_outputs_for(h->shards[0].bank, n_in, n_out);
}

// Input and outputs live on the PRIMARY device (devices[0]); `stream` is a stream of that device.
// Asynchronous: on return everything is enqueued and `stream` is ordered behind all shards.
int sdrg_bank_sharded_process_dev(sdrg_bank_sharded *h, const void *d_in, size_t buffer_size, size_t n_buffers, void *d_bb,
                                  void *d_fm, void *d_am, void *d_usb, size_t out_stride, size_t *n_out, void *stream) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (!h->configured) return set_error(SDRG_ERR_RUNTIME, "bank: process() before config()");
  if (n_out) *n_out = 0;
  if (!buffer_size || !n_buffers) return SDRG_OK;
  DeviceGuard guard;
  const int primary = h->shards[0].device;
  const size_t in_bytes = buffer_size * n_buffers * 2 * scalar_bytes(h->scalar);
  void *outs[4] = {d_bb, d_fm, d_am, d_usb};
  SDRG_CUDA(cudaSetDevice(primary));
  SDRG_CUDA(cudaEventRecord(h->ev_in, (cudaStream_t)stream));
  size_t got = 0;
  for (auto &s : h->shards) {
    SDRG_CUDA(cudaSetDevice(s.device));
    SDRG_CUDA(cudaStreamWaitEvent(s.st, h->ev_in, 0));
    const void *in = d_in;
    if (s.device != primary) {           // broadcast of the input: copy engine, NVLink
      int rc = grow(&s.d_in, &s.in_cap, in_bytes);
      if (rc) return rc;
      SDRG_CUDA(cudaMemcpyPeerAsync(s.d_in, s.device, d_in, primary, in_bytes, s.st));
      in = s.d_in;
    }
    void *dst[4] = {nullptr, nullptr, nullptr, nullptr};
    const size_t rows = s.hi - s.lo;
    for (int k = 0; k < 4; ++k) {
      if (!outs[k]) continue;
      const size_t eb = elem_bytes(h->scalar, k);
      char *final_dst = (char *)outs[k] + s.lo * out_stride * eb;
      if (s.direct) { dst[k] = final_dst; continue; }
      int rc = grow(&s.d_out[k], &s.out_cap[k], rows * out_stride * eb);
      if (rc) return rc;
      dst[k] = s.d_out[k];
      // out-of-place FM leaves element 0 of every buffer untouched: start from the destination's bytes
      if (k == 1) SDRG_CUDA(cudaMemcpyPeerAsync(dst[k], s.device, final_dst, primary, rows * out_stride * eb, s.st));
    }
    int rc = sdrg_bank_process_dev(s.bank, in, buffer_size, n_buffers, dst[0], dst[1], dst[2], dst[3], out_stride, &got, s.st);
    if (rc) return rc;
    if (!s.direct)
      for (int k = 0; k < 4; ++k) {
        if (!outs[k]) continue;
        const size_t eb = elem_bytes(h->scalar, k);
        SDRG_CUDA(cudaMemcpyPeerAsync((char *)outs[k] + s.lo * out_stride * eb, primary, dst[k], s.device, rows * out_stride * eb, s.st));
      }
    SDRG_CUDA(cudaEventRecord(s.done, s.st));
  }
  SDRG_CUDA(cudaSetDevice(primary));
  for (auto &s : h->shards) SDRG_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, s.done, 0));
  if (n_out) *n_out = got;
  return SDRG_OK;
}

// Host pointers: every device uploads the input itself and returns its channel rows to the caller's
// arrays; all devices run concurrently, the call returns when every row is in host memory.
int sdrg_bank_sharded_process(sdrg_bank_sharded *h, const void *in, size_t buffer_size, size_t n_buffers, void *bb, void *fm,
                              void *am, void *usb, size_t out_stride, size_t *n_out) {
  if (!h) return set_error(SDRG_ERR_ARG, "null handle");
  if (!h->configured) return set_error(SDRG_ERR_RUNTIME, "bank: process() before config()");
  if (n_out) *n_out = 0;
  if (!buffer_size || !n_buffers) return SDRG_OK;
  DeviceGuard guard;
  const size_t in_bytes = buffer_size * n_buffers * 2 * scalar_bytes(h->scalar);
  void *host[4] = {bb, fm, am, usb};
  size_t got = 0;
  for (auto &s : h->shards) {
    SDRG_CUDA(cudaSetDevice(s.device));
    int rc = grow(&s.d_in, &s.in_cap, in_bytes);
    if (rc) return rc;
    const size_t rows = s.hi - s.lo;
    void *dst[4] = {nullptr, nullptr, nullptr, nullptr};
    for (int k = 0; k < 4; ++k) {
      if (!host[k]) continue;
      const size_t eb = elem_bytes(h->scalar, k);
      if ((rc = grow(&s.d_out[k], &s.out_cap[k], rows * out_stride * eb))) return rc;
      dst[k] = s.d_out[k];
      if (k == 1) SDRG_CUDA(cudaMemcpyAsync(dst[k], (char *)host[k] + s.lo * out_stride * eb, rows * out_stride * eb, cudaMemcpyHostToDevice, s.st));
    }
    SDRG_CUDA(cudaMemcpyAsync(s.d_in, in, in_bytes, cudaMemcpyHostToDevice, s.st));
    rc = sdrg_bank_process_dev(s.bank, s.d_in, buffer_size, n_buffers, dst[0], dst[1], dst[2], dst[3], out_stride, &got, s.st);
    if (rc) return rc;
    for (int k = 0; k < 4; ++k) {
      if (!host[k]) continue;
      const size_t eb = elem_bytes(h->scalar, k);
      SDRG_CUDA(cudaMemcpyAsync((char *)host[k] + s.lo * out_stride * eb, dst[k], rows * out_stride * eb, cudaMemcpyDeviceToHost, s.st));
    }
  }
  for (auto &s : h->shards) {
    SDRG_CUDA(cudaSetDevice(s.device));
    SDRG_CUDA(cudaStreamSynchronize(s.st));
  }
  if (n_out) *n_out = got;
  return SDRG_OK;
}

}  // extern "C"

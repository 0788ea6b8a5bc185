// Shared plumbing of the sm_100a sources: launch macro, error capture, async-copy helpers.
#pragma once
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <mutex>

#ifdef SGX_EMUL
#include "cuda_emul.h"  // tools/cpu_emul: developer-only CPU single-stepping, never shipped
#else
#include <cuda_runtime.h>
#define SGX_LAUNCH(kernel, grid, block, smem, stream, ...) \
  kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#define SGX_DYN_SMEM(name) extern __shared__ __align__(1024) unsigned char name[]
#endif

#include "../../include/softgnss_b200.h"

// constant tables in headers shared by several translation units: internal linkage
#ifdef SGX_EMUL
#define SGX_TABLE static
#else
#define SGX_TABLE static __constant__
#endif

namespace sgx {

extern char g_err[512];
extern long long g_launches;
extern int g_bound_device;           // the device that owns this process' plan caches and scratch buffers (-1: none yet)
extern std::recursive_mutex g_api_mutex;

inline int fail(int code, const char* what, const char* detail) {
  snprintf(g_err, sizeof(g_err), "%s: %s", what, detail ? detail : "");
  return code;
}

// Every compute entry point of the C ABI holds one of these: the plan caches and scratch buffers (FFT plans, code
// spectra, tracking state, ...) are process-wide and live on ONE device -- the one-process-per-GPU convention of
// bench.py / torch.distributed.  Calls are serialised, and a call made while another device is current fails with
// SGX_ERR_ARG instead of touching memory of the wrong device.
struct ApiGuard {
  std::lock_guard<std::recursive_mutex> lock;
  int rc;
  ApiGuard() : lock(g_api_mutex), rc(0) {
    int d = -1;
    if (cudaGetDevice(&d) != cudaSuccess) { cudaGetLastError(); return; }
    if (g_bound_device < 0) g_bound_device = d;
    else if (d != g_bound_device) {
      char msg[160];
      snprintf(msg, sizeof(msg), "device %d is current, but this process is bound to device %d (one process per GPU)", d,
               g_bound_device);
      rc = fail(SGX_ERR_ARG, "softgnss_b200", msg);
    }
  }
};
#define SGX_API_GUARD()        \
  sgx::ApiGuard api_guard__;   \
  if (api_guard__.rc) return api_guard__.rc

#define SGX_CUDA(call)                                                          \
  do {                                                                          \
    cudaError_t e__ = (call);                                                   \
    if (e__ != cudaSuccess) return sgx::fail(SGX_ERR_CUDA, #call, cudaGetErrorString(e__)); \
  } while (0)

#define SGX_COUNTED_LAUNCH(...)  \
  do {                           \
    SGX_LAUNCH(__VA_ARGS__);     \
    ++sgx::g_launches;           \
  } while (0)

inline bool is_device_ptr(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// Scratch device buffer that only ever grows (plans keep them for the process lifetime).
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int reserve(size_t n) {
    if (n <= cap) return 0;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    if (cudaMalloc(&p, n) != cudaSuccess) return -1;
    cap = n;
    return 0;
  }
  template <class T> T* as() { return (T*)p; }
};

// ---- caller operands of the C-ABI entry points: host or device memory (include/softgnss_b200.h) --------------------
// Device view of `count` elements at p: device memory (and NULL) as it is, host memory copied into buf.
template <class T>
int stage_in(const T* p, size_t count, DevBuf& buf, const T*& dev, cudaStream_t s) {
  dev = p;
  if (!p || is_device_ptr(p)) return SGX_OK;
  if (buf.reserve(sizeof(T) * count)) return fail(SGX_ERR_CUDA, "cudaMalloc", "input staging buffer");
  SGX_CUDA(cudaMemcpyAsync(buf.p, p, sizeof(T) * count, cudaMemcpyHostToDevice, s));
  dev = buf.as<T>();
  return SGX_OK;
}

// Device view of `rows` series of ms elements that start `stride` elements apart.  Device rows are read in place
// (dev_stride = stride); host rows are packed into buf by one 2-D copy that reads those rows and nothing between or
// after them (dev_stride = ms).
template <class T>
int stage_rows_in(const T* p, int64_t stride, int32_t ms, size_t rows, DevBuf& buf, const T*& dev,
                  long long& dev_stride, cudaStream_t s) {
  dev = p;
  dev_stride = stride;
  if (is_device_ptr(p)) return SGX_OK;
  const size_t row = sizeof(T) * (size_t)ms;
  if (buf.reserve(row * rows)) return fail(SGX_ERR_CUDA, "cudaMalloc", "input staging buffer");
  SGX_CUDA(cudaMemcpy2DAsync(buf.p, row, p, sizeof(T) * (size_t)stride, row, rows, cudaMemcpyHostToDevice, s));
  dev = buf.as<T>();
  dev_stride = ms;
  return SGX_OK;
}

// The outputs of one call.  add() gives the kernel a device view of an output: host memory is mapped to scratch,
// device memory and NULL stay as they are.  finish(), after the launch, copies the scratch back and synchronises the
// stream iff an output was staged, so a call whose outputs are all device memory stays asynchronous.
class StagedOutputs {
  struct Copy { void* host; const void* dev; size_t bytes; };
  Copy copies_[8];
  int n_ = 0;

 public:
  template <class T>
  int add(T* p, size_t count, DevBuf& buf, T*& dev) {
    dev = p;
    if (!p || is_device_ptr(p)) return SGX_OK;
    if (n_ == 8) return fail(SGX_ERR_ARG, "StagedOutputs", "more than 8 host outputs");
    if (buf.reserve(sizeof(T) * count)) return fail(SGX_ERR_CUDA, "cudaMalloc", "output staging buffer");
    dev = buf.as<T>();
    copies_[n_++] = {p, dev, sizeof(T) * count};
    return SGX_OK;
  }
  int finish(cudaStream_t s) {
    for (int i = 0; i < n_; ++i)
      SGX_CUDA(cudaMemcpyAsync(copies_[i].host, copies_[i].dev, copies_[i].bytes, cudaMemcpyDeviceToHost, s));
    if (n_) SGX_CUDA(cudaStreamSynchronize(s));
    return SGX_OK;
  }
};

// ---- Ampere-style 16-byte async copy global -> shared (LDGSTS) ------------------------------
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
#ifdef SGX_EMUL
  memcpy(smem_dst, gsrc, 16);
#else
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gsrc) : "memory");
#endif
}
__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gsrc) {
#ifdef SGX_EMUL
  memcpy(smem_dst, gsrc, 8);
#else
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s), "l"(gsrc) : "memory");
#endif
}
__device__ __forceinline__ void cp_async_commit() {
#ifndef SGX_EMUL
  asm volatile("cp.async.commit_group;\n" ::: "memory");
#endif
}
__device__ __forceinline__ void cp_async_wait_all() {
#ifndef SGX_EMUL
  asm volatile("cp.async.wait_all;\n" ::: "memory");
#endif
}

// ---- TMA 1-D bulk copy global -> shared completing on an mbarrier (UBLKCP in SASS) ----------
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
#ifdef SGX_EMUL
  *bar = 0;
  (void)count;
#else
  unsigned s = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(s), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
#endif
}
// ---- explicit shared-window loads --------------------------------------------------------------------------
// A 32-bit shared-window address taken once (smem_addr) and used with ld.shared keeps the compiler from
// rematerialising the window base (S2R SR_CgaCtaId + LEA on sm_100) in front of every access inside a hot loop.
// The generic pointer travels along for the CPU emulator build.
__device__ __forceinline__ unsigned smem_addr(const void* p) {
#ifdef SGX_EMUL
  (void)p; return 0u;
#else
  // (made opaque, so the value is kept in its register instead of being recomputed at every use)
  unsigned a = (unsigned)__cvta_generic_to_shared(p), o;
  asm volatile("mov.u32 %0, %1;" : "=r"(o) : "r"(a));
  return o;
#endif
}
__device__ __forceinline__ unsigned lds_u32(const void* base, unsigned base_s, int byte_off) {
#ifdef SGX_EMUL
  (void)base_s; return *reinterpret_cast<const unsigned*>(reinterpret_cast<const char*>(base) + byte_off);
#else
  (void)base; unsigned v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(base_s + (unsigned)byte_off));
  return v;
#endif
}
__device__ __forceinline__ uint2 lds_u32x2(const void* base, unsigned base_s, int byte_off) {   // 8-byte aligned
#ifdef SGX_EMUL
  (void)base_s; return *reinterpret_cast<const uint2*>(reinterpret_cast<const char*>(base) + byte_off);
#else
  (void)base; uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(base_s + (unsigned)byte_off));
  return v;
#endif
}
__device__ __forceinline__ uint4 lds_u32x4(const void* base, unsigned base_s, int byte_off) {   // 16-byte aligned
#ifdef SGX_EMUL
  (void)base_s; return *reinterpret_cast<const uint4*>(reinterpret_cast<const char*>(base) + byte_off);
#else
  (void)base; uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "r"(base_s + (unsigned)byte_off));
  return v;
#endif
}
__device__ __forceinline__ double2 lds_f64x2(const void* base, unsigned base_s, int byte_off) {   // 16-byte aligned
#ifdef SGX_EMUL
  (void)base_s; return *reinterpret_cast<const double2*>(reinterpret_cast<const char*>(base) + byte_off);
#else
  (void)base; double2 v;
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(base_s + (unsigned)byte_off));
  return v;
#endif
}

// one thread: arm the barrier with the byte count and start the copy (bytes % 16 == 0, both 16B-aligned)
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, unsigned bytes,
                                          unsigned long long* bar) {
#ifdef SGX_EMUL
  memcpy(smem_dst, gsrc, bytes);
  *bar += 1;  // completed phases
#else
  unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  unsigned b = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(b), "r"(bytes) : "memory");
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(d),
      "l"(gsrc), "r"(bytes), "r"(b)
      : "memory");
#endif
}
// all threads: wait until phase `parity` of the barrier has completed
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
#ifdef SGX_EMUL
  // bulk_load bumps the completed-phase count; phase `parity` is done once the count's low bit differs
  while ((*(volatile unsigned long long*)bar & 1ull) == (unsigned long long)parity) sgx_emul::yield_to_sched();
#else
  unsigned b = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}\n" ::"r"(b),
      "r"(parity)
      : "memory");
#endif
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  return v;
}

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  return v;
}

}  // namespace sgx

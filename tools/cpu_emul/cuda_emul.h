// Minimal CPU emulation of the CUDA subset used by softgnss_python_b200/csrc/*.cu.
//
// DEVELOPER AID ONLY -- never built by __graft_entry__.build(), never loaded by the package,
// never timed.  There is no GPU in the build container, so this header lets the *same kernel
// sources* be compiled with g++ (-DSGX_EMUL) and single-stepped / diffed against the oracle
// before a gpurun call is spent.  Every CUDA thread of a block is a fiber (hand-rolled x86-64
// context switch) on one OS thread; __syncthreads() and warp shuffles are cooperative yields,
// so execution is deterministic.  Blocks are distributed over a few OS threads and
// `__shared__` becomes `static thread_local`.
#pragma once
#ifndef __x86_64__
#error "cuda_emul.h: x86-64 only"
#endif
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <thread>
#include <vector>

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __noinline__
#define __restrict__
#define __launch_bounds__(...)
#define __shared__ static thread_local
#define __constant__ static
#define __align__(n) __attribute__((aligned(n)))

struct dim3 {
  unsigned x, y, z;
  dim3(unsigned a = 1, unsigned b = 1, unsigned c = 1) : x(a), y(b), z(c) {}
};
struct uint3_ { unsigned x, y, z; };
struct float2 { float x, y; };
struct float4 { float x, y, z, w; };
struct double2 { double x, y; };
struct int2 { int x, y; };
struct int4 { int x, y, z, w; };
struct uint2 { unsigned x, y; };
struct uint4 { unsigned x, y, z, w; };
static inline float2 make_float2(float a, float b) { return {a, b}; }
static inline float4 make_float4(float a, float b, float c, float d) { return {a, b, c, d}; }
static inline double2 make_double2(double a, double b) { return {a, b}; }
static inline int4 make_int4(int a, int b, int c, int d) { return {a, b, c, d}; }
static inline uint4 make_uint4(unsigned a, unsigned b, unsigned c, unsigned d) { return {a, b, c, d}; }
static inline int2 make_int2(int a, int b) { return {a, b}; }

namespace sgx_emul {

extern "C" void sgx_emul_ctx_switch(void** save_sp, void* load_sp);
asm(".text\n.weak sgx_emul_ctx_switch\n.type sgx_emul_ctx_switch,@function\n"
    "sgx_emul_ctx_switch:\n"
    "  pushq %rbp\n  pushq %rbx\n  pushq %r12\n  pushq %r13\n  pushq %r14\n  pushq %r15\n"
    "  movq %rsp, (%rdi)\n  movq %rsi, %rsp\n"
    "  popq %r15\n  popq %r14\n  popq %r13\n  popq %r12\n  popq %rbx\n  popq %rbp\n  ret\n");

struct Fiber {
  void* sp = nullptr;
  char* stack = nullptr;
  bool done = false;
  unsigned tid = 0;
};

struct WarpState {
  unsigned long long slot[2][32];
  int arrived[2] = {0, 0};
  int gen[2] = {0, 0};
  int phase = 0;
  int alive = 0;
};

struct BlockCtx {
  std::vector<Fiber> fibers;
  std::vector<WarpState> warps;
  void* sched_sp = nullptr;
  int cur = -1;
  int alive = 0;
  int bar_arrived = 0;
  int bar_gen = 0;
  int nbar_arrived[16] = {0};
  int nbar_gen[16] = {0};
  dim3 grid, block;
  uint3_ bidx;
  const std::function<void()>* body = nullptr;
  unsigned char* dyn_smem = nullptr;
};

inline thread_local BlockCtx* g_ctx = nullptr;
constexpr size_t kStack = 256 * 1024;

inline void yield_to_sched() {
  BlockCtx* c = g_ctx;
  Fiber& f = c->fibers[c->cur];
  sgx_emul_ctx_switch(&f.sp, c->sched_sp);
}

inline void fiber_main() {
  BlockCtx* c = g_ctx;
  (*c->body)();
  Fiber& f = c->fibers[c->cur];
  f.done = true;
  c->alive--;
  c->warps[f.tid / 32].alive--;
  yield_to_sched();
  abort();
}

inline void run_block(BlockCtx& c) {
  g_ctx = &c;
  const int n = (int)c.fibers.size();
  c.alive = n;
  c.bar_arrived = 0;
  for (int i = 0; i < 16; ++i) c.nbar_arrived[i] = 0;
  for (auto& w : c.warps) { w = WarpState(); }
  for (int i = 0; i < n; ++i) {
    Fiber& f = c.fibers[i];
    f.done = false;
    f.tid = i;
    c.warps[i / 32].alive++;
    uintptr_t top = ((uintptr_t)(f.stack + kStack)) & ~(uintptr_t)15;
    void** sp = (void**)top;
    *(--sp) = nullptr;                 // fake return address of fiber_main (alignment)
    *(--sp) = (void*)&fiber_main;      // `ret` target
    for (int k = 0; k < 6; ++k) *(--sp) = nullptr;
    f.sp = sp;
  }
  while (c.alive > 0) {
    for (int i = 0; i < n; ++i) {
      if (c.fibers[i].done) continue;
      c.cur = i;
      sgx_emul_ctx_switch(&c.sched_sp, c.fibers[i].sp);
    }
  }
  g_ctx = nullptr;
}

inline void launch(dim3 grid, dim3 block, size_t smem, const std::function<void()>& body) {
  const size_t nblocks = (size_t)grid.x * grid.y * grid.z;
  const unsigned nthreads = block.x * block.y * block.z;
  unsigned nworkers = std::min<size_t>(std::max(1u, std::thread::hardware_concurrency()), nblocks);
  if (getenv("SGX_EMUL_THREADS")) nworkers = std::max(1, atoi(getenv("SGX_EMUL_THREADS")));
  std::atomic<size_t> next{0};
  auto worker = [&]() {
    BlockCtx c;
    c.grid = grid;
    c.block = block;
    c.body = &body;
    c.fibers.resize(nthreads);
    c.warps.resize((nthreads + 31) / 32);
    for (auto& f : c.fibers) f.stack = (char*)malloc(kStack);
    c.dyn_smem = (unsigned char*)aligned_alloc(1024, ((smem + 1023) / 1024 + 1) * 1024);
    for (;;) {
      size_t b = next.fetch_add(1);
      if (b >= nblocks) break;
      c.bidx.x = (unsigned)(b % grid.x);
      c.bidx.y = (unsigned)((b / grid.x) % grid.y);
      c.bidx.z = (unsigned)(b / ((size_t)grid.x * grid.y));
      run_block(c);
    }
    for (auto& f : c.fibers) free(f.stack);
    free(c.dyn_smem);
  };
  std::vector<std::thread> ths;
  for (unsigned i = 1; i < nworkers; ++i) ths.emplace_back(worker);
  worker();
  for (auto& t : ths) t.join();
}

struct ThreadIdxT {
  struct X { operator unsigned() const { return g_ctx->fibers[g_ctx->cur].tid % g_ctx->block.x; } } x;
  struct Y { operator unsigned() const { return (g_ctx->fibers[g_ctx->cur].tid / g_ctx->block.x) % g_ctx->block.y; } } y;
  struct Z { operator unsigned() const { return g_ctx->fibers[g_ctx->cur].tid / (g_ctx->block.x * g_ctx->block.y); } } z;
};
struct BlockIdxT {
  struct X { operator unsigned() const { return g_ctx->bidx.x; } } x;
  struct Y { operator unsigned() const { return g_ctx->bidx.y; } } y;
  struct Z { operator unsigned() const { return g_ctx->bidx.z; } } z;
};
struct BlockDimT {
  struct X { operator unsigned() const { return g_ctx->block.x; } } x;
  struct Y { operator unsigned() const { return g_ctx->block.y; } } y;
  struct Z { operator unsigned() const { return g_ctx->block.z; } } z;
};
struct GridDimT {
  struct X { operator unsigned() const { return g_ctx->grid.x; } } x;
  struct Y { operator unsigned() const { return g_ctx->grid.y; } } y;
  struct Z { operator unsigned() const { return g_ctx->grid.z; } } z;
};

inline void syncthreads() {
  BlockCtx* c = g_ctx;
  int my = c->bar_gen;
  c->bar_arrived++;
  for (;;) {
    if (c->bar_gen != my) break;
    if (c->bar_arrived >= c->alive) { c->bar_arrived = 0; c->bar_gen++; break; }
    yield_to_sched();
  }
}

// bar.sync id, count: a barrier among `count` threads of the block (the callers partition the block statically)
inline void named_barrier(int id, int count) {
  BlockCtx* c = g_ctx;
  int my = c->nbar_gen[id];
  c->nbar_arrived[id]++;
  for (;;) {
    if (c->nbar_gen[id] != my) break;
    if (c->nbar_arrived[id] >= count) { c->nbar_arrived[id] = 0; c->nbar_gen[id]++; break; }
    yield_to_sched();
  }
}

// all-lanes exchange: every live lane of the warp deposits v, waits for the rest, reads src lane
inline unsigned long long warp_exchange(unsigned long long v, int src_lane) {
  BlockCtx* c = g_ctx;
  unsigned tid = c->fibers[c->cur].tid;
  WarpState& w = c->warps[tid / 32];
  int lane = tid % 32;
  int p = w.phase;                      // all lanes observe the same phase on entry
  int my = w.gen[p];
  w.slot[p][lane] = v;
  w.arrived[p]++;
  for (;;) {
    if (w.gen[p] != my) break;
    if (w.arrived[p] >= w.alive) { w.arrived[p] = 0; w.gen[p]++; w.phase = p ^ 1; break; }
    yield_to_sched();
  }
  return w.slot[p][src_lane & 31];
}

template <class T> inline T shfl(T v, int src_lane) {
  static_assert(sizeof(T) <= 8, "shfl size");
  unsigned long long raw = 0;
  memcpy(&raw, &v, sizeof(T));
  raw = warp_exchange(raw, src_lane);
  T out;
  memcpy(&out, &raw, sizeof(T));
  return out;
}
inline int lane_id() { return g_ctx->fibers[g_ctx->cur].tid % 32; }

}  // namespace sgx_emul

static sgx_emul::ThreadIdxT threadIdx;
static sgx_emul::BlockIdxT blockIdx;
static sgx_emul::BlockDimT blockDim;
static sgx_emul::GridDimT gridDim;

static inline void __syncthreads() { sgx_emul::syncthreads(); }
static inline void __syncwarp(unsigned = 0xffffffffu) { sgx_emul::warp_exchange(0, 0); }
template <class T> static inline T __shfl_sync(unsigned, T v, int src, int = 32) { return sgx_emul::shfl(v, src); }
template <class T> static inline T __shfl_xor_sync(unsigned, T v, int m, int = 32) {
  return sgx_emul::shfl(v, sgx_emul::lane_id() ^ m);
}
template <class T> static inline T __shfl_down_sync(unsigned, T v, int d, int = 32) {
  int l = sgx_emul::lane_id();
  return sgx_emul::shfl(v, l + d < 32 ? l + d : l);
}
static inline unsigned __ballot_sync(unsigned, int pred) {
  unsigned r = 0;
  for (int i = 0; i < 32; ++i) { /* one exchange per lane keeps the helper tiny */
    unsigned b = sgx_emul::shfl<unsigned>(pred ? 1u : 0u, i);
    r |= (b & 1u) << i;
  }
  return r;
}

// ---- math / bit intrinsics ------------------------------------------------------------------
static inline void sincospif(float x, float* s, float* c) { *s = (float)sin(M_PI * (double)x); *c = (float)cos(M_PI * (double)x); }
static inline void sincospi(double x, double* s, double* c) { *s = sin(M_PI * x); *c = cos(M_PI * x); }
static inline float __fmaf_rn(float a, float b, float c) { return fmaf(a, b, c); }
static inline float __fmul_rn(float a, float b) { volatile float r = a * b; return r; }
static inline float __fadd_rn(float a, float b) { volatile float r = a + b; return r; }
static inline double __dmul_rn(double a, double b) { volatile double r = a * b; return r; }
static inline double __dadd_rn(double a, double b) { volatile double r = a + b; return r; }
static inline double __dsub_rn(double a, double b) { volatile double r = a - b; return r; }
static inline double __ddiv_rn(double a, double b) { volatile double r = a / b; return r; }
static inline double __fma_rn(double a, double b, double c) { return fma(a, b, c); }
static inline int __double2int_ru(double x) { return (int)ceil(x); }
static inline int __double2int_rd(double x) { return (int)floor(x); }
static inline long long __double2ll_rd(double x) { return (long long)floor(x); }
static inline long long __double2ll_rn(double x) { return (long long)llrint(x); }
static inline double __int2double_rn(int x) { return (double)x; }
static inline double __ll2double_rn(long long x) { return (double)x; }
static inline unsigned __float_as_uint(float f) { unsigned u; memcpy(&u, &f, 4); return u; }
static inline float __uint_as_float(unsigned u) { float f; memcpy(&f, &u, 4); return f; }
static inline int __float_as_int(float f) { int u; memcpy(&u, &f, 4); return u; }
static inline float __int_as_float(int u) { float f; memcpy(&f, &u, 4); return f; }
static inline unsigned __byte_perm(unsigned a, unsigned b, unsigned s) {
  unsigned long long src = ((unsigned long long)b << 32) | a;
  unsigned r = 0;
  for (int i = 0; i < 4; ++i) {
    unsigned sel = (s >> (4 * i)) & 0xF;
    unsigned byte = (unsigned)((src >> (8 * (sel & 7))) & 0xFF);
    if (sel & 8) byte = (byte & 0x80) ? 0xFF : 0x00;
    r |= byte << (8 * i);
  }
  return r;
}
static inline unsigned __funnelshift_r(unsigned lo, unsigned hi, unsigned sh) {
  return (unsigned)(((((unsigned long long)hi) << 32) | lo) >> (sh & 31));
}
static inline unsigned __funnelshift_lc(unsigned lo, unsigned hi, unsigned sh) { if (sh > 32) sh = 32; unsigned long long v = ((unsigned long long)hi << 32) | lo; return sh == 32 ? lo : (unsigned)((v << sh) >> 32); }
static inline unsigned __funnelshift_rc(unsigned lo, unsigned hi, unsigned sh) { if (sh > 32) sh = 32; unsigned long long v = ((unsigned long long)hi << 32) | lo; return (unsigned)(v >> sh); }
static inline int __double2hiint(double x) { long long v; memcpy(&v, &x, 8); return (int)(v >> 32); }
static inline int __double2loint(double x) { long long v; memcpy(&v, &x, 8); return (int)(v & 0xffffffffLL); }
static inline double __hiloint2double(int hi, int lo) { long long v = ((long long)hi << 32) | (unsigned)lo; double x; memcpy(&x, &v, 8); return x; }
static inline double __longlong_as_double(long long v) { double x; memcpy(&x, &v, 8); return x; }
static inline int __dp4a(int a, int b, int c) {
  for (int i = 0; i < 4; ++i) c += (int)(signed char)((a >> (8 * i)) & 0xFF) * (int)(signed char)((b >> (8 * i)) & 0xFF);
  return c;
}
static inline int __popc(unsigned x) { return __builtin_popcount(x); }
static inline int __clz(int x) { return x ? __builtin_clz((unsigned)x) : 32; }
static inline int __ffs(int x) { return __builtin_ffs(x); }
static inline unsigned long long __umul64hi(unsigned long long a, unsigned long long b) {
  return (unsigned long long)(((unsigned __int128)a * b) >> 64);
}
template <class T> static inline T __ldg(const T* p) { return *p; }
template <class T> static inline T __ldcg(const T* p) { return *p; }
template <class T> static inline T __ldcs(const T* p) { return *p; }
template <class T> static inline void __stcg(T* p, T v) { *p = v; }
static inline float rsqrtf(float x) { return 1.0f / sqrtf(x); }
static inline float __fdividef(float a, float b) { return a / b; }
using std::max;
using std::min;

// ---- atomics (blocks run concurrently on a few OS threads) ----------------------------------
static inline int atomicAdd(int* p, int v) { return __atomic_fetch_add(p, v, __ATOMIC_RELAXED); }
static inline unsigned atomicAdd(unsigned* p, unsigned v) { return __atomic_fetch_add(p, v, __ATOMIC_RELAXED); }
static inline unsigned long long atomicAdd(unsigned long long* p, unsigned long long v) { return __atomic_fetch_add(p, v, __ATOMIC_RELAXED); }
static inline unsigned long long atomicMax(unsigned long long* p, unsigned long long v) {
  unsigned long long old = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (old < v && !__atomic_compare_exchange_n(p, &old, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
  return old;
}
static inline int atomicMax(int* p, int v) {
  int old = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (old < v && !__atomic_compare_exchange_n(p, &old, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
  return old;
}
static inline int atomicMin(int* p, int v) {
  int old = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (old > v && !__atomic_compare_exchange_n(p, &old, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
  return old;
}
static inline int atomicExch(int* p, int v) { return __atomic_exchange_n(p, v, __ATOMIC_RELAXED); }
static inline void __threadfence() { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
static inline void __threadfence_block() {}
static inline long long clock64() { return 0; }

// ---- runtime API stubs -----------------------------------------------------------------------
typedef int cudaError_t;
typedef void* cudaStream_t;
typedef void* cudaEvent_t;
enum { cudaSuccess = 0 };
enum cudaMemcpyKind { cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost, cudaMemcpyDeviceToDevice, cudaMemcpyDefault };
enum cudaMemoryType { cudaMemoryTypeUnregistered = 0, cudaMemoryTypeHost = 1, cudaMemoryTypeDevice = 2, cudaMemoryTypeManaged = 3 };
struct cudaPointerAttributes { cudaMemoryType type; int device; };
enum cudaFuncAttribute { cudaFuncAttributeMaxDynamicSharedMemorySize, cudaFuncAttributePreferredSharedMemoryCarveout };
struct cudaDeviceProp { int multiProcessorCount; char name[64]; size_t totalGlobalMem; int major, minor; };
static inline cudaError_t cudaMalloc(void** p, size_t n) { *p = aligned_alloc(256, ((n + 255) / 256 + 1) * 256); return *p ? 0 : 2; }
template <class T> static inline cudaError_t cudaMalloc(T** p, size_t n) { return cudaMalloc((void**)p, n); }
static inline cudaError_t cudaFree(void* p) { free(p); return 0; }
static inline cudaError_t cudaMallocHost(void** p, size_t n) { return cudaMalloc(p, n); }
enum { cudaHostAllocDefault = 0 };
static inline cudaError_t cudaHostAlloc(void** p, size_t n, unsigned) { return cudaMalloc(p, n); }
static inline cudaError_t cudaFreeHost(void* p) { free(p); return 0; }
static inline cudaError_t cudaMemcpy(void* d, const void* s, size_t n, cudaMemcpyKind) { memcpy(d, s, n); return 0; }
static inline cudaError_t cudaMemcpyAsync(void* d, const void* s, size_t n, cudaMemcpyKind, cudaStream_t = 0) { memcpy(d, s, n); return 0; }
static inline cudaError_t cudaMemset(void* d, int v, size_t n) { memset(d, v, n); return 0; }
static inline cudaError_t cudaMemsetAsync(void* d, int v, size_t n, cudaStream_t = 0) { memset(d, v, n); return 0; }
static inline cudaError_t cudaStreamSynchronize(cudaStream_t) { return 0; }
template <class T> static inline cudaError_t cudaMemcpyToSymbolAsync(T& sym, const void* src, size_t n, size_t, cudaMemcpyKind, cudaStream_t = 0) { memcpy(&sym, src, n); return 0; }
static inline cudaError_t cudaDeviceSynchronize() { return 0; }
static inline cudaError_t cudaGetLastError() { return 0; }
static inline cudaError_t cudaPeekAtLastError() { return 0; }
static inline const char* cudaGetErrorString(cudaError_t) { return "emul"; }
static inline cudaError_t cudaGetDeviceCount(int* n) { *n = 1; return 0; }
static inline cudaError_t cudaSetDevice(int) { return 0; }
static inline cudaError_t cudaGetDevice(int* d) { *d = 0; return 0; }
static inline cudaError_t cudaGetDeviceProperties(cudaDeviceProp* p, int) { memset(p, 0, sizeof(*p)); p->multiProcessorCount = 8; strcpy(p->name, "cpu-emul"); p->major = 10; return 0; }
static inline cudaError_t cudaPointerGetAttributes(cudaPointerAttributes* a, const void*) {
  // SGX_EMUL_HOST=1 makes every caller buffer look like host memory, which exercises the staging paths
  a->type = getenv("SGX_EMUL_HOST") ? cudaMemoryTypeUnregistered : cudaMemoryTypeDevice;
  a->device = 0;
  return 0;
}
template <class F> static inline cudaError_t cudaFuncSetAttribute(F, cudaFuncAttribute, int) { return 0; }
struct cudaFuncAttributes { size_t sharedSizeBytes; };
template <class F> static inline cudaError_t cudaFuncGetAttributes(cudaFuncAttributes* a, F) { a->sharedSizeBytes = 0; return 0; }
enum cudaDeviceAttr { cudaDevAttrMultiProcessorCount = 16 };
static inline cudaError_t cudaDeviceGetAttribute(int* v, cudaDeviceAttr, int) { *v = 8; return 0; }
template <class F> static inline cudaError_t cudaOccupancyMaxActiveBlocksPerMultiprocessor(int* n, F, int, size_t) { *n = 2; return 0; }
static inline cudaError_t cudaEventCreate(cudaEvent_t*) { return 0; }
static inline cudaError_t cudaEventRecord(cudaEvent_t, cudaStream_t = 0) { return 0; }
static inline cudaError_t cudaEventSynchronize(cudaEvent_t) { return 0; }
static inline cudaError_t cudaEventElapsedTime(float* ms, cudaEvent_t, cudaEvent_t) { *ms = 0; return 0; }
static inline cudaError_t cudaEventDestroy(cudaEvent_t) { return 0; }
enum { cudaStreamNonBlocking = 1, cudaEventDisableTiming = 2 };
static inline cudaError_t cudaStreamCreateWithFlags(cudaStream_t* s, unsigned) { *s = (cudaStream_t)1; return 0; }
static inline cudaError_t cudaEventCreateWithFlags(cudaEvent_t* e, unsigned) { *e = (cudaEvent_t)1; return 0; }
static inline cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned) { return 0; }
static inline cudaError_t cudaMemcpy2DAsync(void* d, size_t dp, const void* s, size_t sp, size_t w, size_t h, cudaMemcpyKind,
                                            cudaStream_t = 0) {
  for (size_t r = 0; r < h; ++r) memcpy((char*)d + r * dp, (const char*)s + r * sp, w);
  return 0;
}

#define SGX_LAUNCH(kernel, grid, block, smem, stream, ...) \
  sgx_emul::launch((grid), (block), (smem), [&]() { kernel(__VA_ARGS__); })
#define SGX_DYN_SMEM(name) unsigned char* name = sgx_emul::g_ctx->dyn_smem

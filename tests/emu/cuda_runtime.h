// TEST INFRASTRUCTURE ONLY - a CPU SIMT emulation of the slice of CUDA that mapdn_b200/csrc uses, so that the C-ABI
// library (kernels included) can be compiled with g++ (-DMAPDN_HOST_EMU -I tests/emu) into tests/emu/_build/
// libmapdn_b200_emu.so and the kernel SOURCE can be executed by the CPU test tier (tests/test_emu_kernel.py) against the
// oracle. It is never built into or loaded by the product (mapdn_b200/_capi.py only knows libmapdn_b200.so).
//
// Model: one OS thread per CUDA thread, the blocks of a grid run one after the other. __syncthreads / named barriers
// (bar.sync / bar.arrive / bar.red) are counting barriers of the block, __syncwarp / __shfl_xor_sync / __ballot_sync /
// __all_sync are barriers + an exchange array of the warp. The TMA bulk copy is a memcpy by the issuing thread;
// "device memory" is host memory. Device code that reaches a barrier a different number of times on different
// threads deadlocks here exactly like it does on the GPU (a watchdog aborts after MAPDN_EMU_TIMEOUT_S seconds).
#pragma once
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

// ---- qualifiers -------------------------------------------------------------------------------------------------
#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __launch_bounds__(...)
#define __grid_constant__
#define __restrict__
#define __align__(n) __attribute__((aligned(n)))
#define __shared__ static /* one block runs at a time: a block-shared variable is a process-wide static */

// ---- vector types -----------------------------------------------------------------------------------------------
struct __attribute__((aligned(16))) double2 { double x, y; };
struct __attribute__((aligned(16))) int4 { int x, y, z, w; };
struct __attribute__((aligned(16))) float4 { float x, y, z, w; };
struct __attribute__((aligned(8))) uint2 { unsigned x, y; };
struct __attribute__((aligned(4))) ushort2 { unsigned short x, y; };
struct dim3 { unsigned x = 1, y = 1, z = 1; dim3() {} dim3(unsigned a, unsigned b = 1, unsigned c = 1) : x(a), y(b), z(c) {} };
static inline double2 make_double2(double x, double y) { return double2{x, y}; }
static inline int4 make_int4(int x, int y, int z, int w) { return int4{x, y, z, w}; }
static inline float4 make_float4(float x, float y, float z, float w) { return float4{x, y, z, w}; }

// ---- runtime API (host memory stands in for device memory) -----------------------------------------------------------
typedef int cudaError_t;
typedef void* cudaStream_t;
enum { cudaSuccess = 0, cudaErrorInvalidValue = 1, cudaErrorMemoryAllocation = 2 };
enum cudaMemcpyKind { cudaMemcpyHostToHost, cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost, cudaMemcpyDeviceToDevice, cudaMemcpyDefault };
enum cudaMemoryType { cudaMemoryTypeUnregistered = 0, cudaMemoryTypeHost = 1, cudaMemoryTypeDevice = 2, cudaMemoryTypeManaged = 3 };
enum cudaFuncAttribute { cudaFuncAttributeMaxDynamicSharedMemorySize = 8 };
enum { cudaHostAllocDefault = 0, cudaHostAllocMapped = 2, cudaHostRegisterDefault = 0, cudaHostRegisterMapped = 2 };
struct cudaPointerAttributes { cudaMemoryType type; int device; void* devicePointer; void* hostPointer; };
struct cudaFuncAttributes { size_t sharedSizeBytes = 64; size_t constSizeBytes = 0; size_t localSizeBytes = 0; int maxThreadsPerBlock = 1024; int numRegs = 128; int maxDynamicSharedSizeBytes = 0; };
struct cudaDeviceProp {
  char name[256]; int multiProcessorCount; size_t sharedMemPerBlockOptin; size_t sharedMemPerMultiprocessor; size_t reservedSharedMemPerBlock;
  int major, minor; size_t totalGlobalMem; int maxThreadsPerMultiProcessor; int regsPerMultiprocessor; size_t sharedMemPerBlock; int warpSize;
};
static inline const char* cudaGetErrorString(cudaError_t e) { return e == cudaSuccess ? "no error" : "emulated CUDA error"; }
static inline cudaError_t cudaGetLastError() { return cudaSuccess; }
static inline cudaError_t cudaGetDevice(int* d) { *d = 0; return cudaSuccess; }
static inline cudaError_t cudaSetDevice(int) { return cudaSuccess; }
static inline cudaError_t cudaDeviceSynchronize() { return cudaSuccess; }
static inline cudaError_t cudaStreamSynchronize(cudaStream_t) { return cudaSuccess; }
static inline cudaError_t cudaMalloc(void** p, size_t n) { *p = aligned_alloc(256, (n + 255) / 256 * 256); return *p ? cudaSuccess : cudaErrorMemoryAllocation; }
template <class T> static inline cudaError_t cudaMalloc(T** p, size_t n) { return cudaMalloc(reinterpret_cast<void**>(p), n); }
static inline cudaError_t cudaFree(void* p) { free(p); return cudaSuccess; }
static inline cudaError_t cudaHostAlloc(void** p, size_t n, unsigned) { return cudaMalloc(p, n); }
static inline cudaError_t cudaHostRegister(void*, size_t, unsigned) { return cudaSuccess; }
static inline cudaError_t cudaMemcpy(void* d, const void* s, size_t n, cudaMemcpyKind) { memcpy(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemcpyAsync(void* d, const void* s, size_t n, cudaMemcpyKind, cudaStream_t = nullptr) { memcpy(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemset(void* d, int v, size_t n) { memset(d, v, n); return cudaSuccess; }
static inline cudaError_t cudaMemsetAsync(void* d, int v, size_t n, cudaStream_t = nullptr) { memset(d, v, n); return cudaSuccess; }
static inline cudaError_t cudaPointerGetAttributes(cudaPointerAttributes* a, const void* p) {   // every host buffer counts as pinned
  a->type = cudaMemoryTypeHost; a->device = 0; a->devicePointer = const_cast<void*>(p); a->hostPointer = const_cast<void*>(p); return cudaSuccess;
}
// The B200 numbers the host code plans with. MAPDN_EMU_SMS overrides the SM count (read when a handle is created): with
// one SM the planner picks the full-batch launch geometry (envs per CTA, shared-memory plan, several rounds of the
// persistent loop per CTA) at batch sizes the emulation can run.
static inline cudaError_t cudaGetDeviceProperties(cudaDeviceProp* p, int) {
  memset(p, 0, sizeof(*p)); snprintf(p->name, sizeof(p->name), "emulated B200");
  const char* sms = getenv("MAPDN_EMU_SMS");
  p->multiProcessorCount = sms ? std::max(1, atoi(sms)) : 148; p->sharedMemPerBlockOptin = 232448; p->sharedMemPerMultiprocessor = 233472; p->reservedSharedMemPerBlock = 1024;
  p->major = 10; p->minor = 0; p->totalGlobalMem = size_t(180) << 30; p->maxThreadsPerMultiProcessor = 2048; p->regsPerMultiprocessor = 65536;
  p->sharedMemPerBlock = 49152; p->warpSize = 32; return cudaSuccess;
}
template <class F> static inline cudaError_t cudaFuncSetAttribute(F, cudaFuncAttribute, int) { return cudaSuccess; }
template <class F> static inline cudaError_t cudaFuncGetAttributes(cudaFuncAttributes* a, F) { *a = cudaFuncAttributes(); return cudaSuccess; }
template <class F> static inline cudaError_t cudaOccupancyMaxActiveBlocksPerMultiprocessor(int* n, F, int threads, size_t smem) {
  const int by_smem = smem ? int((233472) / (smem + 1024)) : 32, by_thr = 2048 / std::max(1, threads);
  *n = std::max(0, std::min(by_smem, by_thr)); return cudaSuccess;
}

// ---- the SIMT machine -----------------------------------------------------------------------------------------------
namespace emu {

struct Barrier {          // counting barrier with "arrive without waiting" (bar.arrive) and an AND reduction (bar.red)
  std::mutex m; std::condition_variable cv; int count = 0; unsigned gen = 0; bool acc = true, result = true;
  // returns the AND of `pred` over the arrivals of this generation (only meaningful for waiting threads)
  bool arrive(int expected, bool wait, bool pred);
};

struct Block {
  int nthreads = 0;
  unsigned char* smem = nullptr;
  Barrier named[16];
  std::vector<std::unique_ptr<Barrier>> warp_bar;      // one per warp
  std::vector<uint64_t> xchg;                          // 32 slots per warp (shuffle / ballot exchange)
};

struct ThreadCtx { Block* blk = nullptr; int tid = 0, lane = 0, warp = 0; };
extern thread_local ThreadCtx tctx;
extern std::atomic<long long> g_deadline_ms;           // watchdog

inline long long now_ms() { return std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

inline bool Barrier::arrive(int expected, bool wait, bool pred) {
  std::unique_lock<std::mutex> lk(m);
  acc = acc && pred;
  const unsigned my = gen;
  if (++count >= expected) { result = acc; acc = true; count = 0; ++gen; cv.notify_all(); return result; }
  if (!wait) return true;
  while (gen == my) {
    if (cv.wait_for(lk, std::chrono::milliseconds(200)) == std::cv_status::timeout && now_ms() > g_deadline_ms.load()) {
      fprintf(stderr, "[emu] barrier watchdog: %d of %d threads arrived - a divergent barrier in device code\n", count, expected);
      abort();
    }
  }
  return result;
}

template <class F> void launch_impl(unsigned grid, unsigned block, size_t smem_bytes, F&& body);

}  // namespace emu

struct emu_uint3 { unsigned x, y, z; };
extern thread_local emu_uint3 threadIdx, blockIdx;
extern thread_local dim3 blockDim, gridDim;

#ifdef MAPDN_EMU_DEFINE_GLOBALS
thread_local emu::ThreadCtx emu::tctx;
std::atomic<long long> emu::g_deadline_ms{0};
thread_local emu_uint3 threadIdx, blockIdx;
thread_local dim3 blockDim, gridDim;
#endif

namespace emu {

inline unsigned char* dyn_smem() { return tctx.blk->smem; }

template <class F> void launch_impl(unsigned grid, unsigned block, size_t smem_bytes, F&& body) {
  const char* to = getenv("MAPDN_EMU_TIMEOUT_S");
  const long long budget_ms = 1000ll * (to ? atoll(to) : 120);
  for (unsigned b = 0; b < grid; ++b) {
    Block blk;
    blk.nthreads = int(block);
    blk.smem = static_cast<unsigned char*>(aligned_alloc(1024, (smem_bytes + 1023) / 1024 * 1024 + 1024));
    memset(blk.smem, 0xAB, smem_bytes);                 // uninitialised shared memory is garbage on the GPU too
    const int nwarps = (int(block) + 31) / 32;
    for (int w = 0; w < nwarps; ++w) blk.warp_bar.emplace_back(new Barrier());
    blk.xchg.assign(size_t(nwarps) * 32, 0);
    g_deadline_ms.store(now_ms() + budget_ms);
    std::vector<std::thread> th;
    th.reserve(block);
    for (unsigned t = 0; t < block; ++t)
      th.emplace_back([&, t]() {
        tctx.blk = &blk; tctx.tid = int(t); tctx.lane = int(t & 31); tctx.warp = int(t >> 5);
        threadIdx = emu_uint3{t, 0, 0}; blockIdx = emu_uint3{b, 0, 0}; blockDim = dim3(block); gridDim = dim3(grid);
        body();
      });
    for (auto& x : th) x.join();
    free(blk.smem);
  }
}

// kernel<<<grid, block, smem, stream>>>(args...)
template <class K, class... A> void launch(K kernel, unsigned grid, unsigned block, size_t smem, cudaStream_t, A... args) {
  launch_impl(grid, block, smem, [&]() { kernel(args...); });
}

inline int warp_threads() {      // threads of the calling thread's warp (the last warp of a block may be partial)
  const Block* b = tctx.blk;
  return std::min(32, b->nthreads - tctx.warp * 32);
}
inline void bar_sync(int id, int n) { tctx.blk->named[id].arrive(n, true, true); }
inline void bar_arrive(int id, int n) { tctx.blk->named[id].arrive(n, false, true); }
inline bool bar_red_and(int id, int n, bool pred) { return tctx.blk->named[id].arrive(n, true, pred); }

}  // namespace emu

// ---- device intrinsics ------------------------------------------------------------------------------------------------
static inline void __syncthreads() { emu::bar_sync(0, emu::tctx.blk->nthreads); }
static inline void __syncwarp(unsigned = 0xffffffffu) { emu::tctx.blk->warp_bar[emu::tctx.warp]->arrive(emu::warp_threads(), true, true); }
static inline void __threadfence_block() { std::atomic_thread_fence(std::memory_order_seq_cst); }
template <class T> static inline T emu_exchange(T v, int src_lane) {
  static_assert(sizeof(T) <= 8, "shuffle of <= 64-bit values");
  emu::Block* b = emu::tctx.blk;
  uint64_t raw = 0; memcpy(&raw, &v, sizeof(T));
  uint64_t* slot = b->xchg.data() + size_t(emu::tctx.warp) * 32;
  slot[emu::tctx.lane] = raw;
  __syncwarp();
  const uint64_t got = slot[src_lane & 31];
  __syncwarp();
  T out; memcpy(&out, &got, sizeof(T)); return out;
}
template <class T> static inline T __shfl_xor_sync(unsigned, T v, int mask) { return emu_exchange(v, emu::tctx.lane ^ mask); }
template <class T> static inline T __shfl_sync(unsigned, T v, int src) { return emu_exchange(v, src); }
static inline unsigned __ballot_sync(unsigned, bool pred) {
  emu::Block* b = emu::tctx.blk;
  uint64_t* slot = b->xchg.data() + size_t(emu::tctx.warp) * 32;
  slot[emu::tctx.lane] = pred ? 1u : 0u;
  __syncwarp();
  unsigned m = 0;
  for (int l = 0; l < emu::warp_threads(); ++l) m |= unsigned(slot[l] & 1u) << l;
  __syncwarp();
  return m;
}
static inline bool __all_sync(unsigned mask, bool pred) { const unsigned m = __ballot_sync(mask, pred); const int n = emu::warp_threads(); return m == (n == 32 ? 0xffffffffu : ((1u << n) - 1u)); }
template <class T> static inline T __ldg(const T* p) { return *p; }
static inline unsigned __umulhi(unsigned a, unsigned b) { return unsigned((uint64_t(a) * uint64_t(b)) >> 32); }
static inline long long clock64() { return 0; }
static inline size_t __cvta_generic_to_shared(const void* p) { return reinterpret_cast<size_t>(p); }

using std::max;
using std::min;

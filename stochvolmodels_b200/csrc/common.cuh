// common.cuh -- error plumbing, launch geometry and block reductions shared by the b200sv kernels.
// sm_100a only (B200: 148 SMs, 64 fp64 + 128 fp32 lanes / SM / clk, 227 KB smem / CTA).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>

namespace b200sv {

// thread-local last error string returned by b200sv_last_error()
inline std::string& last_error() {
  static thread_local std::string s;
  return s;
}
inline int fail(int code, const std::string& msg) {
  last_error() = msg;
  return code;
}

// The stream every HOST-LEVEL entry point of the calling thread works on: b200sv_set_stream (include/b200sv.h).  Defined once in
// mc_kernels.cu; the other translation units reach it through these accessors (one shared library, one thread-local).
cudaStream_t& current_stream_ref();
inline cudaStream_t current_stream() { return current_stream_ref(); }

#define B200SV_CUDA(call)                                                                           \
  do {                                                                                              \
    cudaError_t e__ = (call);                                                                       \
    if (e__ != cudaSuccess)                                                                         \
      return ::b200sv::fail(-2, std::string(#call) + ": " + cudaGetErrorString(e__));               \
  } while (0)

#define B200SV_REQUIRE(cond, msg)                                                                   \
  do {                                                                                              \
    if (!(cond)) return ::b200sv::fail(-1, std::string("invalid argument: ") + (msg));              \
  } while (0)

// persistent-grid geometry: one wave of resident CTAs (multiple of the SM count), capped by the work
struct Grid {
  int blocks;
  int threads;
};
template <typename K>
inline Grid persistent_grid(K kernel, int threads, long long work_items, int items_per_thread = 1) {
  int dev = 0, sms = 148, per_sm = 1;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0);
  if (per_sm < 1) per_sm = 1;
  long long need = (work_items + (long long)threads * items_per_thread - 1) / ((long long)threads * items_per_thread);
  long long full = (long long)sms * per_sm;
  Grid g;
  g.threads = threads;
  g.blocks = (int)(need < full ? (need < 1 ? 1 : need) : full);
  return g;
}

// ---- warp / block reductions in fp64 (fixed order => run-to-run deterministic) -------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

// reduce NV values per thread across the block; result valid in thread 0 (returned in v[])
template <int NV, int THREADS>
__device__ __forceinline__ void block_sum(double (&v)[NV], double* smem /* NV * THREADS/32 doubles */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int NW = THREADS / 32;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    double s = warp_sum(v[k]);
    if (lane == 0) smem[k * NW + warp] = s;
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      double s = lane < NW ? smem[k * NW + lane] : 0.0;
      s = warp_sum(s);
      v[k] = s;
    }
  }
  __syncthreads();
}

// cudaMallocAsync returns freed blocks to the OS at the next synchronisation unless the pool's release threshold is raised;
// the chain entry points allocate GBs of path state per call, so keep it cached (set once per device).
inline void ensure_pool_threshold() {
  static thread_local int done_for = -1;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev == done_for) return;
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
    unsigned long long thr = ~0ull;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  done_for = dev;
}

// Kernels launched by the calling thread (b200sv_launch_count).  Defined once in mc_kernels.cu.
long long& launch_count();

// Check a kernel launch (a cooperative launch passes its own result): an error becomes -2, a launch is counted.
inline int launched(const char* what, cudaError_t e = cudaGetLastError()) {
  if (e != cudaSuccess) return fail(-2, std::string(what) + ": " + cudaGetErrorString(e));
  ++launch_count();
  return 0;
}

// A stream-ordered device temporary of n T's, freed on its stream when it goes out of scope.
template <typename T>
struct DevBuf {
  T* p = nullptr;
  cudaStream_t st;
  explicit DevBuf(cudaStream_t s) : st(s) {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() {
    if (p) cudaFreeAsync(p, st);
  }
  cudaError_t alloc(size_t n) { return cudaMallocAsync((void**)&p, sizeof(T) * (n ? n : 1), st); }
  // alloc(n), then copy n T's from host memory
  cudaError_t upload(const void* src, size_t n) {
    const cudaError_t e = alloc(n);
    return e != cudaSuccess || n == 0 ? e : cudaMemcpyAsync(p, src, sizeof(T) * n, cudaMemcpyHostToDevice, st);
  }
};

// Body of a host-level entry point: body(stream) runs on the calling thread's stream (b200sv_set_stream) and declares its DevBufs
// inside, so they are freed when it returns.  The stream is then drained once on every path -- no copy into the caller's (possibly
// pinned) memory is in flight after the call -- and the first error is returned.
template <typename Body>
inline int host_call(Body&& body) {
  const cudaStream_t st = current_stream();
  ensure_pool_threshold();
  int rc = body(st);
  const cudaError_t e = cudaStreamSynchronize(st);
  if (rc == 0 && e != cudaSuccess) rc = fail(-2, std::string("cudaStreamSynchronize: ") + cudaGetErrorString(e));
  return rc;
}


}  // namespace b200sv

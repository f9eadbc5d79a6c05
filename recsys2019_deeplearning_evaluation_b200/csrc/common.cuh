// Shared plumbing for libb200rec.so: error reporting across the C ABI, launch accounting, device buffers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <atomic>
#include <new>

#include "b200rec.h"

namespace b200 {

void set_error(const char* fmt, ...);
extern std::atomic<int64_t> g_launches;

inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

struct CudaFail {
  int code;
};

#define B200_CUDA(expr)                                                                                  \
  do {                                                                                                   \
    cudaError_t _e = (expr);                                                                             \
    if (_e != cudaSuccess) {                                                                             \
      b200::set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__, cudaGetErrorString(_e));      \
      throw b200::CudaFail{_e == cudaErrorMemoryAllocation ? B200_E_NOMEM : B200_E_CUDA};                \
    }                                                                                                    \
  } while (0)

#define B200_REQUIRE(cond, ...)             \
  do {                                      \
    if (!(cond)) {                          \
      b200::set_error(__VA_ARGS__);         \
      throw b200::CudaFail{B200_E_INVALID}; \
    }                                       \
  } while (0)

// Wraps a C-ABI body: converts internal throws into return codes.
template <typename F>
inline int guarded(F&& f) {
  try {
    f();
    return B200_OK;
  } catch (const CudaFail& e) {
    return e.code;
  } catch (const std::bad_alloc&) {
    set_error("host allocation failed");
    return B200_E_NOMEM;
  } catch (...) {
    set_error("unexpected internal error");
    return B200_E_CUDA;
  }
}

// Owning device buffer (cudaMalloc/cudaFree); move-only.
template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  DevBuf() = default;
  explicit DevBuf(size_t count) { alloc(count); }
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; }
    return *this;
  }
  ~DevBuf() { release(); }
  void alloc(size_t count) {
    release();
    n = count;
    if (count) B200_CUDA(cudaMalloc(reinterpret_cast<void**>(&p), count * sizeof(T)));
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  T* get() const { return p; }
};

inline int sm_count() {
  int dev = 0, n = 0;
  B200_CUDA(cudaGetDevice(&dev));
  B200_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
  return n;
}

// Host-side replay of glibc's srand(seed) / rand() (TYPE_3 additive-feedback generator; the reference's samplers call libc's
// rand(), SLIM_BPR_Cython_Epoch.pyx:436-480, MatrixFactorization_Cython_Epoch.pyx:881-987): next() is rand().
struct GlibcRandHost {
  int32_t r[31];
  int f = 3, b = 0;
  void seed(unsigned s) {
    int32_t word = s == 0 ? 1 : (int32_t)s;
    r[0] = word;
    for (int i = 1; i < 31; ++i) {
      const long hi = word / 127773, lo = word % 127773;
      long w = 16807 * lo - 2836 * hi;
      if (w < 0) w += 2147483647;
      word = (int32_t)w;
      r[i] = word;
    }
    f = 3; b = 0;
    for (int i = 0; i < 310; ++i) raw();
  }
  uint32_t raw() {
    const uint32_t v = (uint32_t)r[f] + (uint32_t)r[b];
    r[f] = (int32_t)v;
    f = (f + 1) % 31;
    b = (b + 1) % 31;
    return v;
  }
  int next() { return (int)(raw() >> 1); }
};

inline unsigned div_up(long long a, long long b) { return static_cast<unsigned>((a + b - 1) / b); }

// Philox4x32-10: counter = (idx, blk), key = (seed, epoch); four 32-bit words per call.
__device__ __forceinline__ void philox_round(unsigned& c0, unsigned& c1, unsigned& c2, unsigned& c3, unsigned k0, unsigned k1) {
  const unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
  const unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
  c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
}
__device__ __forceinline__ uint4 philox(unsigned long long idx, unsigned blk, unsigned seed, unsigned epoch) {
  unsigned c0 = (unsigned)idx, c1 = (unsigned)(idx >> 32), c2 = blk, c3 = 0x9E3779B9u;
  unsigned k0 = seed, k1 = epoch;
#pragma unroll
  for (int r = 0; r < 10; ++r) { philox_round(c0, c1, c2, c3, k0, k1); k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
  return make_uint4(c0, c1, c2, c3);
}

}  // namespace b200

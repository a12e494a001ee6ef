// Shared helpers for the sm_100a kernels of libgeoformer_b200.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "geoformer_b200.h"

namespace gf {

// ---- error plumbing (thread-local message, int status; never exit()) -------------------------
void set_error(const char *fmt, ...);
void count_launch(int n = 1);

#define GF_CHECK_ARG(cond, ...)      \
  do {                               \
    if (!(cond)) {                   \
      gf::set_error(__VA_ARGS__);    \
      return GF_ERR_INVALID;         \
    }                                \
  } while (0)

#define GF_CUDA(call)                                                                      \
  do {                                                                                     \
    cudaError_t e__ = (call);                                                              \
    if (e__ != cudaSuccess) {                                                              \
      gf::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
      return GF_ERR_CUDA;                                                                  \
    }                                                                                      \
  } while (0)

// after a <<<>>> launch
#define GF_LAUNCHED()                                                                      \
  do {                                                                                     \
    gf::count_launch();                                                                    \
    cudaError_t e__ = cudaGetLastError();                                                  \
    if (e__ != cudaSuccess) {                                                              \
      gf::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__), __FILE__, __LINE__); \
      return GF_ERR_CUDA;                                                                  \
    }                                                                                      \
  } while (0)

int num_sms();

// Optional profiling hook (gf_set_stage_events): record the caller's CUDA events at the stage
// boundaries of the next hot-path call, on the stream the kernels are launched on.
enum Stage { ST_BEGIN = 0, ST_KNN_BUILT = 1, ST_KNN_DONE = 2, ST_GEO_READY = 3, ST_GEO_DONE = 4, ST_COUNT = 5 };
void stage_mark(int stage, cudaStream_t st);

// ---- bump allocator over a caller-provided workspace -------------------------------------------
// A piece of a workspace handed down to a nested layout, which carves it in turn.
struct Span {
  void *ptr;
  size_t bytes;
};

// Every layout is stated once, in a carve function: over a null workspace the Arena only measures (`off` ends as the
// layout's size), over the caller's workspace it hands out the pieces.  Pieces start at multiples of 256 bytes from a
// base that must itself be 256-byte aligned: the kernels read them with 16-byte loads.
struct Arena {
  char *base;
  size_t size, off;
  bool ok;
  Arena(void *p, size_t n) : base((char *)p), size(n), off(0), ok(((uintptr_t)p & 255) == 0) {}
  template <typename T>
  T *take(size_t count) {
    size_t bytes = (count * sizeof(T) + 255) & ~size_t(255);
    if (!ok || base == nullptr || off + bytes > size) {
      ok = false;
      off += bytes;
      return nullptr;
    }
    T *r = (T *)(base + off);
    off += bytes;
    return r;
  }
  Span span(size_t bytes) { return {take<char>(bytes), bytes}; }
  // the error of a carve that failed, once it has measured the whole layout
  int fail(const char *who) const {
    if ((uintptr_t)base & 255)
      set_error("%s: workspace %p is not 256-byte aligned", who, (void *)base);
    else
      set_error("%s: workspace too small (%zu bytes given, %zu needed)", who, size, off);
    return GF_ERR_WORKSPACE;
  }
};

// ---- device helpers ---------------------------------------------------------------------------

// Squared length with the reference kernels' FMA contraction (SASS of sampling_gpu.cu,
// ball_query_gpu.cu, interpolate_gpu.cu built for sm_100: FMUL y*y; FFMA x*x+; FFMA z*z+).
__device__ __forceinline__ float sq3(float ax, float ay, float az) {
  return __fmaf_rn(az, az, __fmaf_rn(ax, ax, __fmul_rn(ay, ay)));
}

// order-preserving map float -> uint32 (total order, -0 < +0)
__device__ __forceinline__ uint32_t f2ord(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

__device__ __forceinline__ float ld_nc_f32(const float *p) { return __ldg(p); }

}  // namespace gf

// Host-side helpers shared by every kernel family: error reporting across the C ABI
// (no exceptions cross it), CUDA status checks, the driver entry point for TMA descriptors.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/tokenhmr_b200.h"

namespace thmr {

inline char* last_error_buf() {
  static thread_local char buf[512] = "";
  return buf;
}
inline int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(last_error_buf(), 512, fmt, ap);
  va_end(ap);
  return code;
}

#define THMR_CUDA(expr)                                                                        \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      return ::thmr::fail(THMR_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                          __FILE__, __LINE__);                                                 \
  } while (0)

#define THMR_CHECK(cond, ...)                                    \
  do {                                                           \
    if (!(cond)) return ::thmr::fail(THMR_ERR_INVALID, __VA_ARGS__); \
  } while (0)

#define THMR_TRY(expr)          \
  do {                          \
    int _s = (expr);            \
    if (_s != THMR_OK) return _s; \
  } while (0)

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// libcuda is not linked (the build box has no driver): resolve cuTensorMapEncodeTiled at run time.
inline EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2D tensor map over a row-major [rows, cols] matrix with row pitch ld (elements), tile box
// [box_rows, box_cols]; swizzle chosen by the caller (box_cols * elem bytes must not exceed the swizzle span).
inline int make_tmap_2d(CUtensorMap* out, CUtensorMapDataType dt, int elem_bytes, const void* base, uint64_t rows,
                        uint64_t cols, uint64_t ld, uint32_t box_rows, uint32_t box_cols, CUtensorMapSwizzle swz) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return fail(THMR_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  THMR_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, "tensor map base %p not 16B aligned", base);
  THMR_CHECK((ld * elem_bytes) % 16 == 0, "tensor map row pitch %llu elements is not a multiple of 16 bytes",
             (unsigned long long)ld);
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstr[1] = {ld * elem_bytes};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, dt, 2, const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(THMR_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu ld=%llu box=%ux%u", (int)r,
                (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, box_rows, box_cols);
  return THMR_OK;
}
inline int make_tmap_2d_f16(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                            uint32_t box_rows, uint32_t box_cols, CUtensorMapSwizzle swz) {
  return make_tmap_2d(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, base, rows, cols, ld, box_rows, box_cols, swz);
}

// Bump allocator over a caller-provided workspace (1 KB aligned carves; base == nullptr only measures).
struct Bump {
  uint8_t* base;
  size_t off = 0;
  explicit Bump(void* b) : base(static_cast<uint8_t*>(b)) {}
  template <typename T>
  T* take(size_t n) {
    off = (off + 1023) & ~size_t(1023);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += n * sizeof(T);
    return p;
  }
};

#ifdef __CUDACC__
// In-graph timing: the first thread of block 0 of a kernel records the global nanosecond timer at kernel start
// (nullptr = off).  Kernels of a stream run back to back, so start(next) - start(this) is this kernel's share of the
// step inside the real CUDA-graph replay, without events between the launches (thmr_engine_forward_stamped).
__device__ __forceinline__ void stamp_start(unsigned long long* stamp) {
  if (stamp != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    *stamp = t;
  }
}
__global__ void stamp_kernel(unsigned long long* stamp) { stamp_start(stamp); }
#endif

inline int num_sms() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

}  // namespace thmr

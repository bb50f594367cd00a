// Shared helpers for the splitp_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/splitp_b200.h"

namespace spb {

void set_error(const char* fmt, ...);
extern unsigned long long g_launches;  // kernels launched by this library (spb_launch_count)

inline int sm_count() {
  static int cached = 0;
  if (cached == 0) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      cached = n;
    else
      return 148;
  }
  return cached;
}

#define SPB_CUDA(call)                                                                    \
  do {                                                                                    \
    cudaError_t e__ = (call);                                                             \
    if (e__ != cudaSuccess) {                                                             \
      spb::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      return SPB_ERR_CUDA;                                                                \
    }                                                                                     \
  } while (0)

#define SPB_LAUNCH_CHECK()                                                                \
  do {                                                                                    \
    __atomic_fetch_add(&spb::g_launches, 1ull, __ATOMIC_RELAXED);                         \
    cudaError_t e__ = cudaGetLastError();                                                 \
    if (e__ != cudaSuccess) {                                                             \
      spb::set_error("%s:%d kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(e__)); \
      return SPB_ERR_CUDA;                                                                \
    }                                                                                     \
  } while (0)

#define SPB_REQUIRE(cond, ...)       \
  do {                               \
    if (!(cond)) {                   \
      spb::set_error(__VA_ARGS__);   \
      return SPB_ERR_ARG;            \
    }                                \
  } while (0)

// Device-side copy of a split: shift of each side's digits inside the key, most significant first.
struct SplitDev {
  int n, a, b;
  uint8_t sh_a[SPB_MAX_TAXA];
  uint8_t sh_b[SPB_MAX_TAXA];
};

inline int make_split_dev(const spb_split* s, SplitDev* d, bool need_key64 = true) {
  if (!s) { set_error("split is NULL"); return SPB_ERR_ARG; }
  if (s->n < 1 || s->n > SPB_MAX_TAXA || s->a < 0 || s->b < 0 || s->a > s->n || s->b > s->n) {
    set_error("bad split sizes n=%d a=%d b=%d", s->n, s->a, s->b);
    return SPB_ERR_ARG;
  }
  if (need_key64 && s->n > 31) { set_error("uint64 keys need n <= 31 (got %d)", s->n); return SPB_ERR_UNSUPPORTED; }
  d->n = s->n; d->a = s->a; d->b = s->b;
  for (int i = 0; i < s->a; ++i) {
    if (s->idx_a[i] >= s->n) { set_error("split index out of range"); return SPB_ERR_ARG; }
    d->sh_a[i] = (uint8_t)(2 * (s->n - 1 - s->idx_a[i]));
  }
  for (int i = 0; i < s->b; ++i) {
    if (s->idx_b[i] >= s->n) { set_error("split index out of range"); return SPB_ERR_ARG; }
    d->sh_b[i] = (uint8_t)(2 * (s->n - 1 - s->idx_b[i]));
  }
  return SPB_OK;
}

// gram.cu: G0 = S0 S0^T (int32, both triangles) of nb tiled u8 matrices on the tensor cores; one K pass (pitch <= 32768).
// d_ncols: NULL (K = pitch) or int32 [nb] occupied columns per matrix.
int gram_u8_i32_launch(const uint8_t* d_s0, int64_t s0_stride, int nb, int64_t rows_pad, int64_t pitch, const int32_t* d_ncols,
                       int32_t* d_Gi, int64_t g_stride, cudaStream_t st);

// pairs.cu: scores of `batch` symmetric k x k matrices (4 < k <= 64, leading dimension ld, stride ld * ld), one warp per matrix
int score_gram_warp_launch(const double* d_G, int k, int64_t ld, int64_t batch, double* d_scores, cudaStream_t st);

__device__ __forceinline__ uint64_t side_index(uint64_t key, const uint8_t* sh, int len) {
  uint64_t r = 0;
  for (int i = 0; i < len; ++i) r = (r << 2) | ((key >> sh[i]) & 3ull);
  return r;
}

__device__ __forceinline__ uint64_t mix64(uint64_t x) {  // murmur3 finaliser
  x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
  return x;
}

}  // namespace spb

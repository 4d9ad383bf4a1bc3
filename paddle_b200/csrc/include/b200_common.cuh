// Common device helpers for the sm_100a kernels (no torch headers in .cu files: keeps nvcc fast).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace b200 {

enum DType : int { kF32 = 0, kF16 = 1, kBF16 = 2 };

#define B200_CUDA_CHECK(expr)                                                                  \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      b200::set_last_error(__FILE__, __LINE__, cudaGetErrorString(_e));                        \
    }                                                                                          \
  } while (0)

void set_last_error(const char* file, int line, const char* msg);

template <typename T> struct VecTraits;
template <> struct VecTraits<float> { static constexpr int kVec = 4; };
template <> struct VecTraits<__half> { static constexpr int kVec = 8; };
template <> struct VecTraits<__nv_bfloat16> { static constexpr int kVec = 8; };

template <typename T> __device__ __forceinline__ float to_f(T v);
template <> __device__ __forceinline__ float to_f<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float to_f<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ __half from_f<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// 16-byte vector of T
template <typename T> struct alignas(16) Vec16 {
  static constexpr int N = 16 / sizeof(T);
  T v[N];
};

template <typename T> __device__ __forceinline__ Vec16<T> ld16(const T* p) {
  Vec16<T> r;
  *reinterpret_cast<uint4*>(&r) = *reinterpret_cast<const uint4*>(p);
  return r;
}
// streaming (read-once) load: bypass L1 allocation
template <typename T> __device__ __forceinline__ Vec16<T> ld16_stream(const T* p) {
  Vec16<T> r;
  uint4 u;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w)
               : "l"(p));
  *reinterpret_cast<uint4*>(&r) = u;
  return r;
}
template <typename T> __device__ __forceinline__ void st16(T* p, const Vec16<T>& v) {
  *reinterpret_cast<uint4*>(p) = *reinterpret_cast<const uint4*>(&v);
}
template <typename T> __device__ __forceinline__ void st16_stream(T* p, const Vec16<T>& v) {
  const uint4 u = *reinterpret_cast<const uint4*>(&v);
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(u.x), "r"(u.y), "r"(u.z), "r"(u.w)
               : "memory");
}

// ---- GEMM epilogue
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752f)); }

// 32 consecutive outputs of one row (the first `valid` of them in bounds), stored or added to what is there: 16-byte vectors when the
// chunk is whole and aligned, element by element otherwise
template <typename TO>
__device__ __forceinline__ void store_row_chunk(TO* __restrict__ dst, const float (&v)[32], int valid, bool accumulate) {
  if (valid >= 32 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
    constexpr int N = Vec16<TO>::N;
#pragma unroll
    for (int q = 0; q < 32 / N; ++q) {
      Vec16<TO> o;
      if (accumulate) {
        Vec16<TO> old = ld16(dst + q * N);
#pragma unroll
        for (int j = 0; j < N; ++j) o.v[j] = from_f<TO>(v[q * N + j] + to_f(old.v[j]));
      } else {
#pragma unroll
        for (int j = 0; j < N; ++j) o.v[j] = from_f<TO>(v[q * N + j]);
      }
      st16(dst + q * N, o);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (j < valid) dst[j] = from_f<TO>(accumulate ? v[j] + to_f(dst[j]) : v[j]);
  }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Block-wide sum; `smem` must hold >= 33 floats. All threads get the result.
__device__ __forceinline__ float block_sum(float v, float* smem) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  if (lane == 0) smem[wid] = v;
  __syncthreads();
  float r = (lane < nw) ? smem[lane] : 0.f;
  r = warp_sum(r);
  __syncthreads();
  return r;
}
__device__ __forceinline__ float block_max(float v, float* smem) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_max(v);
  if (lane == 0) smem[wid] = v;
  __syncthreads();
  float r = (lane < nw) ? smem[lane] : -INFINITY;
  r = warp_max(r);
  __syncthreads();
  return r;
}

#define B200_DISPATCH_DTYPE(dtype, T, ...)                         \
  switch (dtype) {                                                 \
    case b200::kF32: { using T = float; __VA_ARGS__; break; }      \
    case b200::kF16: { using T = __half; __VA_ARGS__; break; }     \
    case b200::kBF16: { using T = __nv_bfloat16; __VA_ARGS__; break; } \
    default: b200::set_last_error(__FILE__, __LINE__, "unsupported dtype"); \
  }

// Driver-API entry points (cuTensorMapEncodeTiled) need the primary context current on the calling thread; autograd worker threads
// arrive cold.  Once per thread is enough, and doing it only once keeps cudaFree (an "unsafe" call under global-mode stream
// capture) out of recorded regions: every thread has been through a warm-up step before a capture starts.
inline void bind_primary_context() {
  static thread_local bool bound = false;
  if (!bound) {
    cudaFree(nullptr);
    bound = true;
  }
}

inline int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

}  // namespace b200

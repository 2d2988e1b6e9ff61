// Shared device/host helpers for libmedimgen_b200.so (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>

#include "../../include/medimgen_b200.h"

namespace mig {

// ---- error plumbing (thread-local message, int status across the ABI) ---------------------------
void set_error(const char* fmt, ...);
int check_launch(const char* what);  // cudaGetLastError -> status

#define MIG_REQUIRE(cond, ...)     \
  do {                             \
    if (!(cond)) {                 \
      mig::set_error(__VA_ARGS__); \
      return 1;                    \
    }                              \
  } while (0)

struct DeviceInfo {
  int sm_count;
  int cc_major, cc_minor;
  int max_smem_optin;
};
const DeviceInfo& device_info();

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
// 16-byte aligned (nullptr counts as aligned)
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Opt-in to > 48 KB of dynamic shared memory. cudaFuncSetAttribute is PER DEVICE, so the "already done" state is kept per
// device (one process may drive several GPUs); atomics make concurrent first calls from several host threads benign (the
// attribute call is idempotent).
struct SmemOptIn {
  std::atomic<int> bytes[16];
};
template <typename Kernel>
inline int ensure_dynamic_smem(Kernel kernel, int smem, SmemOptIn& state, const char* what) {
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 16) dev = 0;
  if (state.bytes[dev].load(std::memory_order_acquire) >= smem) return 0;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) {
    set_error("%s: cannot opt in to %d bytes of shared memory: %s", what, smem, cudaGetErrorString(e));
    return 1;
  }
  state.bytes[dev].store(smem, std::memory_order_release);
  return 0;
}

// ---- dtype helpers ------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ float to_f(T v);
template <>
__device__ __forceinline__ float to_f<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T>
__device__ __forceinline__ T from_f(float v);
template <>
__device__ __forceinline__ float from_f<float>(float v) { return v; }
template <>
__device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// 16-byte vector of T: 4 floats or 8 bf16
template <typename T>
struct Vec16 {
  static constexpr int N = 16 / sizeof(T);
  uint4 raw;
  __device__ __forceinline__ float get(int i) const {
    if constexpr (sizeof(T) == 4) {
      return reinterpret_cast<const float*>(&raw)[i];
    } else {
      return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(&raw)[i]);
    }
  }
  __device__ __forceinline__ void set(int i, float v) {
    if constexpr (sizeof(T) == 4) {
      reinterpret_cast<float*>(&raw)[i] = v;
    } else {
      reinterpret_cast<__nv_bfloat16*>(&raw)[i] = __float2bfloat16_rn(v);
    }
  }
};

template <typename T>
__device__ __forceinline__ Vec16<T> ld16(const T* p) {
  Vec16<T> v;
  v.raw = *reinterpret_cast<const uint4*>(p);
  return v;
}
template <typename T>
__device__ __forceinline__ void st16(T* p, const Vec16<T>& v) {
  *reinterpret_cast<uint4*>(p) = v.raw;
}
// streaming variants (read-once / write-once data): bypass L1 allocation
template <typename T>
__device__ __forceinline__ Vec16<T> ld16_stream(const T* p) {
  Vec16<T> v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.raw.x), "=r"(v.raw.y), "=r"(v.raw.z), "=r"(v.raw.w)
               : "l"(p));
  return v;
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

// block-wide sum, result valid in every thread. `smem` needs 33 floats.
__device__ __forceinline__ float block_sum(float v, float* smem) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) smem[warp] = v;
  __syncthreads();
  if (warp == 0) {
    float t = lane < nw ? smem[lane] : 0.f;
    t = warp_sum(t);
    if (lane == 0) smem[32] = t;
  }
  __syncthreads();
  return smem[32];
}
__device__ __forceinline__ float block_max(float v, float* smem) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) smem[warp] = v;
  __syncthreads();
  if (warp == 0) {
    float t = lane < nw ? smem[lane] : -INFINITY;
    t = warp_max(t);
    if (lane == 0) smem[32] = t;
  }
  __syncthreads();
  return smem[32];
}

// MUFU-based forms (ex2 + rcp, ~2 ulp): the normalisation kernels are otherwise bound by this math, not by HBM
__device__ __forceinline__ float silu_f(float x) { return __fdividef(x, 1.f + __expf(-x)); }
// d/dx [x*sigmoid(x)] = s*(1 + x*(1-s))
__device__ __forceinline__ float silu_grad_f(float x) {
  float s = __fdividef(1.f, 1.f + __expf(-x));
  return s * fmaf(x, 1.f - s, 1.f);
}

// bf16 activations: sigmoid through ONE MUFU op (tanh.approx, rel. error ~2^-11, far below bf16 resolution) instead
// of ex2 + rcp; the fp32 parity path keeps the forms above.
__device__ __forceinline__ float sigmoid_tanh_f(float x) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * x));
  return fmaf(0.5f, t, 0.5f);
}
template <typename T>
__device__ __forceinline__ float silu_t(float x) {
  if constexpr (sizeof(T) == 2) return x * sigmoid_tanh_f(x);
  else return silu_f(x);
}
template <typename T>
__device__ __forceinline__ float silu_grad_t(float x) {
  if constexpr (sizeof(T) == 2) {
    const float s = sigmoid_tanh_f(x);
    return s * fmaf(x, 1.f - s, 1.f);
  } else {
    return silu_grad_f(x);
  }
}

// grid sizing for bandwidth kernels: enough CTAs to fill 148 SMs a few times over, capped.
inline int bw_grid(int64_t work_items, int threads, int per_sm = 8) {
  int64_t blocks = (work_items + threads - 1) / threads;
  int64_t cap = (int64_t)device_info().sm_count * per_sm;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}


// Gather geometry shared by conv fwd (gathers x) and dgrad (gathers dy), SIMT and tcgen05 engines.
// source coordinate along axis i:  pos = m_i*a[i] + tap_i*b[i] + c[i];  valid iff pos >= 0,
// (exact ? pos % d[i] == 0 : true), pos / d[i] < src[i].
struct Gather {
  int N;
  int src[3], dst[3], ks[3];
  int a[3], b[3], c[3], d[3];
  int exact;
  int Csrc;     // channels of the gathered tensor (K per tap)
  int Cdst;     // GEMM N (channels produced)
  int T;        // taps
  int K;        // T*Csrc
  int64_t M;    // N*prod(dst)
  int64_t Mo;   // prod(dst)
};
Gather make_gather_fwd(const mig_conv_geom* g);
Gather make_gather_dgrad(const mig_conv_geom* g);

#define MIG_DISPATCH_DTYPE(dtype, T, ...)                \
  do {                                                   \
    if ((dtype) == MIG_F32) {                            \
      using T = float;                                   \
      __VA_ARGS__;                                       \
    } else if ((dtype) == MIG_BF16) {                    \
      using T = __nv_bfloat16;                           \
      __VA_ARGS__;                                       \
    } else {                                             \
      mig::set_error("unsupported dtype %d", (int)dtype); \
      return 1;                                          \
    }                                                    \
  } while (0)

}  // namespace mig

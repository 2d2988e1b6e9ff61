// Bandwidth-bound elementwise / layout / loss / scheduler / optimizer kernels.
// All are HBM-roofline kernels: 128-bit coalesced accesses, grid = multiple of the SM count,
// warp-shuffle reductions. Algorithmic bytes per element are listed in DESIGN.md.
#include <cmath>

#include "common.cuh"

namespace mig {

// ------------------------------------------------------------------------------------------------
// generic unary / binary maps
// ------------------------------------------------------------------------------------------------
template <typename T, typename F, int NIN>
__global__ void __launch_bounds__(256) map_kernel(const T* __restrict__ a, const T* __restrict__ b,
                                                  const T* __restrict__ c, T* __restrict__ y, int64_t n, int vec,
                                                  F f) {
  constexpr int V = Vec16<T>::N;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t nvec = vec ? n / V : 0;
  for (int64_t i = tid; i < nvec; i += stride) {
    Vec16<T> va = ld16(a + i * V), vb, vc, vy;
    if (NIN > 1) vb = ld16(b + i * V);
    if (NIN > 2) vc = ld16(c + i * V);
#pragma unroll
    for (int j = 0; j < V; ++j)
      vy.set(j, f(va.get(j), NIN > 1 ? vb.get(j) : 0.f, NIN > 2 ? vc.get(j) : 0.f));
    st16(y + i * V, vy);
  }
  for (int64_t i = nvec * V + tid; i < n; i += stride)
    y[i] = from_f<T>(f(to_f(a[i]), NIN > 1 ? to_f(b[i]) : 0.f, NIN > 2 ? to_f(c[i]) : 0.f));
}

template <typename T, int NIN, typename F>
static int launch_map(const void* a, const void* b, const void* c, void* y, int64_t n, void* stream, F f,
                      const char* what) {
  if (n <= 0) return 0;
  int vec = aligned16(a) && aligned16(y) && (NIN < 2 || aligned16(b)) && (NIN < 3 || aligned16(c));
  int grid = bw_grid((n + Vec16<T>::N - 1) / Vec16<T>::N, 256);
  map_kernel<T, F, NIN><<<grid, 256, 0, as_stream(stream)>>>((const T*)a, (const T*)b, (const T*)c, (T*)y, n, vec, f);
  return check_launch(what);
}

struct SiluF { __device__ float operator()(float x, float, float) const { return silu_f(x); } };
struct SiluBwdF { __device__ float operator()(float x, float dy, float) const { return dy * silu_grad_f(x); } };
struct AddF { __device__ float operator()(float a, float b, float) const { return a + b; } };
struct ScaleF { float s; __device__ float operator()(float a, float, float) const { return a * s; } };
struct MulF { __device__ float operator()(float a, float b, float) const { return a * b; } };
struct AddcmulF { __device__ float operator()(float a, float b, float c) const { return fmaf(b, c, a); } };

}  // namespace mig

using namespace mig;

namespace mig {
// y[r][c] = x[r][c] + bias[c] over channels-last rows (bias of the transposed convolution, whose forward runs on the
// dgrad kernels and therefore has no fused epilogue)
template <typename T>
__global__ void __launch_bounds__(256) add_channel_bias_kernel(const T* __restrict__ x, const float* __restrict__ bias,
                                                               T* __restrict__ y, int64_t rows, int C) {
  const int64_t total = rows * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x)
    y[i] = from_f<T>(to_f(x[i]) + bias[(int)(i % C)]);
}
template <typename T>
__global__ void __launch_bounds__(256) add_channel_bias_vec_kernel(const T* __restrict__ x, const float* __restrict__ bias,
                                                                   T* __restrict__ y, int64_t rows, int C) {
  constexpr int V = Vec16<T>::N;
  const int cv = C / V;
  const int64_t total = rows * cv;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c0 = (int)(i % cv) * V;
    Vec16<T> v = ld16(x + i * V), o;
#pragma unroll
    for (int j = 0; j < V; ++j) o.set(j, v.get(j) + bias[c0 + j]);
    st16(y + i * V, o);
  }
}
}  // namespace mig

extern "C" int mig_add_channel_bias(int dtype, const void* x, const float* bias, void* y, int64_t rows, int32_t C,
                                    void* stream) {
  MIG_REQUIRE(x && bias && y && rows >= 0 && C > 0, "add_channel_bias: bad argument");
  if (rows == 0) return 0;
  MIG_DISPATCH_DTYPE(dtype, T, {
    if (C % Vec16<T>::N == 0 && aligned16(x) && aligned16(y))
      add_channel_bias_vec_kernel<T><<<bw_grid(rows * C / Vec16<T>::N, 256), 256, 0, as_stream(stream)>>>(
          (const T*)x, bias, (T*)y, rows, C);
    else
      add_channel_bias_kernel<T><<<bw_grid(rows * C, 256), 256, 0, as_stream(stream)>>>((const T*)x, bias, (T*)y, rows, C);
  });
  return check_launch("add_channel_bias");
}

extern "C" int mig_silu_fwd(int dtype, const void* x, void* y, int64_t n, void* stream) {
  MIG_DISPATCH_DTYPE(dtype, T, return (launch_map<T, 1>(x, nullptr, nullptr, y, n, stream, SiluF{}, "silu_fwd")));
}
extern "C" int mig_silu_bwd(int dtype, const void* x, const void* dy, void* dx, int64_t n, void* stream) {
  MIG_DISPATCH_DTYPE(dtype, T, return (launch_map<T, 2>(x, dy, nullptr, dx, n, stream, SiluBwdF{}, "silu_bwd")));
}
extern "C" int mig_add(int dtype, const void* a, const void* b, void* y, int64_t n, void* stream) {
  MIG_DISPATCH_DTYPE(dtype, T, return (launch_map<T, 2>(a, b, nullptr, y, n, stream, AddF{}, "add")));
}
extern "C" int mig_mul(int dtype, const void* a, const void* b, void* y, int64_t n, void* stream) {
  MIG_DISPATCH_DTYPE(dtype, T, return (launch_map<T, 2>(a, b, nullptr, y, n, stream, MulF{}, "mul")));
}
extern "C" int mig_addcmul(int dtype, const void* a, const void* b, const void* c, void* y, int64_t n, void* stream) {
  MIG_DISPATCH_DTYPE(dtype, T, return (launch_map<T, 3>(a, b, c, y, n, stream, AddcmulF{}, "addcmul")));
}
extern "C" int mig_scale(int dtype, const void* x, void* y, float s, int64_t n, void* stream) {
  MIG_DISPATCH_DTYPE(dtype, T, return (launch_map<T, 1>(x, nullptr, nullptr, y, n, stream, ScaleF{s}, "scale")));
}

// ------------------------------------------------------------------------------------------------
// cast
// ------------------------------------------------------------------------------------------------
namespace mig {
template <typename TS, typename TD>
__global__ void __launch_bounds__(256) cast_kernel(const TS* __restrict__ x, TD* __restrict__ y, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x * 4;
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < n; i += stride) {
    if (i + 3 < n) {
      float v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = to_f(x[i + j]);
#pragma unroll
      for (int j = 0; j < 4; ++j) y[i + j] = from_f<TD>(v[j]);
    } else {
      for (int64_t j = i; j < n; ++j) y[j] = from_f<TD>(to_f(x[j]));
    }
  }
}
}  // namespace mig

extern "C" int mig_cast(int src_dtype, int dst_dtype, const void* x, void* y, int64_t n, void* stream) {
  if (n <= 0) return 0;
  int grid = bw_grid((n + 3) / 4, 256);
  if (src_dtype == MIG_F32 && dst_dtype == MIG_BF16)
    cast_kernel<float, __nv_bfloat16><<<grid, 256, 0, as_stream(stream)>>>((const float*)x, (__nv_bfloat16*)y, n);
  else if (src_dtype == MIG_BF16 && dst_dtype == MIG_F32)
    cast_kernel<__nv_bfloat16, float><<<grid, 256, 0, as_stream(stream)>>>((const __nv_bfloat16*)x, (float*)y, n);
  else if (src_dtype == MIG_F32 && dst_dtype == MIG_F32)
    cast_kernel<float, float><<<grid, 256, 0, as_stream(stream)>>>((const float*)x, (float*)y, n);
  else if (src_dtype == MIG_BF16 && dst_dtype == MIG_BF16)
    cast_kernel<__nv_bfloat16, __nv_bfloat16><<<grid, 256, 0, as_stream(stream)>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)y, n);
  else
    MIG_REQUIRE(false, "mig_cast: bad dtypes %d -> %d", src_dtype, dst_dtype);
  return check_launch("cast");
}

// ------------------------------------------------------------------------------------------------
// GEGLU
// ------------------------------------------------------------------------------------------------
namespace mig {
__device__ __forceinline__ float gelu_f(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ float gelu_grad_f(float x) {
  return 0.5f * (1.f + erff(x * 0.70710678118654752f)) + x * 0.3989422804014327f * __expf(-0.5f * x * x);
}
template <typename T>
__global__ void geglu_fwd_kernel(const T* __restrict__ x, T* __restrict__ y, int64_t rows, int H) {
  const int64_t total = rows * H;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i / H;
    int j = (int)(i - r * H);
    float a = to_f(x[r * 2 * H + j]), g = to_f(x[r * 2 * H + H + j]);
    y[i] = from_f<T>(a * gelu_f(g));
  }
}
template <typename T>
__global__ void geglu_bwd_kernel(const T* __restrict__ x, const T* __restrict__ dy, T* __restrict__ dx, int64_t rows,
                                 int H) {
  const int64_t total = rows * H;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i / H;
    int j = (int)(i - r * H);
    float a = to_f(x[r * 2 * H + j]), g = to_f(x[r * 2 * H + H + j]), d = to_f(dy[i]);
    dx[r * 2 * H + j] = from_f<T>(d * gelu_f(g));
    dx[r * 2 * H + H + j] = from_f<T>(d * a * gelu_grad_f(g));
  }
}
}  // namespace mig

extern "C" int mig_geglu_fwd(int dtype, const void* x, void* y, int64_t rows, int32_t H, void* stream) {
  if (rows * H <= 0) return 0;
  MIG_DISPATCH_DTYPE(dtype, T, (geglu_fwd_kernel<T><<<bw_grid(rows * H, 256), 256, 0, as_stream(stream)>>>(
                                   (const T*)x, (T*)y, rows, H)));
  return check_launch("geglu_fwd");
}
extern "C" int mig_geglu_bwd(int dtype, const void* x, const void* dy, void* dx, int64_t rows, int32_t H,
                             void* stream) {
  if (rows * H <= 0) return 0;
  MIG_DISPATCH_DTYPE(dtype, T, (geglu_bwd_kernel<T><<<bw_grid(rows * H, 256), 256, 0, as_stream(stream)>>>(
                                   (const T*)x, (const T*)dy, (T*)dx, rows, H)));
  return check_launch("geglu_bwd");
}

// ------------------------------------------------------------------------------------------------
// channel concat / split (rows = N*S voxels, channels-last so each row is contiguous)
// ------------------------------------------------------------------------------------------------
namespace mig {
template <typename T, bool SPLIT>
__global__ void __launch_bounds__(256) concat_kernel(T* __restrict__ a, T* __restrict__ b, T* __restrict__ y,
                                                     int64_t rows, int Ca, int Cb, int vec) {
  constexpr int V = Vec16<T>::N;
  const int C = Ca + Cb;
  if (vec) {
    const int cv = C / V, cav = Ca / V;
    const int64_t total = rows * cv;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
      int64_t r = i / cv;
      int c = (int)(i - r * cv);
      T* part = c < cav ? a + r * Ca + (int64_t)c * V : b + r * Cb + (int64_t)(c - cav) * V;
      if (SPLIT) st16(part, ld16(y + i * V)); else st16(y + i * V, ld16(part));
    }
  } else {
    const int64_t total = rows * C;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
      int64_t r = i / C;
      int c = (int)(i - r * C);
      T* part = c < Ca ? a + r * Ca + c : b + r * Cb + (c - Ca);
      if (SPLIT) *part = y[i]; else y[i] = *part;
    }
  }
}
template <typename T, bool SPLIT>
static int launch_concat(const void* a, const void* b, const void* y, int64_t rows, int Ca, int Cb, void* stream) {
  if (rows <= 0) return 0;
  constexpr int V = Vec16<T>::N;
  int vec = (Ca % V == 0) && (Cb % V == 0) && aligned16(a) && aligned16(b) && aligned16(y);
  int64_t items = vec ? rows * ((Ca + Cb) / V) : rows * (Ca + Cb);
  concat_kernel<T, SPLIT><<<bw_grid(items, 256), 256, 0, as_stream(stream)>>>((T*)a, (T*)b, (T*)y, rows, Ca, Cb, vec);
  return check_launch(SPLIT ? "split_channels" : "concat_channels");
}
}  // namespace mig

extern "C" int mig_concat_channels(int dtype, const void* a, const void* b, void* y, int64_t rows, int32_t Ca,
                                   int32_t Cb, void* stream) {
  MIG_DISPATCH_DTYPE(dtype, T, return (launch_concat<T, false>(a, b, y, rows, Ca, Cb, stream)));
}
extern "C" int mig_split_channels(int dtype, const void* y, void* a, void* b, int64_t rows, int32_t Ca, int32_t Cb,
                                  void* stream) {
  MIG_DISPATCH_DTYPE(dtype, T, return (launch_concat<T, true>(a, b, y, rows, Ca, Cb, stream)));
}

// ------------------------------------------------------------------------------------------------
// nearest upsample (integer factors) and its adjoint (sum over each fd*fh*fw cell)
// ------------------------------------------------------------------------------------------------
namespace mig {
struct UpGeom { int N, D, H, W, fd, fh, fw, C; };

template <typename T>
__global__ void __launch_bounds__(256) upsample_fwd_kernel(const T* __restrict__ x, T* __restrict__ y, UpGeom g,
                                                           int cw /*elements per work item*/) {
  const int OD = g.D * g.fd, OH = g.H * g.fh, OW = g.W * g.fw;
  const int cpr = g.C / cw;
  const int64_t total = (int64_t)g.N * OD * OH * OW * cpr;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int c = (int)(i % cpr);
    int64_t v = i / cpr;
    int ow = (int)(v % OW); v /= OW;
    int oh = (int)(v % OH); v /= OH;
    int od = (int)(v % OD);
    int n = (int)(v / OD);
    int64_t src = ((((int64_t)n * g.D + od / g.fd) * g.H + oh / g.fh) * g.W + ow / g.fw) * g.C + (int64_t)c * cw;
    int64_t dst = (i / cpr) * g.C + (int64_t)c * cw;
    if (cw > 1) st16(y + dst, ld16(x + src)); else y[dst] = x[src];
  }
}
template <typename T>
__global__ void __launch_bounds__(256) upsample_bwd_kernel(const T* __restrict__ dy, T* __restrict__ dx, UpGeom g,
                                                           int cw) {
  const int OH = g.H * g.fh, OW = g.W * g.fw;
  const int cpr = g.C / cw;
  const int64_t total = (int64_t)g.N * g.D * g.H * g.W * cpr;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int c = (int)(i % cpr);
    int64_t v = i / cpr;
    int w = (int)(v % g.W); v /= g.W;
    int h = (int)(v % g.H); v /= g.H;
    int d = (int)(v % g.D);
    int n = (int)(v / g.D);
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int a = 0; a < g.fd; ++a)
      for (int b = 0; b < g.fh; ++b)
        for (int e = 0; e < g.fw; ++e) {
          int64_t src = ((((int64_t)n * g.D * g.fd + d * g.fd + a) * OH + h * g.fh + b) * OW + w * g.fw + e) * g.C +
                        (int64_t)c * cw;
          if (cw > 1) {
            Vec16<T> t = ld16(dy + src);
#pragma unroll
            for (int j = 0; j < Vec16<T>::N; ++j) acc[j] += t.get(j);
          } else {
            acc[0] += to_f(dy[src]);
          }
        }
    int64_t dst = (i / cpr) * g.C + (int64_t)c * cw;
    if (cw > 1) {
      Vec16<T> o;
#pragma unroll
      for (int j = 0; j < Vec16<T>::N; ++j) o.set(j, acc[j]);
      st16(dx + dst, o);
    } else {
      dx[dst] = from_f<T>(acc[0]);
    }
  }
}
template <typename T, bool BWD>
static int launch_upsample(const void* src, void* dst, int N, const int32_t* in_dims, const int32_t* f, int C,
                           void* stream) {
  UpGeom g{N, in_dims[0], in_dims[1], in_dims[2], f[0], f[1], f[2], C};
  MIG_REQUIRE(f[0] >= 1 && f[1] >= 1 && f[2] >= 1, "upsample: factors must be >= 1");
  constexpr int V = Vec16<T>::N;
  int cw = (C % V == 0 && aligned16(src) && aligned16(dst)) ? V : 1;
  int64_t vox = (int64_t)N * g.D * g.H * g.W * (BWD ? 1 : (int64_t)f[0] * f[1] * f[2]);
  if (vox == 0) return 0;
  int grid = bw_grid(vox * (C / cw), 256);
  if (BWD) upsample_bwd_kernel<T><<<grid, 256, 0, as_stream(stream)>>>((const T*)src, (T*)dst, g, cw);
  else upsample_fwd_kernel<T><<<grid, 256, 0, as_stream(stream)>>>((const T*)src, (T*)dst, g, cw);
  return check_launch(BWD ? "upsample_bwd" : "upsample_fwd");
}
}  // namespace mig

// ------------------------------------------------------------------------------------------------
// nn.AvgPool{2,3}d(kernel, stride), no padding -- Downsample(use_conv=False) inside ResnetBlock(down=True),
// unet:513-518,641-644 (resblock_updown). Channels-last, one thread per (voxel, 16-byte channel vector).
// ------------------------------------------------------------------------------------------------
namespace mig {
struct PoolGeom { int N, D, H, W, OD, OH, OW, kd, kh, kw, sd, sh, sw, C; };

template <typename T>
__global__ void __launch_bounds__(256) avgpool_fwd_kernel(const T* __restrict__ x, T* __restrict__ y, PoolGeom g, int cw) {
  const int cpr = g.C / cw;
  const int64_t total = (int64_t)g.N * g.OD * g.OH * g.OW * cpr;
  const float inv = 1.f / (float)(g.kd * g.kh * g.kw);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % cpr);
    int64_t v = i / cpr;
    const int ow = (int)(v % g.OW); v /= g.OW;
    const int oh = (int)(v % g.OH); v /= g.OH;
    const int od = (int)(v % g.OD);
    const int n = (int)(v / g.OD);
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int a = 0; a < g.kd; ++a)
      for (int b = 0; b < g.kh; ++b)
        for (int e = 0; e < g.kw; ++e) {
          const int64_t src = ((((int64_t)n * g.D + od * g.sd + a) * g.H + oh * g.sh + b) * g.W + ow * g.sw + e) * g.C +
                              (int64_t)c * cw;
          if (cw > 1) {
            const Vec16<T> t = ld16(x + src);
#pragma unroll
            for (int j = 0; j < Vec16<T>::N; ++j) acc[j] += t.get(j);
          } else {
            acc[0] += to_f(x[src]);
          }
        }
    const int64_t dst = (i / cpr) * g.C + (int64_t)c * cw;
    if (cw > 1) {
      Vec16<T> o;
#pragma unroll
      for (int j = 0; j < Vec16<T>::N; ++j) o.set(j, acc[j] * inv);
      st16(y + dst, o);
    } else {
      y[dst] = from_f<T>(acc[0] * inv);
    }
  }
}
// dx[i] = (1 / window) * sum of dy[o] over the output positions whose window contains i (gather: no atomics, windows
// may overlap when kernel > stride)
template <typename T>
__global__ void __launch_bounds__(256) avgpool_bwd_kernel(const T* __restrict__ dy, T* __restrict__ dx, PoolGeom g, int cw) {
  const int cpr = g.C / cw;
  const int64_t total = (int64_t)g.N * g.D * g.H * g.W * cpr;
  const float inv = 1.f / (float)(g.kd * g.kh * g.kw);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % cpr);
    int64_t v = i / cpr;
    const int w = (int)(v % g.W); v /= g.W;
    const int h = (int)(v % g.H); v /= g.H;
    const int d = (int)(v % g.D);
    const int n = (int)(v / g.D);
    auto lo = [](int p, int k, int s) { const int t = p - k + 1; return t <= 0 ? 0 : (t + s - 1) / s; };
    auto hi = [](int p, int s, int on) { const int t = p / s; return t < on - 1 ? t : on - 1; };
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int od = lo(d, g.kd, g.sd); od <= hi(d, g.sd, g.OD); ++od)
      for (int oh = lo(h, g.kh, g.sh); oh <= hi(h, g.sh, g.OH); ++oh)
        for (int ow = lo(w, g.kw, g.sw); ow <= hi(w, g.sw, g.OW); ++ow) {
          const int64_t src = ((((int64_t)n * g.OD + od) * g.OH + oh) * g.OW + ow) * g.C + (int64_t)c * cw;
          if (cw > 1) {
            const Vec16<T> t = ld16(dy + src);
#pragma unroll
            for (int j = 0; j < Vec16<T>::N; ++j) acc[j] += t.get(j);
          } else {
            acc[0] += to_f(dy[src]);
          }
        }
    const int64_t dst = (i / cpr) * g.C + (int64_t)c * cw;
    if (cw > 1) {
      Vec16<T> o;
#pragma unroll
      for (int j = 0; j < Vec16<T>::N; ++j) o.set(j, acc[j] * inv);
      st16(dx + dst, o);
    } else {
      dx[dst] = from_f<T>(acc[0] * inv);
    }
  }
}

template <typename T>
static int launch_avgpool(bool bwd, const void* a, void* b, int N, const int32_t* in_dims, const int32_t* ksize,
                          const int32_t* stride, int C, void* stream) {
  PoolGeom g;
  g.N = N; g.D = in_dims[0]; g.H = in_dims[1]; g.W = in_dims[2];
  g.kd = ksize[0]; g.kh = ksize[1]; g.kw = ksize[2];
  g.sd = stride[0]; g.sh = stride[1]; g.sw = stride[2];
  g.C = C;
  MIG_REQUIRE(g.kd >= 1 && g.kh >= 1 && g.kw >= 1 && g.sd >= 1 && g.sh >= 1 && g.sw >= 1, "avgpool: bad kernel / stride");
  MIG_REQUIRE(g.D >= g.kd && g.H >= g.kh && g.W >= g.kw, "avgpool: kernel larger than the input");
  g.OD = (g.D - g.kd) / g.sd + 1; g.OH = (g.H - g.kh) / g.sh + 1; g.OW = (g.W - g.kw) / g.sw + 1;
  const int V = Vec16<T>::N;
  const int cw = (C % V == 0 && aligned16(a) && aligned16(b)) ? V : 1;
  const int64_t items = (int64_t)N * (bwd ? (int64_t)g.D * g.H * g.W : (int64_t)g.OD * g.OH * g.OW) * (C / cw);
  if (items == 0) return 0;
  if (bwd) avgpool_bwd_kernel<T><<<bw_grid(items, 256), 256, 0, as_stream(stream)>>>((const T*)a, (T*)b, g, cw);
  else avgpool_fwd_kernel<T><<<bw_grid(items, 256), 256, 0, as_stream(stream)>>>((const T*)a, (T*)b, g, cw);
  return check_launch(bwd ? "avgpool_bwd" : "avgpool_fwd");
}
}  // namespace mig

extern "C" int mig_avgpool_fwd(int dtype, const void* x, void* y, int32_t N, const int32_t in_dims[3],
                               const int32_t ksize[3], const int32_t stride[3], int32_t C, void* stream) {
  MIG_REQUIRE(x && y && in_dims && ksize && stride, "avgpool_fwd: null argument");
  MIG_DISPATCH_DTYPE(dtype, T, return (launch_avgpool<T>(false, x, y, N, in_dims, ksize, stride, C, stream)));
}
extern "C" int mig_avgpool_bwd(int dtype, const void* dy, void* dx, int32_t N, const int32_t in_dims[3],
                               const int32_t ksize[3], const int32_t stride[3], int32_t C, void* stream) {
  MIG_REQUIRE(dy && dx && in_dims && ksize && stride, "avgpool_bwd: null argument");
  MIG_DISPATCH_DTYPE(dtype, T, return (launch_avgpool<T>(true, dy, dx, N, in_dims, ksize, stride, C, stream)));
}

extern "C" int mig_upsample_nearest_fwd(int dtype, const void* x, void* y, int32_t N, const int32_t in_dims[3],
                                        const int32_t factors[3], int32_t C, void* stream) {
  MIG_DISPATCH_DTYPE(dtype, T, return (launch_upsample<T, false>(x, y, N, in_dims, factors, C, stream)));
}
extern "C" int mig_upsample_nearest_bwd(int dtype, const void* dy, void* dx, int32_t N, const int32_t in_dims[3],
                                        const int32_t factors[3], int32_t C, void* stream) {
  MIG_DISPATCH_DTYPE(dtype, T, return (launch_upsample<T, true>(dy, dx, N, in_dims, factors, C, stream)));
}

// ------------------------------------------------------------------------------------------------
// NCDHW <-> NDHWC transposes through a padded smem tile (coalesced on both sides)
// ------------------------------------------------------------------------------------------------
namespace mig {
// src viewed as [B][R][Ccols] row-major -> dst [B][Ccols][R]
template <typename TS, typename TD>
__global__ void __launch_bounds__(256) transpose_kernel(const TS* __restrict__ x, TD* __restrict__ y, int64_t R,
                                                        int64_t Ccols) {
  __shared__ float tile[32][33];
  const int64_t b = blockIdx.z;
  const int64_t r0 = (int64_t)blockIdx.y * 32, c0 = (int64_t)blockIdx.x * 32;
  const TS* xs = x + b * R * Ccols;
  TD* yd = y + b * R * Ccols;
  for (int i = threadIdx.y; i < 32; i += 8) {
    int64_t r = r0 + i, c = c0 + threadIdx.x;
    if (r < R && c < Ccols) tile[i][threadIdx.x] = to_f(xs[r * Ccols + c]);
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    int64_t c = c0 + i, r = r0 + threadIdx.x;
    if (r < R && c < Ccols) yd[c * R + r] = from_f<TD>(tile[threadIdx.x][i]);
  }
}
template <typename TS, typename TD>
static int launch_transpose(const void* x, void* y, int B, int64_t R, int64_t Ccols, void* stream) {
  if (B * R * Ccols == 0) return 0;
  MIG_REQUIRE((R + 31) / 32 < 65536, "transpose: too many row tiles");
  dim3 grid((unsigned)((Ccols + 31) / 32), (unsigned)((R + 31) / 32), (unsigned)B), block(32, 8);
  transpose_kernel<TS, TD><<<grid, block, 0, as_stream(stream)>>>((const TS*)x, (TD*)y, R, Ccols);
  return check_launch("transpose");
}
static int transpose_dispatch(int sd, int dd, const void* x, void* y, int B, int64_t R, int64_t Cc, void* stream) {
  if (sd == MIG_F32 && dd == MIG_F32) return launch_transpose<float, float>(x, y, B, R, Cc, stream);
  if (sd == MIG_F32 && dd == MIG_BF16) return launch_transpose<float, __nv_bfloat16>(x, y, B, R, Cc, stream);
  if (sd == MIG_BF16 && dd == MIG_F32) return launch_transpose<__nv_bfloat16, float>(x, y, B, R, Cc, stream);
  if (sd == MIG_BF16 && dd == MIG_BF16) return launch_transpose<__nv_bfloat16, __nv_bfloat16>(x, y, B, R, Cc, stream);
  set_error("transpose: bad dtypes");
  return 1;
}
}  // namespace mig

extern "C" int mig_nchw_to_nhwc(int src_dtype, int dst_dtype, const void* x, void* y, int32_t N, int32_t C, int64_t S,
                                void* stream) {
  // y is only 65535-limited in grid.y = C tiles; put the long axis (S) on grid.x
  return transpose_dispatch(src_dtype, dst_dtype, x, y, N, C, S, stream);
}
extern "C" int mig_nhwc_to_nchw(int src_dtype, int dst_dtype, const void* x, void* y, int32_t N, int32_t C, int64_t S,
                                void* stream) {
  // [N][S][C] -> [N][C][S]; rows = S may exceed 65535*32 only for > 2M voxels per sample
  if ((S + 31) / 32 >= 65536) {
    set_error("nhwc_to_nchw: sample too large for the transposing grid (S=%lld)", (long long)S);
    return 1;
  }
  return transpose_dispatch(src_dtype, dst_dtype, x, y, N, S, C, stream);
}

// ------------------------------------------------------------------------------------------------
// column sums (bias gradients) and per-(n,c) sums (time-embedding gradient)
// ------------------------------------------------------------------------------------------------
namespace mig {
// out[b][c] (+)= sum_{r in [0,R)} x[b][r][c]; grid (ceil(C/32), chunks, B); block (32, 8)
template <typename T>
__global__ void __launch_bounds__(256) colsum_kernel(const T* __restrict__ x, float* __restrict__ out, int64_t R,
                                                     int C) {
  __shared__ float red[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int64_t b = blockIdx.z;
  const T* xs = x + b * R * C;
  float acc = 0.f;
  if (c < C)
    for (int64_t r = (int64_t)blockIdx.y * 8 + threadIdx.y; r < R; r += (int64_t)gridDim.y * 8) acc += to_f(xs[r * C + c]);
  red[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x];
    atomicAdd(out + b * C + c, t);
  }
}
// Vector path (C a multiple of the 16-byte vector width): a thread owns one 16-byte column vector and walks down rows
// with four independent loads in flight; the thread rows of a CTA are merged through shared memory, then one atomic per
// (CTA, column). grid (slabs, chunks, B), block cvb*rpb <= 256.
template <typename T>
__global__ void __launch_bounds__(256) colsum_vec_kernel(const T* __restrict__ x, float* __restrict__ out, int64_t R, int C,
                                                         int cvb, int rpb, int64_t rows_per_cta) {
  constexpr int V = Vec16<T>::N;
  __shared__ float red[256 * V];
  const int cv = C / V;
  const int tcol = threadIdx.x % cvb, trow = threadIdx.x / cvb;
  const int col = blockIdx.x * cvb + tcol;
  const bool active = col < cv && trow < rpb;
  float s[V];
#pragma unroll
  for (int j = 0; j < V; ++j) s[j] = 0.f;
  if (active) {
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_cta;
    const int64_t r1 = r0 + rows_per_cta < R ? r0 + rows_per_cta : R;
    const T* base = x + (int64_t)blockIdx.z * R * C + (int64_t)col * V;
    int64_t r = r0 + trow;
    const int64_t step = rpb;
    for (; r + 3 * step < r1; r += 4 * step) {
      Vec16<T> v0 = ld16(base + r * C), v1 = ld16(base + (r + step) * C), v2 = ld16(base + (r + 2 * step) * C),
               v3 = ld16(base + (r + 3 * step) * C);
#pragma unroll
      for (int j = 0; j < V; ++j) s[j] += (v0.get(j) + v1.get(j)) + (v2.get(j) + v3.get(j));
    }
    for (; r < r1; r += step) {
      Vec16<T> v = ld16(base + r * C);
#pragma unroll
      for (int j = 0; j < V; ++j) s[j] += v.get(j);
    }
  }
#pragma unroll
  for (int j = 0; j < V; ++j) red[j * 256 + threadIdx.x] = s[j];
  __syncthreads();
  for (int e = threadIdx.x; e < cvb * V; e += blockDim.x) {
    const int j = e / cvb, tc = e - j * cvb;
    const int ccol = blockIdx.x * cvb + tc;
    if (ccol >= cv) continue;
    float t = 0.f;
    for (int rr = 0; rr < rpb; ++rr) t += red[j * 256 + rr * cvb + tc];
    atomicAdd(out + (int64_t)blockIdx.z * C + ccol * V + j, t);
  }
}
// Few columns (C <= 8, e.g. the 1/2/3-channel ends): one thread per row, consecutive threads read consecutive rows.
template <typename T>
__global__ void __launch_bounds__(256) colsum_thin_kernel(const T* __restrict__ x, float* __restrict__ out, int64_t R,
                                                          int C) {
  __shared__ float red[8][8];
  const T* xs = x + (int64_t)blockIdx.z * R * C;
  float s[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = 0.f;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; r + 3 * stride < R; r += 4 * stride) {
    float a[4][8];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int j = 0; j < 8; ++j) a[u][j] = j < C ? to_f(xs[(r + u * stride) * C + j]) : 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] += (a[0][j] + a[1][j]) + (a[2][j] + a[3][j]);
  }
  for (; r < R; r += stride)
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] += j < C ? to_f(xs[r * C + j]) : 0.f;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float v = s[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp][j] = v;
  }
  __syncthreads();
  if (threadIdx.x < C) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[w][threadIdx.x];
    atomicAdd(out + (int64_t)blockIdx.z * C + threadIdx.x, t);
  }
}
template <typename T>
static int launch_colsum(const void* x, float* out, int B, int64_t R, int C, int accumulate, void* stream) {
  if (!accumulate) cudaMemsetAsync(out, 0, sizeof(float) * (size_t)B * C, as_stream(stream));
  if (B * R * C == 0) return 0;
  constexpr int V = Vec16<T>::N;
  const int64_t target = (int64_t)device_info().sm_count * 4;
  if (C % V == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0) {
    // 4 column vectors (64 B of a row) per CTA: the CTA count that saturates HBM then issues 32..64 atomics each,
    // not one per column of the whole row
    const int cv = C / V, cvb = cv < 4 ? cv : 4, rpb = 256 / cvb, slabs = (cv + cvb - 1) / cvb;
    int64_t chunks = target / ((int64_t)B * slabs);
    if (chunks < 1) chunks = 1;
    int64_t rows = (R + chunks - 1) / chunks;
    if (rows < (int64_t)rpb * 4) rows = (int64_t)rpb * 4;
    chunks = (R + rows - 1) / rows;
    if (chunks <= 65535) {
      dim3 grid(slabs, (unsigned)chunks, B);
      colsum_vec_kernel<T><<<grid, cvb * rpb, 0, as_stream(stream)>>>((const T*)x, out, R, C, cvb, rpb, rows);
      return check_launch("colsum_vec");
    }
  }
  if (C <= 8) {
    int64_t blocks = (R + 256 * 8 - 1) / (256 * 8);
    if (blocks > target) blocks = target;
    if (blocks < 1) blocks = 1;
    dim3 grid((unsigned)blocks, 1, B);
    colsum_thin_kernel<T><<<grid, 256, 0, as_stream(stream)>>>((const T*)x, out, R, C);
    return check_launch("colsum_thin");
  }
  int ctiles = (C + 31) / 32;
  int64_t want = (int64_t)device_info().sm_count * 4 / (ctiles * (int64_t)B) + 1;
  int64_t maxchunks = (R + 7) / 8;
  int chunks = (int)(want < maxchunks ? want : maxchunks);
  if (chunks < 1) chunks = 1;
  if (chunks > 65535) chunks = 65535;
  dim3 grid(ctiles, chunks, B), block(32, 8);
  colsum_kernel<T><<<grid, block, 0, as_stream(stream)>>>((const T*)x, out, R, C);
  return check_launch("colsum");
}
}  // namespace mig

extern "C" int mig_colsum(int dtype, const void* x, float* out, int64_t rows, int32_t C, int accumulate, void* stream) {
  MIG_DISPATCH_DTYPE(dtype, T, return (launch_colsum<T>(x, out, 1, rows, C, accumulate, stream)));
}
extern "C" int mig_chan_bias_bwd(int dtype, const void* dy, float* db, int32_t N, int64_t S, int32_t C, void* stream) {
  MIG_DISPATCH_DTYPE(dtype, T, return (launch_colsum<T>(dy, db, N, S, C, 0, stream)));
}

// ------------------------------------------------------------------------------------------------
// row softmax (fp32 math) forward / backward. One CTA per row; rows up to a few thousand columns.
// ------------------------------------------------------------------------------------------------
namespace mig {
template <typename TI, typename TO>
__global__ void __launch_bounds__(256) softmax_fwd_kernel(const TI* __restrict__ x, TO* __restrict__ y, int cols,
                                                          float scale) {
  __shared__ float red[33];
  const TI* xr = x + (int64_t)blockIdx.x * cols;
  TO* yr = y + (int64_t)blockIdx.x * cols;
  float mx = -INFINITY;
  for (int c = threadIdx.x; c < cols; c += blockDim.x) mx = fmaxf(mx, to_f(xr[c]) * scale);
  mx = block_max(mx, red);
  float sum = 0.f;
  for (int c = threadIdx.x; c < cols; c += blockDim.x) sum += __expf(to_f(xr[c]) * scale - mx);
  sum = block_sum(sum, red);
  const float inv = 1.f / sum;
  for (int c = threadIdx.x; c < cols; c += blockDim.x) yr[c] = from_f<TO>(__expf(to_f(xr[c]) * scale - mx) * inv);
}
// Rows of up to 256 * kSoftmaxVPT columns (the LDM's L = 1728 attention rows): the row is loaded ONCE, all loads in
// flight together, and lives in registers for the maximum, the sum and the store -- the three-pass kernel above re-read
// it twice through L1 and evaluated every exponential twice (0.29 of HBM on the 8 x 1728 x 1728 score matrix).
constexpr int kSoftmaxVPT = 8;
template <typename TI, typename TO>
__global__ void __launch_bounds__(256) softmax_fwd_row_kernel(const TI* __restrict__ x, TO* __restrict__ y, int cols,
                                                              float scale) {
  __shared__ float red[33];
  const TI* xr = x + (int64_t)blockIdx.x * cols;
  TO* yr = y + (int64_t)blockIdx.x * cols;
  float v[kSoftmaxVPT];
#pragma unroll
  for (int k = 0; k < kSoftmaxVPT; ++k) {
    const int c = threadIdx.x + k * 256;
    v[k] = c < cols ? to_f(xr[c]) * scale : -INFINITY;
  }
  float mx = v[0];
#pragma unroll
  for (int k = 1; k < kSoftmaxVPT; ++k) mx = fmaxf(mx, v[k]);
  mx = block_max(mx, red);
  float sum = 0.f;
#pragma unroll
  for (int k = 0; k < kSoftmaxVPT; ++k) {
    v[k] = __expf(v[k] - mx);     // exp(-inf) = 0 for the columns past the end
    sum += v[k];
  }
  sum = block_sum(sum, red);
  const float inv = 1.f / sum;
#pragma unroll
  for (int k = 0; k < kSoftmaxVPT; ++k) {
    const int c = threadIdx.x + k * 256;
    if (c < cols) yr[c] = from_f<TO>(v[k] * inv);
  }
}
template <typename TP, typename TD, typename TS = TD>
__global__ void __launch_bounds__(256) softmax_bwd_row_kernel(const TP* __restrict__ p, const TD* __restrict__ dp,
                                                              TS* __restrict__ ds, int cols, float scale) {
  __shared__ float red[33];
  const TP* pr = p + (int64_t)blockIdx.x * cols;
  const TD* dr = dp + (int64_t)blockIdx.x * cols;
  TS* sr = ds + (int64_t)blockIdx.x * cols;
  float pv[kSoftmaxVPT], dv[kSoftmaxVPT];
#pragma unroll
  for (int k = 0; k < kSoftmaxVPT; ++k) {
    const int c = threadIdx.x + k * 256;
    pv[k] = c < cols ? to_f(pr[c]) : 0.f;
    dv[k] = c < cols ? to_f(dr[c]) : 0.f;
  }
  float dot = 0.f;
#pragma unroll
  for (int k = 0; k < kSoftmaxVPT; ++k) dot = fmaf(pv[k], dv[k], dot);
  dot = block_sum(dot, red);
#pragma unroll
  for (int k = 0; k < kSoftmaxVPT; ++k) {
    const int c = threadIdx.x + k * 256;
    if (c < cols) sr[c] = from_f<TS>(scale * pv[k] * (dv[k] - dot));
  }
}
// ds = scale * p * (dp - sum(dp*p))
template <typename TP, typename TD, typename TS = TD>
__global__ void __launch_bounds__(256) softmax_bwd_kernel(const TP* __restrict__ p, const TD* __restrict__ dp,
                                                          TS* __restrict__ ds, int cols, float scale) {
  __shared__ float red[33];
  const TP* pr = p + (int64_t)blockIdx.x * cols;
  const TD* dr = dp + (int64_t)blockIdx.x * cols;
  TS* sr = ds + (int64_t)blockIdx.x * cols;
  float dot = 0.f;
  for (int c = threadIdx.x; c < cols; c += blockDim.x) dot += to_f(pr[c]) * to_f(dr[c]);
  dot = block_sum(dot, red);
  for (int c = threadIdx.x; c < cols; c += blockDim.x)
    sr[c] = from_f<TS>(scale * to_f(pr[c]) * (to_f(dr[c]) - dot));
}
}  // namespace mig

extern "C" int mig_softmax_fwd(int dtype_in, int dtype_out, const void* x, void* y, int64_t rows, int32_t cols,
                               float scale, void* stream) {
  if (rows <= 0 || cols <= 0) return 0;
  MIG_REQUIRE(rows < (1ll << 31), "softmax: too many rows");
  cudaStream_t s = as_stream(stream);
  const bool row = cols <= 256 * kSoftmaxVPT;     // the whole row fits the registers of one CTA
#define MIG_SOFTMAX_FWD(TI, TO)                                                                               \
  do {                                                                                                        \
    if (row) softmax_fwd_row_kernel<TI, TO><<<(unsigned)rows, 256, 0, s>>>((const TI*)x, (TO*)y, cols, scale); \
    else softmax_fwd_kernel<TI, TO><<<(unsigned)rows, 256, 0, s>>>((const TI*)x, (TO*)y, cols, scale);         \
  } while (0)
  if (dtype_in == MIG_F32 && dtype_out == MIG_F32) MIG_SOFTMAX_FWD(float, float);
  else if (dtype_in == MIG_F32 && dtype_out == MIG_BF16) MIG_SOFTMAX_FWD(float, __nv_bfloat16);
  else if (dtype_in == MIG_BF16 && dtype_out == MIG_BF16) MIG_SOFTMAX_FWD(__nv_bfloat16, __nv_bfloat16);
  else
    MIG_REQUIRE(false, "softmax_fwd: unsupported dtype pair %d -> %d", dtype_in, dtype_out);
#undef MIG_SOFTMAX_FWD
  return check_launch("softmax_fwd");
}
extern "C" int mig_softmax_bwd(int dtype_p, int dtype_d, const void* p, const void* dp, void* ds, int64_t rows,
                               int32_t cols, float scale, void* stream) {
  if (rows <= 0 || cols <= 0) return 0;
  cudaStream_t s = as_stream(stream);
  const bool row = cols <= 256 * kSoftmaxVPT;
#define MIG_SOFTMAX_BWD(TP, TD)                                                                                          \
  do {                                                                                                                   \
    if (row) softmax_bwd_row_kernel<TP, TD><<<(unsigned)rows, 256, 0, s>>>((const TP*)p, (const TD*)dp, (TD*)ds, cols, scale); \
    else softmax_bwd_kernel<TP, TD><<<(unsigned)rows, 256, 0, s>>>((const TP*)p, (const TD*)dp, (TD*)ds, cols, scale);         \
  } while (0)
  if (dtype_p == MIG_F32 && dtype_d == MIG_F32) MIG_SOFTMAX_BWD(float, float);
  else if (dtype_p == MIG_BF16 && dtype_d == MIG_F32) MIG_SOFTMAX_BWD(__nv_bfloat16, float);
  else if (dtype_p == MIG_BF16 && dtype_d == MIG_BF16) MIG_SOFTMAX_BWD(__nv_bfloat16, __nv_bfloat16);
  else
    MIG_REQUIRE(false, "softmax_bwd: unsupported dtype pair %d / %d", dtype_p, dtype_d);
#undef MIG_SOFTMAX_BWD
  return check_launch("softmax_bwd");
}

// bf16 probabilities, fp32 dP (the GEMM's accumulator precision) -> bf16 dS in ONE pass: what the bf16 training chain
// feeds its dQ / dK GEMMs (the fp32 dS round trip + cast pass cost 190 MB of traffic per attention block)
extern "C" int mig_softmax_bwd_narrow(const void* p, const void* dp, void* ds, int64_t rows, int32_t cols, float scale,
                                      void* stream) {
  if (rows <= 0 || cols <= 0) return 0;
  MIG_REQUIRE(p && dp && ds && rows < (1ll << 31), "softmax_bwd_narrow: bad arguments");
  cudaStream_t s = as_stream(stream);
  if (cols <= 256 * kSoftmaxVPT)
    softmax_bwd_row_kernel<__nv_bfloat16, float, __nv_bfloat16><<<(unsigned)rows, 256, 0, s>>>(
        (const __nv_bfloat16*)p, (const float*)dp, (__nv_bfloat16*)ds, cols, scale);
  else
    softmax_bwd_kernel<__nv_bfloat16, float, __nv_bfloat16><<<(unsigned)rows, 256, 0, s>>>(
        (const __nv_bfloat16*)p, (const float*)dp, (__nv_bfloat16*)ds, cols, scale);
  return check_launch("softmax_bwd_narrow");
}

// ------------------------------------------------------------------------------------------------
// timestep embedding: out[b][j] = cos(t*f_j) for j < half, sin(t*f_{j-half}) for half <= j < 2*half, 0 pad
// ------------------------------------------------------------------------------------------------
namespace mig {
template <typename T>
__global__ void temb_kernel(const float* __restrict__ t, T* __restrict__ out, int B, int dim, float log_period) {
  const int half = dim / 2;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B * dim; i += gridDim.x * blockDim.x) {
    int b = i / dim, j = i - b * dim;
    float v = 0.f;
    if (j < 2 * half) {
      int k = j < half ? j : j - half;
      // same op order as the reference: exp(-log(P) * k / half), then t * f  (unet:479-481)
      float f = expf((-log_period * (float)k) / (float)half);
      float a = t[b] * f;
      v = j < half ? cosf(a) : sinf(a);
    }
    out[i] = from_f<T>(v);
  }
}
}  // namespace mig

extern "C" int mig_timestep_embedding(const float* t, void* out, int out_dtype, int32_t B, int32_t dim,
                                      float max_period, void* stream) {
  if (B * dim <= 0) return 0;
  float lp = logf(max_period);
  MIG_DISPATCH_DTYPE(out_dtype, T, (temb_kernel<T><<<bw_grid((int64_t)B * dim, 256), 256, 0, as_stream(stream)>>>(
                                       t, (T*)out, B, dim, lp)));
  return check_launch("timestep_embedding");
}

// ------------------------------------------------------------------------------------------------
// DDPM scheduler kernels
// ------------------------------------------------------------------------------------------------
namespace mig {
// grid.y = sample index; coefficients gathered once per CTA (bit-exact indexing: acp[t[b]])
template <typename T>
__global__ void __launch_bounds__(256) add_noise_kernel(const T* __restrict__ x0, const T* __restrict__ noise,
                                                        const int64_t* __restrict__ ts,
                                                        const float* __restrict__ acp, T* __restrict__ out,
                                                        int64_t per, int Tn, int velocity, int vec) {
  constexpr int V = Vec16<T>::N;
  const int b = blockIdx.y;
  int64_t t = ts[b];
  t = t < 0 ? 0 : (t >= Tn ? Tn - 1 : t);
  // the reference casts the table to the sample dtype before the sqrt (scheduler.add_noise)
  const float a_tab = to_f(from_f<T>(acp[t]));
  const float ca = to_f(from_f<T>(sqrtf(a_tab)));
  const float cb = to_f(from_f<T>(sqrtf(to_f(from_f<T>(1.f - a_tab)))));
  const T* xs = x0 + (int64_t)b * per;
  const T* ns = noise + (int64_t)b * per;
  T* os = out + (int64_t)b * per;
  const int64_t nvec = vec ? per / V : 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    Vec16<T> vx = ld16_stream(xs + i * V), vn = ld16_stream(ns + i * V), vo;
#pragma unroll
    for (int j = 0; j < V; ++j)
      vo.set(j, velocity ? ca * vn.get(j) - cb * vx.get(j) : ca * vx.get(j) + cb * vn.get(j));
    st16(os + i * V, vo);
  }
  for (int64_t i = nvec * V + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < per;
       i += (int64_t)gridDim.x * blockDim.x) {
    float x = to_f(xs[i]), n = to_f(ns[i]);
    os[i] = from_f<T>(velocity ? ca * n - cb * x : ca * x + cb * n);
  }
}

struct StepCoef { float sa, sb, c0, ct, sigma; int prediction, clip; };
template <typename T>
__global__ void __launch_bounds__(256) ddpm_step_kernel(const T* __restrict__ eps, const T* __restrict__ x,
                                                        const T* __restrict__ z, T* __restrict__ prev,
                                                        T* __restrict__ x0_out, int64_t n, StepCoef k, int vec) {
  constexpr int V = Vec16<T>::N;
  const int64_t nvec = vec ? n / V : 0;
  auto f = [&](float e, float xv, float zv, float& x0) {
    if (k.prediction == 0) x0 = (xv - k.sb * e) / k.sa;
    else if (k.prediction == 1) x0 = e;
    else x0 = k.sa * xv - k.sb * e;
    if (k.clip) x0 = fminf(fmaxf(x0, -1.f), 1.f);
    return k.c0 * x0 + k.ct * xv + k.sigma * zv;
  };
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    Vec16<T> ve = ld16_stream(eps + i * V), vx = ld16_stream(x + i * V), vz, vp, v0;
    if (z) vz = ld16_stream(z + i * V);
#pragma unroll
    for (int j = 0; j < V; ++j) {
      float x0;
      vp.set(j, f(ve.get(j), vx.get(j), z ? vz.get(j) : 0.f, x0));
      v0.set(j, x0);
    }
    st16(prev + i * V, vp);
    if (x0_out) st16(x0_out + i * V, v0);
  }
  for (int64_t i = nvec * V + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    float x0;
    prev[i] = from_f<T>(f(to_f(eps[i]), to_f(x[i]), z ? to_f(z[i]) : 0.f, x0));
    if (x0_out) x0_out[i] = from_f<T>(x0);
  }
}

// DDIM (Song et al.): prev = ap*clamp(x0) + dir*eps + sigma*z. Unlike ddpm_step, eps enters as its own term and is
// derived from the UNCLIPPED x0, so the clipped and unclipped predictions are both live and no (c0, ct) pair of the
// DDPM posterior can express it. Also serves the inversion step (sigma = 0, ap/dir of the next timestep).
struct DdimCoef { float sa, sb, ap, dir, sigma; int prediction, clip; };
template <typename T>
__global__ void __launch_bounds__(256) ddim_step_kernel(const T* __restrict__ m, const T* __restrict__ x,
                                                        const T* __restrict__ z, T* __restrict__ prev,
                                                        T* __restrict__ x0_out, int64_t n, DdimCoef k, int vec) {
  constexpr int V = Vec16<T>::N;
  const int64_t nvec = vec ? n / V : 0;
  auto f = [&](float mv, float xv, float zv, float& x0) {
    float eps;
    if (k.prediction == 0) { x0 = (xv - k.sb * mv) / k.sa; eps = mv; }
    else if (k.prediction == 1) { x0 = mv; eps = (xv - k.sa * x0) / k.sb; }
    else { x0 = k.sa * xv - k.sb * mv; eps = k.sa * mv + k.sb * xv; }
    if (k.clip) x0 = fminf(fmaxf(x0, -1.f), 1.f);
    return k.ap * x0 + k.dir * eps + k.sigma * zv;
  };
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    Vec16<T> vm = ld16_stream(m + i * V), vx = ld16_stream(x + i * V), vz, vp, v0;
    if (z) vz = ld16_stream(z + i * V);
#pragma unroll
    for (int j = 0; j < V; ++j) {
      float x0;
      vp.set(j, f(vm.get(j), vx.get(j), z ? vz.get(j) : 0.f, x0));
      v0.set(j, x0);
    }
    st16(prev + i * V, vp);
    if (x0_out) st16(x0_out + i * V, v0);
  }
  for (int64_t i = nvec * V + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    float x0;
    prev[i] = from_f<T>(f(to_f(m[i]), to_f(x[i]), z ? to_f(z[i]) : 0.f, x0));
    if (x0_out) x0_out[i] = from_f<T>(x0);
  }
}
}  // namespace mig

extern "C" int mig_ddpm_add_noise(int dtype, const void* x0, const void* noise, const int64_t* timesteps,
                                  const float* alphas_cumprod, void* out, int32_t B, int64_t per_sample, int32_t T,
                                  int velocity, void* stream) {
  if (B <= 0 || per_sample <= 0) return 0;
  MIG_REQUIRE(B < 65536, "add_noise: batch too large");
  MIG_DISPATCH_DTYPE(dtype, TT, {
    constexpr int V = Vec16<TT>::N;
    int vec = aligned16(x0) && aligned16(noise) && aligned16(out) && (per_sample % V == 0);
    int gx = bw_grid((per_sample + V - 1) / V, 256, 8) / B + 1;
    dim3 grid(gx, B);
    add_noise_kernel<TT><<<grid, 256, 0, as_stream(stream)>>>((const TT*)x0, (const TT*)noise, timesteps, alphas_cumprod,
                                                            (TT*)out, per_sample, T, velocity, vec);
  });
  return check_launch("ddpm_add_noise");
}

extern "C" int mig_ddpm_step(int dtype, const void* model_out, const void* x, const void* z, void* prev, void* x0_hat,
                             int64_t n, float sqrt_acp_t, float sqrt_one_minus_acp_t, float c0, float ct, float sigma,
                             int prediction, int clip, void* stream) {
  if (n <= 0) return 0;
  MIG_REQUIRE(z != nullptr || sigma == 0.f, "ddpm_step: noise buffer required when sigma != 0");
  StepCoef k{sqrt_acp_t, sqrt_one_minus_acp_t, c0, ct, sigma, prediction, clip};
  MIG_DISPATCH_DTYPE(dtype, TT, {
    constexpr int V = Vec16<TT>::N;
    int vec = aligned16(model_out) && aligned16(x) && aligned16(prev) && (!z || aligned16(z)) &&
              (!x0_hat || aligned16(x0_hat));
    ddpm_step_kernel<TT><<<bw_grid((n + V - 1) / V, 256), 256, 0, as_stream(stream)>>>(
        (const TT*)model_out, (const TT*)x, (const TT*)z, (TT*)prev, (TT*)x0_hat, n, k, vec);
  });
  return check_launch("ddpm_step");
}

extern "C" int mig_ddim_step(int dtype, const void* model_out, const void* x, const void* z, void* prev, void* x0_hat,
                             int64_t n, float sqrt_acp_t, float sqrt_one_minus_acp_t, float sqrt_acp_prev,
                             float dir_coef, float sigma, int prediction, int clip, void* stream) {
  if (n <= 0) return 0;
  MIG_REQUIRE(z != nullptr || sigma == 0.f, "ddim_step: noise buffer required when sigma != 0");
  MIG_REQUIRE(prediction >= 0 && prediction <= 2, "ddim_step: prediction must be 0, 1 or 2");
  DdimCoef k{sqrt_acp_t, sqrt_one_minus_acp_t, sqrt_acp_prev, dir_coef, sigma, prediction, clip};
  MIG_DISPATCH_DTYPE(dtype, TT, {
    constexpr int V = Vec16<TT>::N;
    int vec = aligned16(model_out) && aligned16(x) && aligned16(prev) && (!z || aligned16(z)) &&
              (!x0_hat || aligned16(x0_hat));
    ddim_step_kernel<TT><<<bw_grid((n + V - 1) / V, 256), 256, 0, as_stream(stream)>>>(
        (const TT*)model_out, (const TT*)x, (const TT*)z, (TT*)prev, (TT*)x0_hat, n, k, vec);
  });
  return check_launch("ddim_step");
}

// ------------------------------------------------------------------------------------------------
// losses
// ------------------------------------------------------------------------------------------------
namespace mig {
constexpr int kLossBlocks = 1024;

template <typename T, int MODE>  // MODE 0: (a-b)^2, 1: |a-b|, 2: KL term of (mu=a, sigma=b)
__global__ void __launch_bounds__(256) loss_partial_kernel(const T* __restrict__ a, const T* __restrict__ b,
                                                           float* __restrict__ partials, int64_t n, int vec) {
  __shared__ float red[33];
  constexpr int V = Vec16<T>::N;
  const int64_t nvec = vec ? n / V : 0;
  float acc = 0.f;
  auto term = [](float x, float y) {
    if (MODE == 0) { float d = x - y; return d * d; }
    if (MODE == 1) return fabsf(x - y);
    float s2 = y * y;
    return 0.5f * (x * x + s2 - logf(s2) - 1.f);
  };
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    Vec16<T> va = ld16_stream(a + i * V), vb = ld16_stream(b + i * V);
#pragma unroll
    for (int j = 0; j < V; ++j) acc += term(va.get(j), vb.get(j));
  }
  for (int64_t i = nvec * V + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    acc += term(to_f(a[i]), to_f(b[i]));
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) partials[blockIdx.x] = acc;
}
// deterministic second stage: one CTA sums the partials in double
__global__ void loss_final_kernel(const float* __restrict__ partials, int nparts, float* __restrict__ out,
                                  double inv_count) {
  __shared__ double red[256];
  double acc = 0.0;
  for (int i = threadIdx.x; i < nparts; i += blockDim.x) acc += (double)partials[i];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = (float)(red[0] * inv_count);
}
template <typename T, int MODE>
static int launch_loss(const void* a, const void* b, float* out, float* partials, int64_t n, double inv_count,
                       void* stream) {
  MIG_REQUIRE(n > 0, "loss: empty input");
  constexpr int V = Vec16<T>::N;
  int vec = aligned16(a) && aligned16(b);
  int grid = bw_grid((n + V - 1) / V, 256, 4);
  if (grid > kLossBlocks) grid = kLossBlocks;
  loss_partial_kernel<T, MODE><<<grid, 256, 0, as_stream(stream)>>>((const T*)a, (const T*)b, partials, n, vec);
  loss_final_kernel<<<1, 256, 0, as_stream(stream)>>>(partials, grid, out, inv_count);
  return check_launch("loss_fwd");
}

template <typename T, int MODE>
__global__ void __launch_bounds__(256) loss_bwd_kernel(const T* __restrict__ a, const T* __restrict__ b,
                                                       const float* __restrict__ gscale, T* __restrict__ da,
                                                       T* __restrict__ db, int64_t n, float k) {
  const float g = gscale[0] * k;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float x = to_f(a[i]), y = to_f(b[i]);
    if (MODE == 0) {
      da[i] = from_f<T>(2.f * (x - y) * g);
    } else if (MODE == 1) {
      float d = x - y;
      da[i] = from_f<T>((d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f)) * g);
    } else {  // KL: d/dmu = mu ; d/dsigma = sigma - 1/sigma
      da[i] = from_f<T>(x * g);
      db[i] = from_f<T>((y - 1.f / y) * g);
    }
  }
}
}  // namespace mig

extern "C" int mig_mse_fwd(int dtype, const void* a, const void* b, float* out, float* partials, int64_t n, int l1,
                           void* stream) {
  MIG_DISPATCH_DTYPE(dtype, T, {
    if (l1) return (launch_loss<T, 1>(a, b, out, partials, n, 1.0 / (double)n, stream));
    return (launch_loss<T, 0>(a, b, out, partials, n, 1.0 / (double)n, stream));
  });
}
extern "C" int mig_mse_bwd(int dtype, const void* a, const void* b, const float* gscale, void* da, int64_t n, int l1,
                           void* stream) {
  if (n <= 0) return 0;
  MIG_DISPATCH_DTYPE(dtype, T, {
    int grid = bw_grid(n, 256);
    if (l1) loss_bwd_kernel<T, 1><<<grid, 256, 0, as_stream(stream)>>>((const T*)a, (const T*)b, gscale, (T*)da, nullptr, n, 1.f / (float)n);
    else loss_bwd_kernel<T, 0><<<grid, 256, 0, as_stream(stream)>>>((const T*)a, (const T*)b, gscale, (T*)da, nullptr, n, 1.f / (float)n);
  });
  return check_launch("mse_bwd");
}
extern "C" int mig_kl_fwd(int dtype, const void* mu, const void* sigma, float* out, float* partials, int64_t n,
                          int32_t B, void* stream) {
  MIG_REQUIRE(B > 0, "kl: batch must be positive");
  MIG_DISPATCH_DTYPE(dtype, T, return (launch_loss<T, 2>(mu, sigma, out, partials, n, 1.0 / (double)B, stream)));
}
extern "C" int mig_kl_bwd(int dtype, const void* mu, const void* sigma, const float* gscale, void* dmu, void* dsigma,
                          int64_t n, int32_t B, void* stream) {
  if (n <= 0) return 0;
  MIG_DISPATCH_DTYPE(dtype, T, (loss_bwd_kernel<T, 2><<<bw_grid(n, 256), 256, 0, as_stream(stream)>>>(
                                   (const T*)mu, (const T*)sigma, gscale, (T*)dmu, (T*)dsigma, n, 1.f / (float)B)));
  return check_launch("kl_bwd");
}

// ------------------------------------------------------------------------------------------------
// VAE reparameterisation tail
// ------------------------------------------------------------------------------------------------
namespace mig {
template <typename T>
__global__ void vae_sample_fwd_kernel(const T* __restrict__ mu, const T* __restrict__ logvar,
                                      const T* __restrict__ eps, T* __restrict__ sigma, T* __restrict__ z, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float lv = fminf(fmaxf(to_f(logvar[i]), -30.f), 20.f);
    float s = expf(0.5f * lv);
    sigma[i] = from_f<T>(s);
    if (z) z[i] = from_f<T>(to_f(mu[i]) + to_f(eps[i]) * s);
  }
}
// dmu = dz ; dsigma_total = dz*eps + dsigma_ext ; dlogvar = dsigma_total * sigma/2 inside the clamp, else 0
template <typename T>
__global__ void vae_sample_bwd_kernel(const T* __restrict__ logvar, const T* __restrict__ eps,
                                      const T* __restrict__ sigma, const T* __restrict__ dz,
                                      const T* __restrict__ dsig_ext, T* __restrict__ dmu, T* __restrict__ dlogvar,
                                      int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float g = dz ? to_f(dz[i]) : 0.f;
    float ds = (dz ? g * to_f(eps[i]) : 0.f) + (dsig_ext ? to_f(dsig_ext[i]) : 0.f);
    float lv = to_f(logvar[i]);
    bool inside = lv >= -30.f && lv <= 20.f;
    if (dmu) dmu[i] = from_f<T>(g);
    dlogvar[i] = from_f<T>(inside ? ds * 0.5f * to_f(sigma[i]) : 0.f);
  }
}
}  // namespace mig

extern "C" int mig_vae_sample_fwd(int dtype, const void* mu, const void* logvar, const void* eps, void* sigma, void* z,
                                  int64_t n, void* stream) {
  if (n <= 0) return 0;
  MIG_DISPATCH_DTYPE(dtype, T, (vae_sample_fwd_kernel<T><<<bw_grid(n, 256), 256, 0, as_stream(stream)>>>(
                                   (const T*)mu, (const T*)logvar, (const T*)eps, (T*)sigma, (T*)z, n)));
  return check_launch("vae_sample_fwd");
}
extern "C" int mig_vae_sample_bwd(int dtype, const void* logvar, const void* eps, const void* sigma, const void* dz,
                                  const void* dsigma_ext, void* dmu, void* dlogvar, int64_t n, void* stream) {
  if (n <= 0) return 0;
  MIG_DISPATCH_DTYPE(dtype, T, (vae_sample_bwd_kernel<T><<<bw_grid(n, 256), 256, 0, as_stream(stream)>>>(
                                   (const T*)logvar, (const T*)eps, (const T*)sigma, (const T*)dz,
                                   (const T*)dsigma_ext, (T*)dmu, (T*)dlogvar, n)));
  return check_launch("vae_sample_bwd");
}

// ------------------------------------------------------------------------------------------------
// optimizer: sum of squares + fused clip/AdamW over flat fp32 buffers
// ------------------------------------------------------------------------------------------------
namespace mig {
// Strided view used by the sharded optimiser: `count` pieces of `piece4` float4s, `stride4` float4s apart (the slice a
// rank owns of every gradient bucket). piece4 == 0: one contiguous range.
struct Pieces { int64_t piece4, stride4; };
__device__ __forceinline__ int64_t piece_index(const Pieces& s, int64_t i) {
  if (s.piece4 == 0) return i;
  const int64_t b = i / s.piece4;
  return b * s.stride4 + (i - b * s.piece4);
}

__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ g, float* __restrict__ out, int64_t n,
                                                    int vec, Pieces ps) {
  __shared__ float red[33];
  float acc = 0.f;
  const int64_t nvec = vec ? n / 4 : 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
    float4 v = reinterpret_cast<const float4*>(g)[piece_index(ps, i)];
    acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  for (int64_t i = nvec * 4 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    acc += g[i] * g[i];
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) out[blockIdx.x] = acc;   // per-CTA partial; summed in a fixed order by loss_final_kernel
}

struct AdamArgs { float lr, b1, b2, eps, wd, bc1, bc2_sqrt, max_norm; };
__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                    float* __restrict__ m, float* __restrict__ v, int64_t n,
                                                    AdamArgs a, const float* __restrict__ sumsq,
                                                    __nv_bfloat16* __restrict__ shadow,
                                                    const int* __restrict__ step_dev, Pieces ps) {
  if (step_dev) {   // step counter lives on the device (CUDA-graph replay): bias corrections computed here
    const double t = (double)step_dev[0];
    a.bc1 = (float)(1.0 - pow((double)a.b1, t));
    a.bc2_sqrt = (float)sqrt(1.0 - pow((double)a.b2, t));
  }
  float clip = 1.f;
  if (a.max_norm > 0.f && sumsq) {
    // torch.nn.utils.clip_grad_norm_: coef = max_norm / (total_norm + 1e-6), clamped to 1. The clamp keeps a NaN
    // (a NaN anywhere in the gradient): every parameter becomes NaN, as in torch, instead of taking an unclipped step
    float c = a.max_norm / (sqrtf(sumsq[0]) + 1e-6f);
    clip = (c < 1.f || isnan(c)) ? c : 1.f;
  }
  auto upd = [&](float& pi, float gi, float& mi, float& vi) {
    gi *= clip;
    pi *= (1.f - a.lr * a.wd);
    mi = a.b1 * mi + (1.f - a.b1) * gi;
    vi = a.b2 * vi + (1.f - a.b2) * gi * gi;
    const float denom = sqrtf(vi) / a.bc2_sqrt + a.eps;
    pi -= (a.lr / a.bc1) * (mi / denom);
  };
  const bool vec = (n % 4 == 0) && (((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) |
                                      reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v)) & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(shadow) & 7) == 0);
  if (vec) {   // 128-bit streaming accesses: 7 fp32 streams + the bf16 shadow, one pass over the flat buffers
    const int64_t n4 = n / 4;
    for (int64_t ii = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; ii < n4; ii += (int64_t)gridDim.x * blockDim.x) {
      const int64_t i = piece_index(ps, ii);
      float4 P = reinterpret_cast<float4*>(p)[i], G = reinterpret_cast<const float4*>(g)[i];
      float4 M = reinterpret_cast<float4*>(m)[i], V = reinterpret_cast<float4*>(v)[i];
      upd(P.x, G.x, M.x, V.x); upd(P.y, G.y, M.y, V.y); upd(P.z, G.z, M.z, V.z); upd(P.w, G.w, M.w, V.w);
      reinterpret_cast<float4*>(p)[i] = P;
      reinterpret_cast<float4*>(m)[i] = M;
      reinterpret_cast<float4*>(v)[i] = V;
      if (shadow) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(P.x, P.y), hi = __floats2bfloat162_rn(P.z, P.w);
        uint2 pk;
        pk.x = *reinterpret_cast<uint32_t*>(&lo);
        pk.y = *reinterpret_cast<uint32_t*>(&hi);
        reinterpret_cast<uint2*>(shadow)[i] = pk;
      }
    }
    return;
  }
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float pi = p[i], mi = m[i], vi = v[i];
    upd(pi, g[i], mi, vi);
    p[i] = pi; m[i] = mi; v[i] = vi;
    if (shadow) shadow[i] = __float2bfloat16_rn(pi);
  }
}
}  // namespace mig

extern "C" int mig_sumsq(const float* g, float* out, float* partials, int64_t n, void* stream) {
  MIG_REQUIRE(n > 0 && partials != nullptr, "sumsq: empty input or missing partials buffer");
  // deterministic: per-CTA partials, then one CTA adds them in a fixed order (in double). Data-parallel replicas
  // must compute bit-identical clip coefficients or they drift apart.
  int grid = bw_grid((n + 3) / 4, 256, 4);
  if (grid > kLossBlocks) grid = kLossBlocks;
  sumsq_kernel<<<grid, 256, 0, as_stream(stream)>>>(g, partials, n, aligned16(g), Pieces{0, 0});
  loss_final_kernel<<<1, 256, 0, as_stream(stream)>>>(partials, grid, out, 1.0);
  return check_launch("sumsq");
}
// the same over `count` pieces of `piece` elements, `stride` elements apart, starting at g (sharded optimiser: the
// slice this rank owns of every gradient bucket). piece, stride: multiples of 4; g 16-byte aligned.
extern "C" int mig_sumsq_strided(const float* g, float* out, float* partials, int64_t piece, int64_t stride,
                                 int64_t count, void* stream) {
  MIG_REQUIRE(piece > 0 && count > 0 && partials != nullptr, "sumsq_strided: empty input or missing partials buffer");
  MIG_REQUIRE(piece % 4 == 0 && stride % 4 == 0 && aligned16(g), "sumsq_strided: pieces must be 16-byte aligned");
  const int64_t n = piece * count;
  int grid = bw_grid((n + 3) / 4, 256, 4);
  if (grid > kLossBlocks) grid = kLossBlocks;
  sumsq_kernel<<<grid, 256, 0, as_stream(stream)>>>(g, partials, n, 1, Pieces{piece / 4, stride / 4});
  loss_final_kernel<<<1, 256, 0, as_stream(stream)>>>(partials, grid, out, 1.0);
  return check_launch("sumsq_strided");
}
extern "C" int mig_adamw_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1,
                              float beta2, float eps, float weight_decay, int32_t step, const float* sumsq,
                              float max_norm, void* bf16_shadow, const int32_t* step_device, void* stream) {
  if (n <= 0) return 0;
  MIG_REQUIRE(step >= 1 || step_device != nullptr, "adamw: step counts from 1");
  const int s = step >= 1 ? step : 1;
  AdamArgs a{lr, beta1, beta2, eps, weight_decay, (float)(1.0 - pow((double)beta1, (double)s)),
             (float)sqrt(1.0 - pow((double)beta2, (double)s)), max_norm};
  adamw_kernel<<<bw_grid(n, 256), 256, 0, as_stream(stream)>>>(p, g, m, v, n, a, sumsq, (__nv_bfloat16*)bf16_shadow,
                                                               step_device, Pieces{0, 0});
  return check_launch("adamw");
}
// mig_adamw_step over `count` pieces of `piece` elements, `stride` elements apart (all buffers share the layout and are
// passed at the first owned element): the update of the slices ONE data-parallel rank owns (ZeRO-1 style sharding).
extern "C" int mig_adamw_step_strided(float* p, const float* g, float* m, float* v, int64_t piece, int64_t stride,
                                      int64_t count, float lr, float beta1, float beta2, float eps, float weight_decay,
                                      int32_t step, const float* sumsq, float max_norm, void* bf16_shadow,
                                      const int32_t* step_device, void* stream) {
  if (piece <= 0 || count <= 0) return 0;
  MIG_REQUIRE(step >= 1 || step_device != nullptr, "adamw: step counts from 1");
  MIG_REQUIRE(piece % 4 == 0 && stride % 4 == 0 && aligned16(p) && aligned16(g) && aligned16(m) && aligned16(v) &&
                  (reinterpret_cast<uintptr_t>(bf16_shadow) & 7) == 0,
              "adamw_strided: pieces must be 16-byte aligned");
  const int s = step >= 1 ? step : 1;
  AdamArgs a{lr, beta1, beta2, eps, weight_decay, (float)(1.0 - pow((double)beta1, (double)s)),
             (float)sqrt(1.0 - pow((double)beta2, (double)s)), max_norm};
  const int64_t n = piece * count;
  adamw_kernel<<<bw_grid(n, 256), 256, 0, as_stream(stream)>>>(p, g, m, v, n, a, sumsq, (__nv_bfloat16*)bf16_shadow,
                                                               step_device, Pieces{piece / 4, stride / 4});
  return check_launch("adamw_strided");
}

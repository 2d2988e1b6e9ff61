// GroupNorm(+SiLU) forward / backward for bf16 channels-last activations as TMA-staged streaming kernels.
//
// Replaces nn.GroupNorm + nn.SiLU at unet:628-629,648,677,698,1932-1933 and ae:157,167,194,198,451,604 (bf16 production
// path; groupnorm.cu keeps the register-streaming kernels for fp32 parity mode and odd channel counts).
//
// Why a second implementation: ncu on the register-streaming kernels (profiles/r02_ncu_full_groupnorm_before.csv) showed
// neither DRAM (30-38 %) nor the SMs (31-42 %) busy: 80 registers per thread allowed 3 CTAs per SM, the 592-CTA grid
// ran as 1.33 waves, and every thread alternated between "8 loads in flight" and a long SiLU' dependency chain, so the
// memory system idled while the ALUs worked and vice versa. Here
//   * a CTA owns ONE (sample, 256-channel slab, row chunk) and streams it through a 3-4 stage shared-memory ring filled
//     by TMA (cp.async.bulk.tensor, one elected thread): 48-64 KB per CTA are in flight regardless of registers;
//   * the grid is exactly one wave (2 CTAs per SM x SM count), sized on the host;
//   * every thread keeps a fixed 16-byte channel vector, so per-channel coefficients / partial sums live in registers;
//   * backward statistics are written as per-CTA partials (no atomics, deterministic) and summed by one small kernel
//     that also forms the group sums and the per-(sample, channel) column sums of dx -- the bias / time-embedding gradient of the convolution that produced x (saves that conv's colsum
//     passes over dy).
// Forward statistics arrive either from the producing convolution's epilogue (conv_tma.cu, mig_conv_fwd_stats) or from
// gt_stats_kernel; the apply kernel turns the raw fp64 sums into mean / rstd itself (no finalize launch).
#include <cuda.h>

#include "common.cuh"
#include "tc_common.cuh"
#include "tc_host.cuh"

namespace mig {

using namespace tc;

constexpr int GT_THREADS = 256;
constexpr int GT_TENSOR_STAGE = 16384;   // bytes of one tensor in one stage
constexpr int GT_MAX_STAGES = 4;

struct GtGeom {
  int N, C, G, cpg;
  int64_t S;
  int slabs, cb, cvb, rpp, R;   // channel slabs, channels / 16-byte vectors per slab row, rows per pass, rows per stage
  int chunks;                   // row chunks per (sample, slab)
  int64_t rows_per_chunk;       // multiple of R
};

// largest power of two <= 256 dividing C (C % 8 == 0 is required by the callers)
static int slab_channels(int C) {
  int cb = 256;
  while (cb > 8 && C % cb != 0) cb >>= 1;
  return cb;
}

bool gt_eligible(int N, int64_t S, int C, int G) {
  if (C % 8 != 0 || G <= 0 || C % G != 0) return false;
  if (slab_channels(C) < 32) return false;
  if ((int64_t)N * S >= (int64_t)1 << 31) return false;
  return N > 0 && N < 65536 && S > 0;
}

static GtGeom gt_geom(int N, int64_t S, int C, int G) {
  GtGeom g;
  g.N = N; g.C = C; g.G = G; g.cpg = C / G; g.S = S;
  g.cb = slab_channels(C);
  g.slabs = C / g.cb;
  g.cvb = g.cb / 8;
  g.rpp = GT_THREADS / g.cvb;
  g.R = GT_TENSOR_STAGE / (g.cb * 2);
  const int64_t target = 2 * (int64_t)device_info().sm_count;   // one wave at two CTAs per SM
  int64_t chunks = target / ((int64_t)N * g.slabs);
  if (chunks < 1) chunks = 1;
  int64_t rows = (S + chunks - 1) / chunks;
  rows = (rows + g.R - 1) / g.R * g.R;
  g.rows_per_chunk = rows;
  g.chunks = (int)((S + rows - 1) / rows);
  return g;
}

static int gt_map(CUtensorMap* m, const void* base, const GtGeom& g) {
  const uint64_t dims[2] = {(uint64_t)g.C, (uint64_t)((int64_t)g.N * g.S)};
  const uint64_t strides[1] = {(uint64_t)g.C * 2};
  const uint32_t box[2] = {(uint32_t)g.cb, (uint32_t)g.R};
  return make_map(m, base, 2, dims, strides, box, "groupnorm map", CU_TENSOR_MAP_SWIZZLE_NONE);
}

__device__ __forceinline__ uint4 lds16(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void unpack8(const uint4& raw, float f[8]) {
  const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {   // bf16 -> fp32 is a 16-bit shift
    f[2 * i] = __uint_as_float(w[i] << 16);
    f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}
__device__ __forceinline__ uint4 pack8(const float f[8]) {
  uint4 o;
  __nv_bfloat162 a = __floats2bfloat162_rn(f[0], f[1]), b = __floats2bfloat162_rn(f[2], f[3]),
                 c = __floats2bfloat162_rn(f[4], f[5]), d = __floats2bfloat162_rn(f[6], f[7]);
  o.x = *reinterpret_cast<uint32_t*>(&a); o.y = *reinterpret_cast<uint32_t*>(&b);
  o.z = *reinterpret_cast<uint32_t*>(&c); o.w = *reinterpret_cast<uint32_t*>(&d);
  return o;
}

// The streaming skeleton: NT input tensors, STAGES ring slots; body(row_in_sample, smem address of this thread's vector
// of tensor 0, of tensor 1) is called for every valid row of the thread.
template <int NT, int STAGES, typename Body>
__device__ __forceinline__ void gt_stream(const CUtensorMap* m0, const CUtensorMap* m1, const GtGeom& g, uint32_t smem,
                                          uint32_t bars, int n, int slab, int chunk, Body&& body) {
  constexpr uint32_t STAGE_BYTES = NT * GT_TENSOR_STAGE;
  const int tcol = threadIdx.x % g.cvb, trow = threadIdx.x / g.cvb;
  const int64_t r0 = (int64_t)chunk * g.rows_per_chunk;
  const int64_t r1 = r0 + g.rows_per_chunk < g.S ? r0 + g.rows_per_chunk : g.S;
  const int nst = (int)((r1 - r0 + g.R - 1) / g.R);
  const int col0 = slab * g.cb;
  const int64_t grow0 = (int64_t)n * g.S + r0;
  auto issue = [&](int it) {
    const int s = it % STAGES;
    const uint32_t dst = smem + s * STAGE_BYTES, bar = bars + 8 * s;
    mbar_arrive_expect_tx(bar, STAGE_BYTES);
    tma_load_2d(dst, m0, bar, col0, (int)(grow0 + (int64_t)it * g.R));
    if (NT == 2) tma_load_2d(dst + GT_TENSOR_STAGE, m1, bar, col0, (int)(grow0 + (int64_t)it * g.R));
  };
  if (threadIdx.x == 0)
    for (int it = 0; it < STAGES && it < nst; ++it) issue(it);
  const uint32_t toff = (uint32_t)(trow * g.cb * 2 + tcol * 16);
  const uint32_t pass_bytes = (uint32_t)(g.rpp * g.cb * 2);
  for (int it = 0; it < nst; ++it) {
    const int s = it % STAGES;
    mbar_wait(bars + 8 * s, (uint32_t)(it / STAGES) & 1u);
    const uint32_t base = smem + s * STAGE_BYTES + toff;
    const int64_t rb = r0 + (int64_t)it * g.R + trow;
#pragma unroll
    for (int k = 0; k < 4; ++k) {   // R / rpp == 4 for every slab width
      const int64_t r = rb + (int64_t)k * g.rpp;
      if (r < r1) body(r, base + k * pass_bytes, base + k * pass_bytes + GT_TENSOR_STAGE);
    }
    __syncthreads();   // every thread is done with slot s: it may be refilled
    if (threadIdx.x == 0 && it + STAGES < nst) issue(it + STAGES);
  }
}

__device__ __forceinline__ void gt_init_bars(uint64_t* bars, int stages) {
  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) mbar_init(smem_u32(&bars[s]), 1);
    fence_barrier_init();
  }
  __syncthreads();
}

// ---- forward statistics: fp64 atomics into sums[n][g][2] (a handful per CTA) ------------------------------------------
__global__ void __launch_bounds__(GT_THREADS, 2) gt_stats_kernel(const __grid_constant__ CUtensorMap xm,
                                                                 double* __restrict__ sums, GtGeom g) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem = (smem_u32(smem_raw) + 127u) & ~127u;
  __shared__ __align__(8) uint64_t bars[GT_MAX_STAGES];
  __shared__ float gacc[2 * 256];   // [group in slab][2] (cpg >= 1 -> at most 256 groups per slab)
  gt_init_bars(bars, GT_MAX_STAGES);
  const int n = blockIdx.z, slab = blockIdx.y, chunk = blockIdx.x;
  float s[8], ss[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = ss[j] = 0.f;
  gt_stream<1, 4>(&xm, &xm, g, smem, smem_u32(&bars[0]), n, slab, chunk, [&](int64_t, uint32_t a0, uint32_t) {
    float f[8];
    unpack8(lds16(a0), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) { s[j] += f[j]; ss[j] = fmaf(f[j], f[j], ss[j]); }
  });
  for (int i = threadIdx.x; i < 2 * 256; i += GT_THREADS) gacc[i] = 0.f;
  __syncthreads();
  const int tcol = threadIdx.x % g.cvb;
  const int c0 = slab * g.cb + tcol * 8, g0 = (slab * g.cb) / g.cpg;
  int j = 0;
  while (j < 8) {   // merge the channels of this vector that share a group before touching shared memory
    const int grp = (c0 + j) / g.cpg;
    float a = 0.f, b = 0.f;
    while (j < 8 && (c0 + j) / g.cpg == grp) { a += s[j]; b += ss[j]; ++j; }
    atomicAdd(&gacc[2 * (grp - g0)], a);
    atomicAdd(&gacc[2 * (grp - g0) + 1], b);
  }
  __syncthreads();
  const int ng = (g.cb + g.cpg - 1) / g.cpg + 1;
  for (int i = threadIdx.x; i < 2 * ng && i < 2 * 256; i += GT_THREADS) {
    const int grp = g0 + (i >> 1);
    const float v = gacc[i];
    if (grp < g.G && v != 0.f) atomicAdd(&sums[((int64_t)n * g.G + grp) * 2 + (i & 1)], (double)v);
  }
}

// mean / rstd of group `grp` of sample n from the raw sums
__device__ __forceinline__ void gt_group_stats(const double* __restrict__ sums, int n, int G, int grp, double inv_count,
                                               double eps, float& mean, float& rstd) {
  const double m = sums[((int64_t)n * G + grp) * 2] * inv_count;
  double var = sums[((int64_t)n * G + grp) * 2 + 1] * inv_count - m * m;
  if (var < 0.0) var = 0.0;
  mean = (float)m;
  rstd = (float)(1.0 / sqrt(var + eps));
}

// ---- forward apply: y = silu?((x - mean) * rstd * gamma + beta) -------------------------------------------------------
template <bool SILU>
__global__ void __launch_bounds__(GT_THREADS, 2) gt_apply_kernel(const __grid_constant__ CUtensorMap xm,
                                                                 const float* __restrict__ gamma,
                                                                 const float* __restrict__ beta,
                                                                 const double* __restrict__ sums,
                                                                 __nv_bfloat16* __restrict__ y, float* __restrict__ mean,
                                                                 float* __restrict__ rstd, GtGeom g, double inv_count,
                                                                 double eps) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem = (smem_u32(smem_raw) + 127u) & ~127u;
  __shared__ __align__(8) uint64_t bars[GT_MAX_STAGES];
  gt_init_bars(bars, GT_MAX_STAGES);
  const int n = blockIdx.z, slab = blockIdx.y, chunk = blockIdx.x;
  if (chunk == 0 && slab == 0 && mean)   // publish mean / rstd for the backward pass
    for (int grp = threadIdx.x; grp < g.G; grp += GT_THREADS) {
      float m, r;
      gt_group_stats(sums, n, g.G, grp, inv_count, eps, m, r);
      mean[n * g.G + grp] = m;
      rstd[n * g.G + grp] = r;
    }
  const int tcol = threadIdx.x % g.cvb;
  const int c0 = slab * g.cb + tcol * 8;
  float a[8], b[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float m, r;
    gt_group_stats(sums, n, g.G, (c0 + j) / g.cpg, inv_count, eps, m, r);
    a[j] = r * gamma[c0 + j];
    b[j] = fmaf(-m, a[j], beta[c0 + j]);
  }
  __nv_bfloat16* ybase = y + ((int64_t)n * g.S) * g.C + c0;
  gt_stream<1, 4>(&xm, &xm, g, smem, smem_u32(&bars[0]), n, slab, chunk, [&](int64_t r, uint32_t a0, uint32_t) {
    float f[8];
    unpack8(lds16(a0), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float z = fmaf(f[j], a[j], b[j]);
      f[j] = SILU ? z * sigmoid_tanh_f(z) : z;
    }
    *reinterpret_cast<uint4*>(ybase + r * g.C) = pack8(f);
  });
}

// ---- backward statistics: per-CTA partials of (sum dz*xhat, sum dz, sum x) per channel --------------------------------
template <bool SILU>
__global__ void __launch_bounds__(GT_THREADS, 2) gt_bwd_stats_kernel(const __grid_constant__ CUtensorMap xm,
                                                                     const __grid_constant__ CUtensorMap dym,
                                                                     const float* __restrict__ gamma,
                                                                     const float* __restrict__ beta,
                                                                     const float* __restrict__ mean,
                                                                     const float* __restrict__ rstd,
                                                                     float* __restrict__ part, GtGeom g) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem = (smem_u32(smem_raw) + 127u) & ~127u;
  __shared__ __align__(8) uint64_t bars[GT_MAX_STAGES];
  gt_init_bars(bars, 3);
  const int n = blockIdx.z, slab = blockIdx.y, chunk = blockIdx.x;
  const int tcol = threadIdx.x % g.cvb;
  const int c0 = slab * g.cb + tcol * 8;
  float rs[8], m2[8], ga[8], be[8], p1[8], p2[8], p3[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int gi = n * g.G + (c0 + j) / g.cpg;
    rs[j] = rstd[gi];
    m2[j] = -mean[gi] * rs[j];
    ga[j] = gamma[c0 + j];
    be[j] = beta[c0 + j];
    p1[j] = p2[j] = p3[j] = 0.f;
  }
  gt_stream<2, 3>(&xm, &dym, g, smem, smem_u32(&bars[0]), n, slab, chunk, [&](int64_t, uint32_t a0, uint32_t a1) {
    float x[8], d[8];
    unpack8(lds16(a0), x);
    unpack8(lds16(a1), d);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float xh = fmaf(x[j], rs[j], m2[j]);
      float dz = d[j];
      if (SILU) {
        const float z = fmaf(xh, ga[j], be[j]);
        const float sg = sigmoid_tanh_f(z);
        dz *= sg * fmaf(z, 1.f - sg, 1.f);
      }
      p1[j] = fmaf(dz, xh, p1[j]);
      p2[j] += dz;
      p3[j] += x[j];
    }
  });
  // reduce the row lanes of the CTA through the (now idle) stage memory: [24 values][256 threads], conflict-free
  float* red = reinterpret_cast<float*>(smem_raw + (smem - smem_u32(smem_raw)));
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    red[(3 * j) * GT_THREADS + threadIdx.x] = p1[j];
    red[(3 * j + 1) * GT_THREADS + threadIdx.x] = p2[j];
    red[(3 * j + 2) * GT_THREADS + threadIdx.x] = p3[j];
  }
  __syncthreads();
  float* dst = part + (((int64_t)n * g.chunks + chunk) * g.C + slab * g.cb) * 3;
  for (int e = threadIdx.x; e < g.cvb * 24; e += GT_THREADS) {
    const int q = e / g.cvb, tc = e - q * g.cvb;
    float sum = 0.f;
    for (int rr = 0; rr < g.rpp; ++rr) sum += red[q * GT_THREADS + rr * g.cvb + tc];
    dst[(tc * 8 + q / 3) * 3 + (q % 3)] = sum;
  }
}

// Totals and group sums in ONE small launch. Block (q, n) owns a quarter of the groups of sample n: its threads add the
// per-CTA partials of the block's channels (coalesced: consecutive threads, consecutive (channel, moment) items), keep
// the totals in shared memory, then one thread per group forms A = sum_c gamma_c * (sum dz xhat), B = sum_c gamma_c *
// (sum dz) and the column sums of dx. tot[n][c][3] goes to global memory for dgamma / dbeta (summed over n by the
// apply kernel's first CTAs).
__global__ void __launch_bounds__(256) gt_bwd_reduce_kernel(const float* __restrict__ part, const float* __restrict__ gamma,
                                                            const float* __restrict__ mean,
                                                            const float* __restrict__ rstd, float* __restrict__ tot,
                                                            float* __restrict__ grp, float* __restrict__ dxsum, int N,
                                                            int C, int G, int chunks, float S) {
  extern __shared__ float tl[];   // [(c1 - c0) * 3]
  const int n = blockIdx.y, cpg = C / G;
  const int gq = (G + gridDim.x - 1) / gridDim.x;
  const int g0 = blockIdx.x * gq, g1 = min(G, g0 + gq);
  if (g0 >= g1) return;
  const int c0 = g0 * cpg, nitem = (g1 - g0) * cpg * 3;
  const float* p = part + ((int64_t)n * chunks) * C * 3 + (int64_t)c0 * 3;
  for (int i = threadIdx.x; i < nitem; i += blockDim.x) {
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    int k = 0;
    for (; k + 3 < chunks; k += 4) {
      s0 += p[(int64_t)k * C * 3 + i];
      s1 += p[(int64_t)(k + 1) * C * 3 + i];
      s2 += p[(int64_t)(k + 2) * C * 3 + i];
      s3 += p[(int64_t)(k + 3) * C * 3 + i];
    }
    for (; k < chunks; ++k) s0 += p[(int64_t)k * C * 3 + i];
    const float s = (s0 + s1) + (s2 + s3);
    tl[i] = s;
    tot[((int64_t)n * C + c0) * 3 + i] = s;
  }
  __syncthreads();
  for (int gi = g0 + threadIdx.x; gi < g1; gi += blockDim.x) {
    float a = 0.f, b = 0.f;
    for (int c = gi * cpg; c < (gi + 1) * cpg; ++c) {
      a = fmaf(gamma[c], tl[(c - c0) * 3], a);
      b = fmaf(gamma[c], tl[(c - c0) * 3 + 1], b);
    }
    grp[2 * (n * G + gi)] = a;
    grp[2 * (n * G + gi) + 1] = b;
    if (dxsum) {
      // sum_s dx[n,s,c] = rstd * (gamma_c * sum dz - (A * sum xhat + B * S) / cnt),  sum xhat = rstd * (sum x - S mean)
      const float r = rstd[n * G + gi], m = mean[n * G + gi], inv = 1.f / (S * (float)cpg);
      for (int c = gi * cpg; c < (gi + 1) * cpg; ++c) {
        const float sxh = r * (tl[(c - c0) * 3 + 2] - S * m);
        dxsum[(int64_t)n * C + c] = r * (gamma[c] * tl[(c - c0) * 3 + 1] - (a * sxh + b * S) * inv);
      }
    }
  }
}

// ---- backward apply: dx = rstd * (dz*gamma - (xhat*A + B) / cnt) ------------------------------------------------------
template <bool SILU>
__global__ void __launch_bounds__(GT_THREADS, 2) gt_bwd_apply_kernel(const __grid_constant__ CUtensorMap xm,
                                                                     const __grid_constant__ CUtensorMap dym,
                                                                     const float* __restrict__ gamma,
                                                                     const float* __restrict__ beta,
                                                                     const float* __restrict__ mean,
                                                                     const float* __restrict__ rstd,
                                                                     const float* __restrict__ grp,
                                                                     const float* __restrict__ tot,
                                                                     __nv_bfloat16* __restrict__ dx,
                                                                     const __nv_bfloat16* __restrict__ addend,
                                                                     float* __restrict__ dgamma,
                                                                     float* __restrict__ dbeta, int accumulate, GtGeom g,
                                                                     float inv_count) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem = (smem_u32(smem_raw) + 127u) & ~127u;
  __shared__ __align__(8) uint64_t bars[GT_MAX_STAGES];
  gt_init_bars(bars, 3);
  const int n = blockIdx.z, slab = blockIdx.y, chunk = blockIdx.x;
  const int tcol = threadIdx.x % g.cvb;
  const int c0 = slab * g.cb + tcol * 8;
  // dx = k1*dz - k2*xhat - k3 with xhat = x*rs + m2, z = xhat*ga + be
  float rs[8], m2[8], ga[8], be[8], k1[8], k2[8], k3[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int gi = n * g.G + (c0 + j) / g.cpg;
    rs[j] = rstd[gi];
    m2[j] = -mean[gi] * rs[j];
    ga[j] = gamma[c0 + j];
    be[j] = beta[c0 + j];
    k1[j] = rs[j] * ga[j];
    k2[j] = rs[j] * grp[2 * gi] * inv_count;
    k3[j] = rs[j] * grp[2 * gi + 1] * inv_count;
  }
  if (n == 0 && chunk == 0 && threadIdx.x < g.cvb) {   // dgamma / dbeta = totals summed over the samples
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float a = 0.f, b = 0.f;
      for (int nn = 0; nn < g.N; ++nn) {
        a += tot[((int64_t)nn * g.C + c0 + j) * 3];
        b += tot[((int64_t)nn * g.C + c0 + j) * 3 + 1];
      }
      if (dgamma) dgamma[c0 + j] = accumulate ? dgamma[c0 + j] + a : a;
      if (dbeta) dbeta[c0 + j] = accumulate ? dbeta[c0 + j] + b : b;
    }
  }
  __nv_bfloat16* obase = dx + ((int64_t)n * g.S) * g.C + c0;
  const __nv_bfloat16* abase = addend ? addend + ((int64_t)n * g.S) * g.C + c0 : nullptr;
  gt_stream<2, 3>(&xm, &dym, g, smem, smem_u32(&bars[0]), n, slab, chunk, [&](int64_t r, uint32_t a0, uint32_t a1) {
    float x[8], d[8];
    unpack8(lds16(a0), x);
    unpack8(lds16(a1), d);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float xh = fmaf(x[j], rs[j], m2[j]);
      float dz = d[j];
      if (SILU) {
        const float z = fmaf(xh, ga[j], be[j]);
        const float sg = sigmoid_tanh_f(z);
        dz *= sg * fmaf(z, 1.f - sg, 1.f);
      }
      x[j] = fmaf(k1[j], dz, -fmaf(k2[j], xh, k3[j]));
    }
    if (abase) {   // the gradient arriving through the block's skip path (x also feeds the residual add): one fused read
      float ad[8];
      unpack8(*reinterpret_cast<const uint4*>(abase + r * g.C), ad);
#pragma unroll
      for (int j = 0; j < 8; ++j) x[j] += ad[j];
    }
    *reinterpret_cast<uint4*>(obase + r * g.C) = pack8(x);
  });
}

// ---- host side ----------------------------------------------------------------------------------------------------------
template <typename K>
static int gt_optin(K kernel, int smem, SmemOptIn& st, const char* what) {
  return ensure_dynamic_smem(kernel, smem, st, what);
}

int64_t gt_bwd_workspace_bytes(int N, int64_t S, int C, int G) {
  if (!gt_eligible(N, S, C, G)) return 0;
  GtGeom g = gt_geom(N, S, C, G);
  return ((int64_t)N * g.chunks * C * 3 + (int64_t)N * C * 3 + (int64_t)N * G * 2) * 4 + 256;
}

int gt_stats(const void* x, double* sums, int N, int64_t S, int C, int G, void* stream) {
  cudaStream_t st = as_stream(stream);
  GtGeom g = gt_geom(N, S, C, G);
  CUtensorMap xm;
  if (gt_map(&xm, x, g)) return 1;
  constexpr int smem = 4 * GT_TENSOR_STAGE + 128;
  static SmemOptIn o;
  if (int rc = gt_optin(gt_stats_kernel, smem, o, "groupnorm_stats")) return rc;
  cudaMemsetAsync(sums, 0, sizeof(double) * (size_t)N * G * 2, st);
  gt_stats_kernel<<<dim3(g.chunks, g.slabs, N), GT_THREADS, smem, st>>>(xm, sums, g);
  return check_launch("groupnorm_stats");
}

int gt_apply(const void* x, const float* gamma, const float* beta, const double* sums, void* y, float* mean, float* rstd,
             int N, int64_t S, int C, int G, float eps, int silu, void* stream) {
  cudaStream_t st = as_stream(stream);
  GtGeom g = gt_geom(N, S, C, G);
  CUtensorMap xm;
  if (gt_map(&xm, x, g)) return 1;
  constexpr int smem = 4 * GT_TENSOR_STAGE + 128;
  const double inv = 1.0 / ((double)S * g.cpg);
  dim3 grid(g.chunks, g.slabs, N);
  if (silu) {
    static SmemOptIn o;
    if (int rc = gt_optin(gt_apply_kernel<true>, smem, o, "groupnorm_apply")) return rc;
    gt_apply_kernel<true><<<grid, GT_THREADS, smem, st>>>(xm, gamma, beta, sums, (__nv_bfloat16*)y, mean, rstd, g, inv,
                                                          (double)eps);
  } else {
    static SmemOptIn o;
    if (int rc = gt_optin(gt_apply_kernel<false>, smem, o, "groupnorm_apply")) return rc;
    gt_apply_kernel<false><<<grid, GT_THREADS, smem, st>>>(xm, gamma, beta, sums, (__nv_bfloat16*)y, mean, rstd, g, inv,
                                                           (double)eps);
  }
  return check_launch("groupnorm_apply");
}

int gt_bwd(const void* x, const void* dy, const float* gamma, const float* beta, const float* mean, const float* rstd,
           void* dx, float* dgamma, float* dbeta, float* dx_colsum, const void* dx_addend, int accumulate_dparams, int N,
           int64_t S, int C, int G, int silu, void* ws, int64_t ws_bytes, void* stream) {
  MIG_REQUIRE(ws_bytes >= gt_bwd_workspace_bytes(N, S, C, G), "groupnorm_bwd: workspace too small");
  cudaStream_t st = as_stream(stream);
  GtGeom g = gt_geom(N, S, C, G);
  CUtensorMap xm, dym;
  if (gt_map(&xm, x, g) || gt_map(&dym, dy, g)) return 1;
  float* part = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  float* tot = part + (int64_t)N * g.chunks * C * 3;
  float* grp = tot + (int64_t)N * C * 3;
  constexpr int smem = 3 * 2 * GT_TENSOR_STAGE + 128;
  dim3 grid(g.chunks, g.slabs, N);
  if (silu) {
    static SmemOptIn o;
    if (int rc = gt_optin(gt_bwd_stats_kernel<true>, smem, o, "groupnorm_bwd")) return rc;
    gt_bwd_stats_kernel<true><<<grid, GT_THREADS, smem, st>>>(xm, dym, gamma, beta, mean, rstd, part, g);
  } else {
    static SmemOptIn o;
    if (int rc = gt_optin(gt_bwd_stats_kernel<false>, smem, o, "groupnorm_bwd")) return rc;
    gt_bwd_stats_kernel<false><<<grid, GT_THREADS, smem, st>>>(xm, dym, gamma, beta, mean, rstd, part, g);
  }
  {
    const int pb = G >= 4 ? 4 : 1, gq = (G + pb - 1) / pb;
    gt_bwd_reduce_kernel<<<dim3(pb, N), 256, (size_t)gq * g.cpg * 3 * sizeof(float), st>>>(
        part, gamma, mean, rstd, tot, grp, dx_colsum, N, C, G, g.chunks, (float)S);
  }
  const float inv = 1.f / ((float)S * (float)g.cpg);
  if (silu) {
    static SmemOptIn o;
    if (int rc = gt_optin(gt_bwd_apply_kernel<true>, smem, o, "groupnorm_bwd")) return rc;
    gt_bwd_apply_kernel<true><<<grid, GT_THREADS, smem, st>>>(xm, dym, gamma, beta, mean, rstd, grp, tot,
                                                              (__nv_bfloat16*)dx, (const __nv_bfloat16*)dx_addend, dgamma,
                                                              dbeta, accumulate_dparams, g, inv);
  } else {
    static SmemOptIn o;
    if (int rc = gt_optin(gt_bwd_apply_kernel<false>, smem, o, "groupnorm_bwd")) return rc;
    gt_bwd_apply_kernel<false><<<grid, GT_THREADS, smem, st>>>(xm, dym, gamma, beta, mean, rstd, grp, tot,
                                                               (__nv_bfloat16*)dx, (const __nv_bfloat16*)dx_addend, dgamma,
                                                               dbeta, accumulate_dparams, g, inv);
  }
  return check_launch("groupnorm_bwd");
}

}  // namespace mig

// SSIM / multi-scale SSIM statistics with a separable window (replaces monai-generative's compute_ssim_and_cs,
// train_ldm.py:241-330): five depthwise "valid" correlations (mu_x, mu_y, E[x^2], E[y^2], E[xy]) and the SSIM / cs maps,
// reduced to per-pair means, without any filtered map leaving the chip.
//
// One CTA owns a 32 (W) x 8 (H) tile of output voxels of one (pair, channel) and streams a chunk of output planes along
// D. Per input plane it stages the x / y tile with its halo in shared memory, filters the five products along W (into
// shared memory) and then along H (one output voxel per thread), and keeps the last kd H-filtered planes in a register
// ring. The ring is R >= kd deep and the plane loop is unrolled by R, so every ring slot index is a compile-time
// constant and the ring never touches local memory (R = 1, 4, 8, 12, 16; 12 serves the default 11-tap window with
// half the registers of 16). Once kd planes are in the ring, the D filter finishes the five means
// and the thread accumulates ssim and cs. D is cut into chunks (recomputing the kd - 1 overlap planes) only when the
// tiles of all pairs cannot fill the machine.
//
// Reduction: fp32 per thread, a fixed warp-shuffle tree, the 8 warp sums added in order in fp64 -> one (ssim, cs) pair
// of doubles per CTA; a second kernel adds each pair's CTA partials in a fixed order in fp64. No atomics: the same
// call on the same inputs gives bit-identical results, and swapping a and b gives bit-identical results too (every
// expression is symmetric in x and y with commutative IEEE operations; the one sum of two products that FMA contraction
// would make asymmetric, mu_x^2 + mu_y^2, is written with explicit round-to-nearest operations).
#include "common.cuh"

namespace mig {

constexpr int kSsimTW = 32, kSsimTH = 8, kSsimThreads = kSsimTW * kSsimTH, kSsimKMax = 16;
constexpr int kSsimTargetCtas = 4 * 148;  // fixed (not the device's SM count) so the split, and the bits, are portable

struct SsimArgs {
  float taps[3][kSsimKMax];  // d, h, w
  int k[3];                  // kd, kh, kw
  int dims[3];               // D, H, W of the inputs
  int out[3];                // valid extents: dims - k + 1
  int C, na, nb;
  int tiles_w, tiles, chunks, chunk_len;
  float c1, c2;
};

template <typename T, int R>
__global__ void __launch_bounds__(kSsimThreads) ssim_partial_kernel(const T* __restrict__ a, const T* __restrict__ b,
                                                                    const int32_t* __restrict__ pairs, SsimArgs s,
                                                                    double2* __restrict__ partial) {
  constexpr int TW = kSsimTW, TH = kSsimTH, KM = kSsimKMax;
  __shared__ float taps[3][KM];
  __shared__ float sx[(TH + KM - 1) * (TW + KM - 1)], sy[(TH + KM - 1) * (TW + KM - 1)];
  __shared__ float hw[5][(TH + KM - 1) * TW];
  __shared__ double wsum[2][kSsimThreads / 32];

  const int tid = threadIdx.x;
  int64_t bid = blockIdx.x;
  const int tile = (int)(bid % s.tiles);
  bid /= s.tiles;
  const int chunk = (int)(bid % s.chunks);
  bid /= s.chunks;
  const int c = (int)(bid % s.C);
  const int p = (int)(bid / s.C);
  const int i = pairs[2 * p], j = pairs[2 * p + 1];
  if (i < 0 || i >= s.na || j < 0 || j >= s.nb) {  // an index outside a / b: NaN for this pair, no stray read
    if (tid == 0) partial[blockIdx.x] = make_double2(__longlong_as_double(0x7ff8000000000000LL),
                                                     __longlong_as_double(0x7ff8000000000000LL));
    return;
  }
  if (tid < 3 * KM) taps[tid / KM][tid % KM] = s.taps[tid / KM][tid % KM];

  const int D = s.dims[0], H = s.dims[1], W = s.dims[2], C = s.C;
  const int kd = s.k[0], kh = s.k[1], kw = s.k[2];
  const int w0 = (tile % s.tiles_w) * TW, h0 = (tile / s.tiles_w) * TH;
  const int tx = tid % TW, ty = tid / TW;
  const bool valid = w0 + tx < s.out[2] && h0 + ty < s.out[1];
  const int od0 = chunk * s.chunk_len, od1 = min(od0 + s.chunk_len, s.out[0]);
  const int zend = od1 + kd - 1;  // input planes [od0, zend)
  const int rows = TH + kh - 1, cols = TW + kw - 1;
  const int64_t plane = (int64_t)H * W * C;
  const T* xa = a + (int64_t)i * D * plane + c;
  const T* yb = b + (int64_t)j * D * plane + c;

  float ring[R][5];
  float acc_ssim = 0.f, acc_cs = 0.f;
  for (int zb = od0; zb < zend; zb += R) {
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int z = zb + r;
      if (z >= zend) break;
      __syncthreads();  // the previous plane's readers of sx / sy / hw are done
      for (int e = tid; e < rows * cols; e += kSsimThreads) {
        const int rr = e / cols, q = e - rr * cols, h = h0 + rr, w = w0 + q;
        float xv = 0.f, yv = 0.f;
        if (h < H && w < W) {
          const int64_t off = z * plane + ((int64_t)h * W + w) * C;
          xv = to_f(xa[off]);
          yv = to_f(yb[off]);
        }
        sx[e] = xv;
        sy[e] = yv;
      }
      __syncthreads();
      for (int e = tid; e < rows * TW; e += kSsimThreads) {  // W filter of the five products, halo rows included
        const int rr = e / TW, q = e % TW;
        const float* px = sx + rr * cols + q;
        const float* py = sy + rr * cols + q;
        float m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f, m4 = 0.f;
        for (int t = 0; t < kw; ++t) {
          const float g = taps[2][t], xv = px[t], yv = py[t];
          m0 = fmaf(g, xv, m0);
          m1 = fmaf(g, yv, m1);
          m2 = fmaf(g, xv * xv, m2);
          m3 = fmaf(g, yv * yv, m3);
          m4 = fmaf(g, xv * yv, m4);
        }
        hw[0][e] = m0;
        hw[1][e] = m1;
        hw[2][e] = m2;
        hw[3][e] = m3;
        hw[4][e] = m4;
      }
      __syncthreads();
#pragma unroll
      for (int q = 0; q < 5; ++q) ring[r][q] = 0.f;
      for (int t = 0; t < kh; ++t) {  // H filter: this thread's output voxel of plane z
        const float g = taps[1][t];
        const int e = (ty + t) * TW + tx;
#pragma unroll
        for (int q = 0; q < 5; ++q) ring[r][q] = fmaf(g, hw[q][e], ring[r][q]);
      }
      if (z - od0 >= kd - 1) {  // D filter over planes z - kd + 1 .. z: output plane z - kd + 1
        float m[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int u = 0; u < R; ++u) {
          if (u < kd) {
            const float g = taps[0][kd - 1 - u];
#pragma unroll
            for (int q = 0; q < 5; ++q) m[q] = fmaf(g, ring[(r - u + R) % R][q], m[q]);
          }
        }
        const float mx = m[0], my = m[1];
        const float sxx = m[2] - mx * mx, syy = m[3] - my * my, sxy = m[4] - mx * my;
        const float cs = (2.f * sxy + s.c2) / (sxx + syy + s.c2);
        const float lum = (2.f * mx * my + s.c1) / (__fadd_rn(__fmul_rn(mx, mx), __fmul_rn(my, my)) + s.c1);
        if (valid) {
          acc_ssim += lum * cs;
          acc_cs += cs;
        }
      }
    }
  }
  acc_ssim = warp_sum(acc_ssim);
  acc_cs = warp_sum(acc_cs);
  if ((tid & 31) == 0) {
    wsum[0][tid >> 5] = acc_ssim;
    wsum[1][tid >> 5] = acc_cs;
  }
  __syncthreads();
  if (tid == 0) {
    double ts = 0.0, tc = 0.0;
    for (int w = 0; w < kSsimThreads / 32; ++w) {
      ts += wsum[0][w];
      tc += wsum[1][w];
    }
    partial[blockIdx.x] = make_double2(ts, tc);
  }
}

// out[p] = (mean ssim, mean cs) of pair p: its `per_pair` CTA partials added in a fixed order (one warp per pair)
__global__ void __launch_bounds__(256) ssim_finish_kernel(const double2* __restrict__ partial, int64_t per_pair,
                                                          double inv_count, double* __restrict__ out, int P) {
  const int p = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (p >= P) return;
  const double2* src = partial + (int64_t)p * per_pair;
  double ts = 0.0, tc = 0.0;
  for (int64_t e = lane; e < per_pair; e += 32) {
    ts += src[e].x;
    tc += src[e].y;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ts += __shfl_xor_sync(0xffffffffu, ts, o);
    tc += __shfl_xor_sync(0xffffffffu, tc, o);
  }
  if (lane == 0) {
    out[2 * p] = ts * inv_count;
    out[2 * p + 1] = tc * inv_count;
  }
}

struct SsimPlan {
  int out[3], tiles_w, tiles, chunks, chunk_len;
  int64_t ctas;
};

static SsimPlan ssim_plan(int32_t P, int32_t C, const int32_t dims[3], const int32_t ksize[3]) {
  SsimPlan pl;
  for (int a = 0; a < 3; ++a) pl.out[a] = dims[a] - ksize[a] + 1;
  pl.tiles_w = (pl.out[2] + kSsimTW - 1) / kSsimTW;
  pl.tiles = pl.tiles_w * ((pl.out[1] + kSsimTH - 1) / kSsimTH);
  const int64_t base = (int64_t)P * C * pl.tiles;
  int chunks = 1;
  if (base < kSsimTargetCtas) {
    // split D, but keep each chunk at least twice the kd - 1 recomputed overlap planes long
    const int min_len = ksize[0] - 1 > 2 ? 2 * (ksize[0] - 1) : 4;
    chunks = (int)((kSsimTargetCtas + base - 1) / base);
    chunks = min(chunks, max(1, pl.out[0] / min_len));
  }
  pl.chunk_len = (pl.out[0] + chunks - 1) / chunks;
  pl.chunks = (pl.out[0] + pl.chunk_len - 1) / pl.chunk_len;
  pl.ctas = base * pl.chunks;
  return pl;
}

static bool ssim_shape_ok(int32_t P, int32_t C, const int32_t* dims, const int32_t* ksize) {
  if (!dims || !ksize || P < 0 || C <= 0) return false;
  for (int a = 0; a < 3; ++a)
    if (ksize[a] < 1 || ksize[a] > kSsimKMax || dims[a] < ksize[a]) return false;
  return true;
}

}  // namespace mig

using namespace mig;

extern "C" int64_t mig_ssim_workspace_bytes(int32_t P, int32_t C, const int32_t dims[3], const int32_t ksize[3]) {
  if (!ssim_shape_ok(P, C, dims, ksize)) return -1;
  return ssim_plan(P, C, dims, ksize).ctas * (int64_t)sizeof(double2);
}

extern "C" int mig_ssim_pairs(int dtype, const void* a, const void* b, int32_t na, int32_t nb, const int32_t* pairs,
                              int32_t P, const int32_t dims[3], int32_t C, const int32_t ksize[3],
                              const float* taps_host, float c1, float c2, double* out, void* workspace,
                              int64_t workspace_bytes, void* stream) {
  MIG_REQUIRE(dims && ksize && taps_host, "ssim_pairs: dims, ksize and taps_host must not be NULL");
  MIG_REQUIRE(C > 0, "ssim_pairs: C must be positive, got %d", (int)C);
  MIG_REQUIRE(P >= 0 && na > 0 && nb > 0, "ssim_pairs: need P >= 0 and na, nb > 0 (P=%d na=%d nb=%d)", (int)P, (int)na,
              (int)nb);
  for (int ax = 0; ax < 3; ++ax)
    MIG_REQUIRE(ksize[ax] >= 1 && ksize[ax] <= kSsimKMax && dims[ax] >= ksize[ax],
                "ssim_pairs: window %d on axis %d needs 1 <= k <= %d and k <= the extent %d", (int)ksize[ax], ax,
                kSsimKMax, (int)dims[ax]);
  if (P == 0) return 0;
  MIG_REQUIRE(a && b && pairs && out, "ssim_pairs: a, b, pairs and out must not be NULL");
  const SsimPlan pl = ssim_plan(P, C, dims, ksize);
  MIG_REQUIRE(pl.ctas <= 0x7fffffffLL, "ssim_pairs: %lld CTAs exceed the grid limit", (long long)pl.ctas);
  const int64_t need = pl.ctas * (int64_t)sizeof(double2);
  MIG_REQUIRE(workspace && workspace_bytes >= need, "ssim_pairs: workspace too small (%lld < %lld bytes)",
              (long long)workspace_bytes, (long long)need);

  SsimArgs s{};
  int off = 0;
  for (int ax = 0; ax < 3; ++ax) {
    for (int t = 0; t < ksize[ax]; ++t) s.taps[ax][t] = taps_host[off + t];
    off += ksize[ax];
    s.k[ax] = ksize[ax];
    s.dims[ax] = dims[ax];
    s.out[ax] = pl.out[ax];
  }
  s.C = C;
  s.na = na;
  s.nb = nb;
  s.tiles_w = pl.tiles_w;
  s.tiles = pl.tiles;
  s.chunks = pl.chunks;
  s.chunk_len = pl.chunk_len;
  s.c1 = c1;
  s.c2 = c2;
  cudaStream_t st = as_stream(stream);
  double2* partial = (double2*)workspace;
  const int kd = ksize[0];
  MIG_DISPATCH_DTYPE(dtype, TT, {
    const TT* A = (const TT*)a;
    const TT* B = (const TT*)b;
    if (kd == 1) ssim_partial_kernel<TT, 1><<<(unsigned)pl.ctas, kSsimThreads, 0, st>>>(A, B, pairs, s, partial);
    else if (kd <= 4) ssim_partial_kernel<TT, 4><<<(unsigned)pl.ctas, kSsimThreads, 0, st>>>(A, B, pairs, s, partial);
    else if (kd <= 8) ssim_partial_kernel<TT, 8><<<(unsigned)pl.ctas, kSsimThreads, 0, st>>>(A, B, pairs, s, partial);
    else if (kd <= 12) ssim_partial_kernel<TT, 12><<<(unsigned)pl.ctas, kSsimThreads, 0, st>>>(A, B, pairs, s, partial);
    else ssim_partial_kernel<TT, 16><<<(unsigned)pl.ctas, kSsimThreads, 0, st>>>(A, B, pairs, s, partial);
  });
  const int64_t per_pair = pl.ctas / P;
  const double inv_count = 1.0 / ((double)C * pl.out[0] * pl.out[1] * pl.out[2]);
  ssim_finish_kernel<<<(unsigned)((P + 7) / 8), 256, 0, st>>>(partial, per_pair, inv_count, out, P);
  return check_launch("ssim_pairs");
}

// tcgen05 engine, part 4: narrow-channel convolution (Cin = 32, Cout <= 32, stride 1) with a shared-memory-resident
// halo tile -- the 32-channel full-resolution layers of the AutoencoderKL (ae:158-176 at 96^3) and of pixel-space
// DDPM U-Nets (BASELINE configs 2 and 4).
//
// With 32 channels an implicit GEMM has N = 32 and K = 27*32: the tensor cores are idle and the cost is operand feed.
// The generic kernels read every input voxel once per tap (27x). Here a persistent CTA
//   1. keeps the WHOLE filter (27 x 32 x Cout bf16 = 55 KB) in shared memory for its lifetime,
//   2. TMA-loads an output tile's input footprint (8x16x1 voxels + halo = 10x18x3 voxels x 64 B) ONCE,
//   3. re-lays it out in smem as four 8-channel planes [chunk][voxel] x 16 B, which is the UMMA "no swizzle" K-major
//      core-matrix format (8 rows x 16 B contiguous): a filter tap is then just a different START ADDRESS of the same
//      planes (leading byte offset = plane stride, stride byte offset = one voxel line), no data movement,
//   4. issues 27 taps x 2 UMMAs (128 x N x 16) into a double-buffered TMEM accumulator, while the next tile's halo
//      is in flight and the previous tile's epilogue (+bias, +time embedding, +residual, bf16 store) runs.
// Input traffic drops from 27x to 4.2x (halo overhead) and all address arithmetic disappears from the main loop.
// fwd and dgrad (mirrored taps, transposed filter) share the kernel.
#include <cuda.h>

#include "common.cuh"
#include "residue_classes.cuh"
#include "tc_common.cuh"
#include "tc_host.cuh"

namespace mig {

using namespace tc;

int filter_transpose(int dtype, const void* w, void* wt, int Cout, int Tn, int Cin, void* stream);

constexpr int HT_X = 8, HT_Y = 16;            // output tile: 8 (x) x 16 (y) x 1 (z) = 128 voxels = UMMA M
constexpr int H_THREADS = 192;
constexpr int H_C = 32;                        // source channels
constexpr int H_MAXVOX = (HT_X + 2) * (HT_Y + 2) * 3;

__device__ __forceinline__ void tma_load_5d_h(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2,
                                              int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::
          "r"(dst),
      "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
// no-swizzle K-major descriptor: core matrix = 8 rows x 16 bytes stored contiguously (128 B);
// LBO = byte distance between the two 8-element K chunks of one UMMA, SBO = byte distance between 8-row groups
__device__ __forceinline__ uint64_t make_desc_noswz(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;   // descriptor version (sm_100); layout type bits [61,64) = 0: no swizzle
  return d;
}

struct HaloParams {
  int N, D, H, W;         // SOURCE extent
  int OD, OH, OW;         // output extent
  int ks[3];              // filter size (each <= 3)
  int lo[3];              // halo origin relative to the output coordinate: src = out + lo + h, h in [0, hz/hy/hx)
  int hz, hy, hx;         // halo extent: 1+kz-1, 16+ky-1, 8+kx-1
  int sign;               // +1 fwd (halo offset of tap t = t), -1 dgrad (ks-1-t)
  int Cdst, Npad;         // output channels, UMMA N (16 or 32)
  // where an output row lands: coordinate = row*os + oo inside a (TD,TH,TW) tensor (identity except strided dgrad,
  // where each stride-residue class of input voxels is its own dense problem)
  int os[3], oo[3], TD, TH, TW;
  int tiles_x, tiles_y;
  int64_t num_tiles;      // N*OD*tiles_y*tiles_x
  const __nv_bfloat16* w; // [Cdst][taps][32]
  const float* bias;
  const float* chan_bias;
  const __nv_bfloat16* residual;
  __nv_bfloat16* out;
};

__global__ void __launch_bounds__(H_THREADS, 1) conv_halo_kernel(const __grid_constant__ CUtensorMap xmap, HaloParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 127u) & ~127u;
  const int T = p.ks[0] * p.ks[1] * p.ks[2];
  const int nvox = p.hz * p.hy * p.hx;
  // one 8-channel plane, padded so that the four planes start 32 B apart modulo 128 B: the 16-byte re-layout stores of
  // a quarter warp (2 voxels x 4 planes) then hit eight different 16-byte bank groups
  const uint32_t plane = (uint32_t)nvox * 16u + ((160u - ((uint32_t)nvox * 16u) % 128u) % 128u);
  const uint32_t stage_bytes = (uint32_t)nvox * 64u;    // TMA staging [voxel][32 ch]
  const uint32_t w_bytes = (uint32_t)T * 4u * p.Npad * 16u;
  const uint32_t w_smem = smem_base;
  const uint32_t stg_smem = (w_smem + w_bytes + 127u) & ~127u;
  const uint32_t stg_stride = (stage_bytes + 127u) & ~127u;
  // two staging buffers when they fit; with a 64-wide filter (110 KB resident) only one
  const int nstg = p.Npad > 32 ? 1 : 2;
  const uint32_t pl_smem = stg_smem + nstg * stg_stride;
  const uint32_t pl_stride = (4u * plane + 127u) & ~127u;
  __shared__ __align__(8) uint64_t bars[12];
  __shared__ uint32_t tmem_slot;
  __shared__ __align__(16) float add_s[2][64];   // bias + per-sample channel bias of the tile in accumulator a
  const uint32_t b0 = smem_u32(&bars[0]);
  const uint32_t stg_full = b0, stg_empty = b0 + 16, pl_full = b0 + 32, pl_empty = b0 + 48, acc_full = b0 + 64,
                 acc_empty = b0 + 80;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(stg_full + 8 * i, 1);  mbar_init(stg_empty + 8 * i, 128);
      mbar_init(pl_full + 8 * i, 128); mbar_init(pl_empty + 8 * i, 1);
      mbar_init(acc_full + 8 * i, 1);  mbar_init(acc_empty + 8 * i, 128);
    }
    fence_barrier_init();
  }
  if (warp == 4) tmem_alloc<128>(smem_u32(&tmem_slot));
  if (warp == 5 && lane == 0) tma_prefetch_desc(&xmap);
  // resident filter: global [co][tap][32] -> smem [tap][chunk][n][8 ch] (16-byte units), rows n >= Cdst are zero
  for (int i = threadIdx.x; i < T * 4 * p.Npad; i += H_THREADS) {
    const int n = i % p.Npad, c = (i / p.Npad) & 3, tap = i / (p.Npad * 4);
    uint4 v = make_uint4(0, 0, 0, 0);
    if (n < p.Cdst) v = *reinterpret_cast<const uint4*>(p.w + ((int64_t)n * T + tap) * H_C + c * 8);
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(w_smem + (uint32_t)i * 16u), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w) : "memory");
  }
  fence_proxy_async();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_slot;
  const int64_t my_tiles = p.num_tiles > blockIdx.x ? (p.num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  // 32-bit arithmetic (the host refuses more than 2^31 tiles): these divisions sit on every role's per-tile path
  auto tile_coords = [&](int64_t i, int& n, int& z, int& y0, int& x0) {
    uint32_t t = blockIdx.x + (uint32_t)i * gridDim.x;
    uint32_t q = t / (uint32_t)p.tiles_x;
    x0 = (int)(t - q * p.tiles_x) * HT_X; t = q;
    q = t / (uint32_t)p.tiles_y;
    y0 = (int)(t - q * p.tiles_y) * HT_Y; t = q;
    q = t / (uint32_t)p.OD;
    z = (int)(t - q * p.OD);
    n = (int)q;
  };

  if (warp < 4) {
    // ============ workers: re-layout staging -> planes, then the epilogue of the previous tile ============
    const int r = warp * 32 + lane;
    auto epilogue = [&](int64_t i) {
      const int a = (int)(i & 1);
      mbar_wait(acc_full + 8 * a, (uint32_t)(i >> 1) & 1u);
      tcgen05_fence_after();
      int n, z, y0, x0;
      tile_coords(i, n, z, y0, x0);
      const int y = y0 + (r >> 3), x = x0 + (r & 7);
      const bool ok = y < p.OH && x < p.OW;
      const int64_t m = (((int64_t)n * p.TD + z * p.os[0] + p.oo[0]) * p.TH + y * p.os[1] + p.oo[1]) * p.TW +
                        x * p.os[2] + p.oo[2];
      const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16) + a * 64;
      // one TMEM round trip for the whole 64-column accumulator slot (columns >= Npad are stale and ignored)
      float vw[64];
      tmem_ld64(trow, vw);
#pragma unroll
      for (int c0 = 0; c0 < 64; c0 += 16) {
        if (c0 >= p.Npad || !ok) continue;
        float* v = vw + c0;
        const float4* ap = reinterpret_cast<const float4*>(&add_s[a][c0]);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float4 b4 = ap[e];
          v[4 * e] += b4.x; v[4 * e + 1] += b4.y; v[4 * e + 2] += b4.z; v[4 * e + 3] += b4.w;
        }
        __nv_bfloat16* dst = p.out + m * p.Cdst + c0;
        if (c0 + 16 <= p.Cdst && (p.Cdst & 7) == 0) {
          if (p.residual) {
            const uint4* rp = reinterpret_cast<const uint4*>(p.residual + m * p.Cdst + c0);
            uint4 r0 = rp[0], r1 = rp[1];
            const __nv_bfloat16* a0 = reinterpret_cast<const __nv_bfloat16*>(&r0);
            const __nv_bfloat16* a1 = reinterpret_cast<const __nv_bfloat16*>(&r1);
#pragma unroll
            for (int e = 0; e < 8; ++e) { v[e] += __bfloat162float(a0[e]); v[8 + e] += __bfloat162float(a1[e]); }
          }
          uint4 o0, o1;
          __nv_bfloat162* q0 = reinterpret_cast<__nv_bfloat162*>(&o0);
          __nv_bfloat162* q1 = reinterpret_cast<__nv_bfloat162*>(&o1);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            q0[e] = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
            q1[e] = __floats2bfloat162_rn(v[8 + 2 * e], v[8 + 2 * e + 1]);
          }
          reinterpret_cast<uint4*>(dst)[0] = o0;
          reinterpret_cast<uint4*>(dst)[1] = o1;
        } else {
#pragma unroll
          for (int e = 0; e < 16; ++e)
            if (c0 + e < p.Cdst) {
              float rr = p.residual ? __bfloat162float(p.residual[m * p.Cdst + c0 + e]) : 0.f;
              dst[e] = __float2bfloat16_rn(v[e] + rr);
            }
        }
      }
      tcgen05_fence_before();
      mbar_arrive(acc_empty + 8 * a);
    };
    for (int64_t i = 0; i < my_tiles; ++i) {
      const int s = (int)(i & 1);
      const uint32_t ph = (uint32_t)(i >> 1) & 1u;
      const int ss = nstg == 2 ? s : 0;
      mbar_wait(stg_full + 8 * ss, nstg == 2 ? ph : (uint32_t)i & 1u);
      mbar_wait(pl_empty + 8 * s, ph ^ 1u);
      // every worker is past epilogue(i-2), the last reader of add_s[s]; the barrier of iteration i+1 (or the one
      // before the final epilogue) orders these writes before epilogue(i) reads them
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (r < 64) {
        float add = 0.f;
        if (r < p.Cdst) {
          int n, z, y0, x0;
          tile_coords(i, n, z, y0, x0);
          if (p.bias) add += p.bias[r];
          if (p.chan_bias) add += p.chan_bias[(int64_t)n * p.Cdst + r];
        }
        add_s[s][r] = add;
      }
      const uint32_t src = stg_smem + ss * stg_stride, dst = pl_smem + s * pl_stride;
      // six 16-byte moves per round: the loads are issued back to back, then the stores (one dependent load -> store
      // pair per iteration left the workers waiting on shared-memory latency 17 times per tile)
      for (int idx0 = r; idx0 < nvox * 4; idx0 += 6 * 128) {
        uint32_t a[6][4];
#pragma unroll
        for (int u = 0; u < 6; ++u) {
          const int idx = idx0 + u * 128;
          if (idx < nvox * 4)
            asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(a[u][0]), "=r"(a[u][1]), "=r"(a[u][2]), "=r"(a[u][3])
                         : "r"(src + idx * 16));
        }
#pragma unroll
        for (int u = 0; u < 6; ++u) {
          const int idx = idx0 + u * 128;
          if (idx < nvox * 4)
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(dst + (idx & 3) * plane + (idx >> 2) * 16), "r"(a[u][0]),
                         "r"(a[u][1]), "r"(a[u][2]), "r"(a[u][3]) : "memory");
        }
      }
      fence_proxy_async();
      mbar_arrive(pl_full + 8 * s);
      mbar_arrive(stg_empty + 8 * ss);
      if (i >= 1) epilogue(i - 1);
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");
    if (my_tiles >= 1) epilogue(my_tiles - 1);
  } else if (warp == 4) {
    // ============ UMMA issuer: 27 taps x 2 K-steps per tile, A = shifted windows of the planes ============
    const uint32_t idesc = make_idesc(128, p.Npad, 0, 0);
    const uint32_t sbo_a = (uint32_t)p.hx * 16u;
    for (int64_t i = 0; i < my_tiles; ++i) {
      const int s = (int)(i & 1);
      const uint32_t ph = (uint32_t)(i >> 1) & 1u;
      mbar_wait(pl_full + 8 * s, ph);
      mbar_wait(acc_empty + 8 * s, ph ^ 1u);
      tcgen05_fence_after();
      if (elect_one()) {
        // The UMMAs are tiny (128 x N x 16 = 16 tensor cycles), so the single issuing thread is the limiter: the
        // descriptors are built once per tile and advanced with ONE 64-bit add per UMMA (the start-address field is
        // the low 14 bits in 16-byte units; shared-memory addresses never carry out of it).
        const uint32_t acc = tmem_base + s * 64;
        const uint64_t a0 = make_desc_noswz(pl_smem + s * pl_stride, plane, sbo_a);
        const uint64_t a_ks = (uint64_t)((2u * plane) >> 4);
        uint64_t bd = make_desc_noswz(w_smem, p.Npad * 16u, 128u);
        const uint64_t b_ks = (uint64_t)((2u * p.Npad * 16u) >> 4);
        uint32_t first = 0;
        for (int t0 = 0; t0 < p.ks[0]; ++t0) {
          const int h0 = p.sign > 0 ? t0 : p.ks[0] - 1 - t0;
          for (int t1 = 0; t1 < p.ks[1]; ++t1) {
            const int h1 = p.sign > 0 ? t1 : p.ks[1] - 1 - t1;
            const uint64_t row = a0 + (uint64_t)((h0 * p.hy + h1) * p.hx);
#pragma unroll 3
            for (int t2 = 0; t2 < p.ks[2]; ++t2) {
              const uint64_t ad = row + (uint64_t)(p.sign > 0 ? t2 : p.ks[2] - 1 - t2);
              umma_bf16(acc, ad, bd, idesc, first);
              first = 1u;
              umma_bf16(acc, ad + a_ks, bd + b_ks, idesc, 1u);
              bd += 2 * b_ks;
            }
          }
        }
        umma_commit(pl_empty + 8 * s);
        umma_commit(acc_full + 8 * s);
      }
      __syncwarp();
    }
  } else if (elect_one()) {
    // ============ TMA issuer: one halo box per tile ============
    for (int64_t i = 0; i < my_tiles; ++i) {
      const int s = nstg == 2 ? (int)(i & 1) : 0;
      mbar_wait(stg_empty + 8 * s, ((nstg == 2 ? (uint32_t)(i >> 1) : (uint32_t)i) & 1u) ^ 1u);
      int n, z, y0, x0;
      tile_coords(i, n, z, y0, x0);
      mbar_arrive_expect_tx(stg_full + 8 * s, stage_bytes);
      tma_load_5d_h(stg_smem + s * stg_stride, &xmap, stg_full + 8 * s, 0, x0 + p.lo[2], y0 + p.lo[1], z + p.lo[0], n);
    }
  }
  __syncthreads();
  if (warp == 4) {
    tcgen05_fence_after();
    tmem_dealloc<128>(tmem_base);
  }
}

// which: 0 fwd, 1 dgrad
bool halo_conv_eligible(const mig_conv_geom* g, int which) {
  const int csrc = which == 1 ? g->Cout : g->Cin, cdst = which == 1 ? g->Cin : g->Cout;
  if (csrc != H_C || cdst < 1 || cdst > 64) return false;
  for (int i = 0; i < 3; ++i)
    if (g->stride[i] != 1 || g->ksize[i] > 3) return false;
  const int64_t vox = (int64_t)g->N * g->out_dims[0] * g->out_dims[1] * g->out_dims[2];
  const int32_t* od = which == 1 ? g->in_dims : g->out_dims;
  return vox >= 32768 && od[2] >= HT_X && od[1] >= HT_Y / 2;
}

// one dense stride-1 problem: rows (n, z, y, x) over ext[], source voxel = row + lo + halo offset
struct HaloProblem {
  int N;
  int src[3];       // source extent
  int ext[3];       // row extent (the output tensor itself, or one stride-residue class of it)
  int ks[3], lo[3];
  int sign;
  int Cdst;
  int os[3], oo[3], tgt[3];   // row -> output coordinate = row*os + oo inside tgt[]
};

// 5-d map (C, W, H, D, N) with box (C, bx, by, bz, 1), no swizzle: staging rows are plain voxels of C channels
static int halo_map(CUtensorMap* m, const void* base, int N, int D, int H, int W, int C, int bx, int by, int bz) {
  const uint64_t dims[5] = {(uint64_t)C, (uint64_t)W, (uint64_t)H, (uint64_t)D, (uint64_t)N};
  const uint64_t strides[4] = {(uint64_t)C * 2, (uint64_t)W * C * 2, (uint64_t)H * W * C * 2,
                               (uint64_t)D * H * W * C * 2};
  const uint32_t box[5] = {(uint32_t)C, (uint32_t)bx, (uint32_t)by, (uint32_t)bz, 1};
  return make_map(m, base, 5, dims, strides, box, "halo map", CU_TENSOR_MAP_SWIZZLE_NONE);
}

static int launch_halo(const HaloProblem& h, const void* src, const void* wk, const float* bias, const float* chan_bias,
                       const void* residual, void* out, void* stream) {
  HaloParams p{};
  p.N = h.N; p.D = h.src[0]; p.H = h.src[1]; p.W = h.src[2];
  p.OD = h.ext[0]; p.OH = h.ext[1]; p.OW = h.ext[2];
  p.sign = h.sign;
  for (int i = 0; i < 3; ++i) { p.ks[i] = h.ks[i]; p.lo[i] = h.lo[i]; p.os[i] = h.os[i]; p.oo[i] = h.oo[i]; }
  p.TD = h.tgt[0]; p.TH = h.tgt[1]; p.TW = h.tgt[2];
  p.hz = 1 + p.ks[0] - 1; p.hy = HT_Y + p.ks[1] - 1; p.hx = HT_X + p.ks[2] - 1;
  p.Cdst = h.Cdst;
  p.Npad = p.Cdst <= 16 ? 16 : p.Cdst <= 32 ? 32 : 64;
  p.tiles_x = (p.OW + HT_X - 1) / HT_X;
  p.tiles_y = (p.OH + HT_Y - 1) / HT_Y;
  p.num_tiles = (int64_t)p.N * p.OD * p.tiles_y * p.tiles_x;
  p.w = (const __nv_bfloat16*)wk;
  p.bias = bias; p.chan_bias = chan_bias;
  p.residual = (const __nv_bfloat16*)residual;
  p.out = (__nv_bfloat16*)out;
  CUtensorMap xm;
  if (halo_map(&xm, src, p.N, p.D, p.H, p.W, H_C, p.hx, p.hy, p.hz)) return 1;
  const int T = p.ks[0] * p.ks[1] * p.ks[2];
  const int nvox = p.hz * p.hy * p.hx;
  const int nstg = p.Npad > 32 ? 1 : 2;
  const int smem = T * 4 * p.Npad * 16 + nstg * (nvox * 64 + 128) + 2 * (nvox * 64 + 512 + 128) + 512;
  static SmemOptIn optin;
  if (int rc = ensure_dynamic_smem(conv_halo_kernel, smem, optin, "conv_halo")) return rc;
  int64_t grid = device_info().sm_count;
  if (grid > p.num_tiles) grid = p.num_tiles;
  conv_halo_kernel<<<(unsigned)grid, H_THREADS, smem, as_stream(stream)>>>(xm, p);
  return check_launch("conv_halo_kernel");
}

static int run_halo(const mig_conv_geom* g, int which, const void* src, const void* wk, const float* bias,
                    const float* chan_bias, const void* residual, void* out, void* stream) {
  HaloProblem h{};
  const int32_t* sd = which == 1 ? g->out_dims : g->in_dims;   // source extent
  const int32_t* od = which == 1 ? g->in_dims : g->out_dims;   // extent of the tensor being produced
  h.N = g->N;
  h.sign = which == 1 ? -1 : 1;
  for (int i = 0; i < 3; ++i) {
    h.src[i] = sd[i]; h.ext[i] = od[i]; h.tgt[i] = od[i]; h.os[i] = 1; h.oo[i] = 0;
    h.ks[i] = g->ksize[i];
    const int off = which == 1 ? g->pad[i] : -g->pad[i];
    h.lo[i] = off + (h.sign > 0 ? 0 : -(g->ksize[i] - 1));
  }
  h.Cdst = which == 1 ? g->Cin : g->Cout;
  return launch_halo(h, src, wk, bias, chan_bias, residual, out, stream);
}

// ---------------------------------------------------------------------------------------------------
// strided dgrad (the backward of the 32-channel Downsample convolution) by stride-residue classes
// ---------------------------------------------------------------------------------------------------
// Every class (residue_classes.cuh) is a dense stride-1 problem with a sub-filter (8 classes of 1..8 taps for k = 3,
// s = 2), whose rows scatter into dx with the stride. Here each class runs on the halo kernel.
bool halo_dgrad_strided_eligible(const mig_conv_geom* g) {
  if (g->Cout != H_C || g->Cin < 1 || g->Cin > 64) return false;
  bool any = false;
  for (int i = 0; i < 3; ++i) {
    if (g->stride[i] < 1 || g->stride[i] > 2 || g->ksize[i] > 3) return false;
    any = any || g->stride[i] == 2;
  }
  if (!any) return false;
  const int64_t vox = (int64_t)g->N * g->in_dims[0] * g->in_dims[1] * g->in_dims[2];
  if (vox < 32768) return false;
  for (int r1 = 0; r1 < g->stride[1]; ++r1)
    if (axis_class(g->in_dims[1], g->ksize[1], g->stride[1], g->pad[1], r1).ext < HT_Y / 2) return false;
  for (int r2 = 0; r2 < g->stride[2]; ++r2)
    if (axis_class(g->in_dims[2], g->ksize[2], g->stride[2], g->pad[2], r2).ext < HT_X) return false;
  return true;
}

int halo_conv_dgrad_strided(const mig_conv_geom* g, const void* dy, const void* w, void* dx, void* ws, int64_t ws_bytes,
                            void* stream) {
  auto launch_class = [&](const ResidueClass& c, const void* wsub) {
    HaloProblem h{};
    h.N = g->N;
    h.sign = -1;
    h.Cdst = g->Cin;
    for (int i = 0; i < 3; ++i) {
      const AxisClass& a = c.a[i];
      h.src[i] = g->out_dims[i]; h.ext[i] = a.ext; h.tgt[i] = g->in_dims[i];
      h.ks[i] = a.nu; h.lo[i] = a.base - (a.nu - 1);
      h.os[i] = g->stride[i]; h.oo[i] = a.o;
    }
    return launch_halo(h, dy, wsub, nullptr, nullptr, nullptr, dx, stream);
  };
  return dgrad_by_residue_classes(g, w, dx, ws, ws_bytes, stream, "conv_dgrad(halo, strided)", launch_class);
}

// ---------------------------------------------------------------------------------------------------
// wgrad for the same layers: dW[co][tap*32 + ci] += sum_v dY[v][co] * X[v + tap][ci]
// ---------------------------------------------------------------------------------------------------
// Both operands are MN-major no-swizzle planes in shared memory: X halo planes [ci chunk][voxel] x 16 B (the same
// re-layout as the forward kernel; a tap is a start-address offset) and dY planes [co chunk][voxel] x 16 B. One UMMA
// (64 x 32 x 16) reduces 16 voxels (two 8-voxel lines) of one tap; a CTA owns half of the taps (grid parity) and
// keeps ALL of its tap accumulators (<= 14 x 32 columns) in tensor memory over its whole tile loop, so the fp32
// reduction into dW happens once per CTA. Output channel m sits in TMEM lane (m % 16) + 32 (m / 16) (M = 64 layout); the chunks above Cout read
// zero planes.
struct HaloWgradParams {
  int N, D, H, W;          // X extent
  int OD, OH, OW;          // dY extent
  int ks[3], lo[3];
  int hz, hy, hx;
  int Cout;                // <= 32, multiple of 8
  int tiles_x, tiles_y;
  int64_t num_tiles;
  int taps_total, taps_per_half;
  float* dw;               // [Cout][taps][32]
};

__global__ void __launch_bounds__(H_THREADS, 1) wgrad_halo_kernel(const __grid_constant__ CUtensorMap xmap,
                                                                  const __grid_constant__ CUtensorMap dymap,
                                                                  HaloWgradParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 127u) & ~127u;
  const int nvox = p.hz * p.hy * p.hx;
  // plane strides are padded by 16 B so that consecutive channel-chunk planes start in different shared-memory banks
  // (a multiple of 128 B would put every chunk of a UMMA operand fetch on the same banks)
  const uint32_t xplane = (uint32_t)nvox * 16u + ((160u - ((uint32_t)nvox * 16u) % 128u) % 128u);
  const uint32_t x_stage_bytes = (uint32_t)nvox * 64u;
  const uint32_t dy_stage_bytes = 128u * (uint32_t)p.Cout * 2u;
  constexpr uint32_t dyplane = 128u * 16u + 16u;              // one 8-channel plane of the 128-voxel dY tile
  // layout: [X staging][dY staging][X planes x2][dY planes x2 (8 chunk planes each = the 64 rows of an M = 64 UMMA;
  // chunks >= Cout/8 stay zero)]
  const uint32_t xs_smem = smem_base;
  const uint32_t dys_smem = (xs_smem + x_stage_bytes + 127u) & ~127u;
  const uint32_t xp_smem = (dys_smem + dy_stage_bytes + 127u) & ~127u;
  const uint32_t xp_stride = (4u * xplane + 127u) & ~127u;
  const uint32_t dyp_smem = xp_smem + 2 * xp_stride;
  constexpr uint32_t dyp_stride = 8u * dyplane;
  __shared__ __align__(8) uint64_t bars[8];
  __shared__ uint32_t tmem_slot;
  const uint32_t b0 = smem_u32(&bars[0]);
  const uint32_t stg_full = b0, stg_empty = b0 + 8, pl_full = b0 + 16 /*2*/, pl_empty = b0 + 32 /*2*/, acc_done = b0 + 48;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int half = blockIdx.x & 1;
  const int tap_begin = half * p.taps_per_half;
  const int ntap = min(p.taps_total, tap_begin + p.taps_per_half) - tap_begin;
  const int cta = blockIdx.x >> 1, nctas = gridDim.x >> 1;
  const int64_t my_tiles = p.num_tiles > cta ? (p.num_tiles - cta + nctas - 1) / nctas : 0;

  if (threadIdx.x == 0) {
    mbar_init(stg_full, 1); mbar_init(stg_empty, 128);
    for (int i = 0; i < 2; ++i) { mbar_init(pl_full + 8 * i, 128); mbar_init(pl_empty + 8 * i, 1); }
    mbar_init(acc_done, 1);
    fence_barrier_init();
  }
  if (warp == 4) tmem_alloc<512>(smem_u32(&tmem_slot));
  if (warp == 5 && lane == 0) { tma_prefetch_desc(&xmap); tma_prefetch_desc(&dymap); }
  // zero the dY planes once (the chunk planes >= Cout/8 are never written again)
  for (uint32_t i = threadIdx.x; i < 2 * dyp_stride / 16; i += H_THREADS)
    asm volatile("st.shared.v4.b32 [%0], {%1,%1,%1,%1};" ::"r"(dyp_smem + i * 16u), "r"(0u) : "memory");
  fence_proxy_async();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_slot;

  auto tile_coords = [&](int64_t i, int& n, int& z, int& y0, int& x0) {
    uint32_t t = (uint32_t)cta + (uint32_t)i * (uint32_t)nctas;
    uint32_t q = t / (uint32_t)p.tiles_x;
    x0 = (int)(t - q * p.tiles_x) * HT_X; t = q;
    q = t / (uint32_t)p.tiles_y;
    y0 = (int)(t - q * p.tiles_y) * HT_Y; t = q;
    q = t / (uint32_t)p.OD;
    z = (int)(t - q * p.OD);
    n = (int)q;
  };

  if (warp < 4) {
    const int r = warp * 32 + lane;
    const int nchunk = p.Cout / 8;
    for (int64_t i = 0; i < my_tiles; ++i) {
      const int s = (int)(i & 1);
      const uint32_t ph = (uint32_t)(i >> 1) & 1u;
      mbar_wait(stg_full, (uint32_t)i & 1u);
      mbar_wait(pl_empty + 8 * s, ph ^ 1u);
      const uint32_t xdst = xp_smem + s * xp_stride, ddst = dyp_smem + s * dyp_stride;
      for (int idx0 = r; idx0 < nvox * 4; idx0 += 6 * 128) {
        uint32_t a[6][4];
#pragma unroll
        for (int u = 0; u < 6; ++u) {
          const int idx = idx0 + u * 128;
          if (idx < nvox * 4)
            asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(a[u][0]), "=r"(a[u][1]), "=r"(a[u][2]), "=r"(a[u][3])
                         : "r"(xs_smem + idx * 16));
        }
#pragma unroll
        for (int u = 0; u < 6; ++u) {
          const int idx = idx0 + u * 128;
          if (idx < nvox * 4)
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(xdst + (idx & 3) * xplane + (idx >> 2) * 16), "r"(a[u][0]),
                         "r"(a[u][1]), "r"(a[u][2]), "r"(a[u][3]) : "memory");
        }
      }
      // dY tile: TMA staged [voxel r][Cout] -> planes [chunk][voxel]; out-of-range voxels were zero-filled by TMA
      for (int c = 0; c < nchunk; ++c) {
        uint32_t a0, a1, a2, a3;
        asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3)
                     : "r"(dys_smem + (uint32_t)r * p.Cout * 2u + c * 16u));
        asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(ddst + c * dyplane + r * 16), "r"(a0), "r"(a1), "r"(a2),
                     "r"(a3) : "memory");
      }
      fence_proxy_async();
      mbar_arrive(pl_full + 8 * s);
      mbar_arrive(stg_empty);
    }
    // ---- epilogue: an M = 64 accumulator keeps row m in TMEM lane (m % 16) + 32 * (m / 16): warp w reads the dW rows
    // 16w .. 16w+15 from the first 16 lanes of its own quadrant; Cout <= 32 -> warps 0 and 1 carry data ----
    mbar_wait(acc_done, 0);
    tcgen05_fence_after();
    if (warp * 16 < p.Cout && my_tiles > 0) {
      const int co = warp * 16 + lane;
      const bool cok = lane < 16 && co < p.Cout;
      for (int t = 0; t < ntap; ++t) {
#pragma unroll 1
        for (int c0 = 0; c0 < 32; c0 += 16) {
          float v[16];
          tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + t * 32 + c0, v);
          if (cok) red_add_16(p.dw + ((int64_t)co * p.taps_total + tap_begin + t) * H_C + c0, v, 16);
        }
      }
    }
    tcgen05_fence_before();
  } else if (warp == 4) {
    const uint32_t idesc = make_idesc(64, 32, 1, 1);   // M = 64: the A fetch is 2 KB instead of 4 KB per UMMA
    const uint32_t lbo_b = (uint32_t)p.hx * 16u;   // next 8-voxel line of the X halo
    for (int64_t i = 0; i < my_tiles; ++i) {
      const int s = (int)(i & 1);
      mbar_wait(pl_full + 8 * s, (uint32_t)(i >> 1) & 1u);
      tcgen05_fence_after();
      if (elect_one()) {
        // descriptors built once per tile, advanced by one add per UMMA (the issuing thread is the limiter here)
        // A: dY planes, M = co chunks (SBO = plane), K = 16 voxels = lines 2yk, 2yk+1 (LBO = one 8-voxel line)
        const uint64_t a0 = make_desc_noswz(dyp_smem + s * dyp_stride, HT_X * 16u, dyplane);
        // B: X halo planes, N = ci chunks (SBO = plane), K = the same voxels shifted by the tap
        const uint64_t b0d = make_desc_noswz(xp_smem + s * xp_stride, lbo_b, xplane);
        const uint64_t a_inc = (uint64_t)(2 * HT_X), b_inc = (uint64_t)(2 * p.hx);   // two voxel lines, 16-byte units
        const uint32_t acc_flag = i ? 1u : 0u;
        int tap = tap_begin;
        int t2 = tap % p.ks[2], t1 = (tap / p.ks[2]) % p.ks[1], t0 = tap / (p.ks[2] * p.ks[1]);
        for (int t = 0; t < ntap; ++t) {
          const uint64_t bt = b0d + (uint64_t)((t0 * p.hy + t1) * p.hx + t2);
          const uint32_t acc = tmem_base + t * 32;
          umma_bf16(acc, a0, bt, idesc, acc_flag);
#pragma unroll
          for (int yk = 1; yk < HT_Y / 2; ++yk) umma_bf16(acc, a0 + yk * a_inc, bt + yk * b_inc, idesc, 1u);
          if (++t2 == p.ks[2]) { t2 = 0; if (++t1 == p.ks[1]) { t1 = 0; ++t0; } }
        }
        umma_commit(pl_empty + 8 * s);
        if (i == my_tiles - 1) umma_commit(acc_done);
      }
      __syncwarp();
    }
    if (my_tiles == 0 && lane == 0) mbar_arrive(acc_done);
  } else if (elect_one()) {
    for (int64_t i = 0; i < my_tiles; ++i) {
      mbar_wait(stg_empty, ((uint32_t)i & 1u) ^ 1u);
      int n, z, y0, x0;
      tile_coords(i, n, z, y0, x0);
      mbar_arrive_expect_tx(stg_full, x_stage_bytes + dy_stage_bytes);
      tma_load_5d_h(xs_smem, &xmap, stg_full, 0, x0 + p.lo[2], y0 + p.lo[1], z + p.lo[0], n);
      tma_load_5d_h(dys_smem, &dymap, stg_full, 0, x0, y0, z, n);
    }
  }
  __syncthreads();
  if (warp == 4) {
    tcgen05_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

bool halo_wgrad_eligible(const mig_conv_geom* g) {
  if (g->Cin != H_C || g->Cout > 32 || g->Cout < 8 || g->Cout % 8 != 0) return false;
  for (int i = 0; i < 3; ++i)
    if (g->stride[i] != 1 || g->ksize[i] > 3) return false;
  const int T = g->ksize[0] * g->ksize[1] * g->ksize[2];
  if ((T + 1) / 2 * 32 > 512) return false;
  const int64_t vox = (int64_t)g->N * g->out_dims[0] * g->out_dims[1] * g->out_dims[2];
  return vox >= 32768 && g->out_dims[2] >= HT_X && g->out_dims[1] >= HT_Y / 2;
}

int halo_conv_wgrad(const mig_conv_geom* g, const void* x, const void* dy, float* dw, void* stream) {
  HaloWgradParams p{};
  p.N = g->N; p.D = g->in_dims[0]; p.H = g->in_dims[1]; p.W = g->in_dims[2];
  p.OD = g->out_dims[0]; p.OH = g->out_dims[1]; p.OW = g->out_dims[2];
  for (int i = 0; i < 3; ++i) { p.ks[i] = g->ksize[i]; p.lo[i] = -g->pad[i]; }
  p.hz = p.ks[0]; p.hy = HT_Y + p.ks[1] - 1; p.hx = HT_X + p.ks[2] - 1;
  p.Cout = g->Cout;
  p.tiles_x = (p.OW + HT_X - 1) / HT_X;
  p.tiles_y = (p.OH + HT_Y - 1) / HT_Y;
  p.num_tiles = (int64_t)p.N * p.OD * p.tiles_y * p.tiles_x;
  p.taps_total = p.ks[0] * p.ks[1] * p.ks[2];
  p.taps_per_half = (p.taps_total + 1) / 2;
  p.dw = dw;
  CUtensorMap xm, dym;
  if (halo_map(&xm, x, p.N, p.D, p.H, p.W, H_C, p.hx, p.hy, p.hz)) return 1;
  if (halo_map(&dym, dy, p.N, p.OD, p.OH, p.OW, p.Cout, HT_X, HT_Y, 1)) return 1;
  const int nvox = p.hz * p.hy * p.hx;
  const int smem = (nvox * 64 + 128) + (128 * p.Cout * 2 + 128) + 2 * (nvox * 64 + 512 + 128) + 2 * 8 * (128 * 16 + 16) + 512;
  static SmemOptIn optin;
  if (int rc = ensure_dynamic_smem(wgrad_halo_kernel, smem, optin, "wgrad_halo")) return rc;
  int64_t pairs = device_info().sm_count / 2;
  if (pairs > p.num_tiles) pairs = p.num_tiles;
  if (pairs < 1) pairs = 1;
  wgrad_halo_kernel<<<(unsigned)(2 * pairs), H_THREADS, smem, as_stream(stream)>>>(xm, dym, p);
  return check_launch("wgrad_halo_kernel");
}

int halo_conv_fwd(const mig_conv_geom* g, const void* x, const void* w, const float* bias, const float* chan_bias,
                  const void* residual, void* y, void* stream) {
  return run_halo(g, 0, x, w, bias, chan_bias, residual, y, stream);
}

int halo_conv_dgrad(const mig_conv_geom* g, const void* dy, const void* w, void* dx, void* ws, int64_t ws_bytes,
                    void* stream) {
  const int T = g->ksize[0] * g->ksize[1] * g->ksize[2];
  const int64_t wt_bytes = (int64_t)g->Cin * T * g->Cout * 2;
  MIG_REQUIRE(ws && ws_bytes >= wt_bytes, "conv_dgrad(halo): workspace too small");
  if (filter_transpose(MIG_BF16, w, ws, g->Cout, T, g->Cin, stream)) return 2;
  return run_halo(g, 1, dy, ws, nullptr, nullptr, nullptr, dx, stream);
}

}  // namespace mig

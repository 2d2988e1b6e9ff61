// Fused flash-style attention BACKWARD on tcgen05 (training path of unet:396-416 / ae:283-323; replaces the
// baddbmm -> softmax -> bmm autograd chain and xformers' memory_efficient_attention backward). No L x L tensor exists:
// P is recomputed tile by tile from Q, K and the log-sum-exp the forward kernel saved.
//
//   S = scale * Q K^T,  P = exp(S - lse),  dP = dO V^T,  D = rowsum(dO * O),  dS = scale * P * (dP - D)
//   dV = P^T dO,   dK = dS^T Q,   dQ = dS K
//
// One kernel template, two launches:
//   MODE 0 (key-stationary)   a CTA owns 128 keys and a DV-column slice of dK and dV; it streams the query tiles:
//                             G1 = K Q_j^T, G2 = V dO_j^T (full head dim) -> P^T, dS^T (bf16, shared memory)
//                             -> dV[:, slice] += P^T dO_j[:, slice],  dK[:, slice] += dS^T Q_j[:, slice]
//   MODE 1 (query-stationary) a CTA owns 128 queries and a DV-column slice of dQ; it streams the key tiles:
//                             G1 = Q K_j^T, G2 = dO V_j^T -> dS -> dQ[:, slice] += dS K_j[:, slice]
// Tensor memory (512 columns): G1 [0,128), G2 [128,256), accumulators from 256 (MODE 0: 2 x DV <= 256; MODE 1: DV <= 256).
// The LDM default uses single heads of 512 / 768 channels: the accumulators of a whole head do not fit next to the two
// score tiles, so the output columns are sliced (DV = 128 resp. 256) and every slice recomputes G1 / G2 -- the same
// trade the forward kernel makes for O.
//
// Roles (192 threads): warps 0-3 turn (G1, G2) into the bf16 tiles (thread = stationary row = TMEM lane), warp 4
// issues the UMMAs and owns the TMEM allocation, warp 5 issues the TMA loads.
#include <cuda.h>

#include "common.cuh"
#include "tc_common.cuh"
#include "tc_host.cuh"

namespace mig {

using namespace tc;

constexpr int FB_BM = 128, FB_BN = 128;
constexpr int FB_QK_STAGE_BYTES = 2 * FB_BM * 128;   // stationary chunk + streaming chunk, 64 channels each
constexpr int FB_T_BYTES = 2 * FB_BM * 128;          // one 128 x 128 bf16 tile as two 64-column panels
constexpr int FB_PANEL = 64 * 128;
constexpr int FB_V_RING_BYTES = 64 * 1024;

__device__ __forceinline__ float fb_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

struct FlashBwdParams {
  int B, H, Lq, Lk, dh, DV;
  int qk_stages, v_stages;
  float scale, scale_log2;
  const float* lse;      // [B*H][Lq], log2 domain (from the forward kernel)
  const float* delta;    // [B*H][Lq], rowsum(dO * O)
  __nv_bfloat16* out1;   // MODE 0: dV          MODE 1: unused
  __nv_bfloat16* out2;   // MODE 0: dK          MODE 1: dQ
};

// bars: qk_full[3] qk_empty[3] v_full[4] v_empty[4] g_full g_empty t_full t_empty o_full
template <int MODE>
__global__ void __launch_bounds__(192, 1) flash_bwd_kernel(const __grid_constant__ CUtensorMap x1map,   // K  | Q   (128-row boxes)
                                                           const __grid_constant__ CUtensorMap y1map,   // Q  | K
                                                           const __grid_constant__ CUtensorMap x2map,   // V  | dO
                                                           const __grid_constant__ CUtensorMap y2map,   // dO | V
                                                           const __grid_constant__ CUtensorMap b1map,   // dO | -   (64-row boxes)
                                                           const __grid_constant__ CUtensorMap b2map,   // Q  | K
                                                           FlashBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t qk_smem = smem_base;
  const uint32_t t_smem = qk_smem + p.qk_stages * FB_QK_STAGE_BYTES;   // T1 then T2
  const uint32_t v_smem = t_smem + 2 * FB_T_BYTES;
  __shared__ __align__(8) uint64_t bars[19];
  __shared__ uint32_t tmem_slot;
  __shared__ __align__(16) float stat_s[2][2][FB_BN];   // MODE 0: (lse, D * scale) of the streamed query tile, by tile parity
  const uint32_t b0 = smem_u32(&bars[0]);
  const uint32_t qk_full = b0, qk_empty = b0 + 8 * 3, v_full = b0 + 8 * 6, v_empty = b0 + 8 * 10, g_full = b0 + 8 * 14,
                 g_empty = b0 + 8 * 15, t_full = b0 + 8 * 16, t_empty = b0 + 8 * 17, o_full = b0 + 8 * 18;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int x0 = blockIdx.x * FB_BM;        // first stationary row (key in MODE 0, query in MODE 1)
  const int slice = blockIdx.y;
  const int b = blockIdx.z / p.H, h = blockIdx.z - b * p.H;
  const int Lx = MODE == 0 ? p.Lk : p.Lq, Ly = MODE == 0 ? p.Lq : p.Lk;
  const int ntile = (Ly + FB_BN - 1) / FB_BN;
  const int nkc = p.dh / 64;
  const int v_stage_bytes = (p.DV / 64) * FB_PANEL;
  constexpr int NPROD = MODE == 0 ? 2 : 1;   // accumulated products per streamed tile

  if (threadIdx.x == 0) {
    for (int i = 0; i < 3; ++i) { mbar_init(qk_full + 8 * i, 1); mbar_init(qk_empty + 8 * i, 1); }
    for (int i = 0; i < 4; ++i) { mbar_init(v_full + 8 * i, 1); mbar_init(v_empty + 8 * i, 1); }
    mbar_init(g_full, 1);
    mbar_init(g_empty, 128);
    mbar_init(t_full, 128);
    mbar_init(t_empty, 1);
    mbar_init(o_full, 1);
    fence_barrier_init();
  }
  if (warp == 4) tmem_alloc<512>(smem_u32(&tmem_slot));
  if (warp == 5 && lane == 0) {
    tma_prefetch_desc(&x1map); tma_prefetch_desc(&y1map); tma_prefetch_desc(&x2map); tma_prefetch_desc(&y2map);
    tma_prefetch_desc(&b1map); tma_prefetch_desc(&b2map);
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_slot;
  const uint32_t tmem_acc = tmem_base + 256;

  if (warp < 4) {
    // ===================== (G1, G2) -> bf16 tiles; epilogue =====================
    const int r = warp * 32 + lane;
    const int xr = x0 + r;
    const bool xok = xr < Lx;
    const uint32_t lane_off = (uint32_t)(warp * 32) << 16;
    const float* lse_bh = p.lse + (int64_t)blockIdx.z * p.Lq;
    const float* del_bh = p.delta + (int64_t)blockIdx.z * p.Lq;
    float lse_r = INFINITY, del_r = 0.f;   // del_* hold delta * scale: dS = P * (dP * scale - delta * scale)
    if (MODE == 1 && xok) { lse_r = lse_bh[xr]; del_r = del_bh[xr] * p.scale; }
    for (int j = 0; j < ntile; ++j) {
      const int y0 = j * FB_BN;
      if (MODE == 0) {   // per-column statistics of this query tile (lse = +inf for queries past the end: P = 0)
        const int q = y0 + r;
        stat_s[j & 1][0][r] = q < p.Lq ? lse_bh[q] : INFINITY;
        stat_s[j & 1][1][r] = q < p.Lq ? del_bh[q] * p.scale : 0.f;
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
      mbar_wait(g_full, (uint32_t)j & 1u);
      tcgen05_fence_after();
      mbar_wait(t_empty, ((uint32_t)j & 1u) ^ 1u);   // the products of tile j-1 have consumed the bf16 tiles
#pragma unroll 1
      for (int half = 0; half < 2; ++half) {
        float g1[64], g2[64];
        tmem_ld64(tmem_base + lane_off + half * 64, g1);
        tmem_ld64(tmem_base + lane_off + 128 + half * 64, g2);
        const uint32_t t1 = t_smem + half * (FB_BM * 128), t2 = t1 + FB_T_BYTES;
        // Rows past the end of the stationary tile need no masking: their G rows are zero-filled by TMA and whatever
        // they produce only lands in accumulator rows the epilogue never stores. Columns past the end of the streamed
        // tile do: MODE 0 (queries) gets P = 0 from lse = +inf, MODE 1 (keys) is masked on the ragged last tile only.
        const bool ragged = MODE == 1 && y0 + half * 64 + 64 > p.Lk;
#pragma unroll
        for (int c = 0; c < 8; ++c) {   // 16-byte chunks of the 128-byte row
          uint32_t o1[4], o2[4];
          float lc[8], dc[8];
          if (MODE == 0) {   // per-column statistics: two 16-byte broadcast reads per 4 columns
            const float4* ls = reinterpret_cast<const float4*>(&stat_s[j & 1][0][half * 64 + c * 8]);
            const float4* ds = reinterpret_cast<const float4*>(&stat_s[j & 1][1][half * 64 + c * 8]);
            const float4 l0 = ls[0], l1 = ls[1], d0 = ds[0], d1 = ds[1];
            lc[0] = l0.x; lc[1] = l0.y; lc[2] = l0.z; lc[3] = l0.w; lc[4] = l1.x; lc[5] = l1.y; lc[6] = l1.z; lc[7] = l1.w;
            dc[0] = d0.x; dc[1] = d0.y; dc[2] = d0.z; dc[3] = d0.w; dc[4] = d1.x; dc[5] = d1.y; dc[6] = d1.z; dc[7] = d1.w;
          }
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float pv[2], dv[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              const int cc = 2 * e + u, col = c * 8 + cc;
              const float lse_c = MODE == 0 ? lc[cc] : lse_r, del_c = MODE == 0 ? dc[cc] : del_r;
              float pe = fb_ex2(fmaf(g1[col], p.scale_log2, -lse_c));
              if (ragged) pe = (y0 + half * 64 + col < p.Lk) ? pe : 0.f;
              pv[u] = pe;
              dv[u] = pe * fmaf(g2[col], p.scale, -del_c);
            }
            __nv_bfloat162 a = __floats2bfloat162_rn(pv[0], pv[1]), d = __floats2bfloat162_rn(dv[0], dv[1]);
            o1[e] = *reinterpret_cast<uint32_t*>(&a);
            o2[e] = *reinterpret_cast<uint32_t*>(&d);
          }
          if (MODE == 0)
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(t1 + sw128_offset(r, c)), "r"(o1[0]), "r"(o1[1]),
                         "r"(o1[2]), "r"(o1[3]) : "memory");
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(t2 + sw128_offset(r, c)), "r"(o2[0]), "r"(o2[1]),
                       "r"(o2[2]), "r"(o2[3]) : "memory");
        }
      }
      tcgen05_fence_before();
      mbar_arrive(g_empty);          // G1 / G2 are in registers no longer needed: the next tile may overwrite them
      fence_proxy_async();           // generic-proxy writes of the bf16 tiles -> visible to the UMMA (async proxy)
      mbar_arrive(t_full);
    }
    // ---- epilogue: accumulators -> bf16 rows of dV / dK (MODE 0) or dQ (MODE 1) ----
    mbar_wait(o_full, 0);
    tcgen05_fence_after();
    const int64_t rowoff = ((int64_t)b * Lx + xr) * ((int64_t)p.H * p.dh) + (int64_t)h * p.dh + slice * p.DV;
#pragma unroll 1
    for (int pr = 0; pr < NPROD; ++pr) {
      __nv_bfloat16* orow = ((MODE == 0 && pr == 0) ? p.out1 : p.out2) + rowoff;
      const uint32_t ta = tmem_acc + lane_off + pr * p.DV;
#pragma unroll 1
      for (int cw = 0; cw < p.DV; cw += 64) {
        float vw[64];
        tmem_ld64(ta + cw, vw);
        if (!xok) continue;
#pragma unroll
        for (int c0 = 0; c0 < 64; c0 += 8) {
          uint4 o;
          __nv_bfloat162* hh = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
          for (int e = 0; e < 4; ++e) hh[e] = __floats2bfloat162_rn(vw[c0 + 2 * e], vw[c0 + 2 * e + 1]);
          *reinterpret_cast<uint4*>(orow + cw + c0) = o;
        }
      }
    }
    tcgen05_fence_before();
  } else if (warp == 4) {
    // ===================== UMMA issuer =====================
    const uint32_t idesc_g = make_idesc(FB_BM, FB_BN, 0, 0);
    const uint32_t idesc_o = make_idesc(FB_BM, p.DV, 0, 1);
    int qs = 0, vs = 0;
    uint32_t qph = 0, vph = 0;
    auto issue_g = [&](int j) {
      mbar_wait(g_empty, ((uint32_t)j & 1u) ^ 1u);   // tile j-1 has been read out of G1 / G2
      tcgen05_fence_after();
      for (int gi = 0; gi < 2; ++gi)
        for (int c = 0; c < nkc; ++c) {
          mbar_wait(qk_full + 8 * qs, qph);
          tcgen05_fence_after();
          if (elect_one()) {
            const uint32_t a = qk_smem + qs * FB_QK_STAGE_BYTES, bsm = a + FB_BM * 128;
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
              umma_bf16(tmem_base + gi * 128, make_smem_desc(a + kk * 32, 16, 1024), make_smem_desc(bsm + kk * 32, 16, 1024),
                        idesc_g, (c | kk) ? 1u : 0u);
            umma_commit(qk_empty + 8 * qs);
            if (gi == 1 && c == nkc - 1) umma_commit(g_full);
          }
          __syncwarp();
          if (++qs == p.qk_stages) { qs = 0; qph ^= 1u; }
        }
    };
    issue_g(0);
    for (int j = 0; j < ntile; ++j) {
      if (j + 1 < ntile) issue_g(j + 1);
      mbar_wait(t_full, (uint32_t)j & 1u);
      tcgen05_fence_after();
      for (int half = 0; half < 2; ++half)
        for (int pr = 0; pr < NPROD; ++pr) {
          mbar_wait(v_full + 8 * vs, vph);
          tcgen05_fence_after();
          if (elect_one()) {
            // MODE 0: product 0 uses T1 (P^T) with dO, product 1 uses T2 (dS^T) with Q; MODE 1: T2 (dS) with K
            const uint32_t a = t_smem + ((MODE == 0 && pr == 0) ? 0 : FB_T_BYTES) + half * (FB_BM * 128);
            const uint32_t bsm = v_smem + vs * v_stage_bytes;
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
              umma_bf16(tmem_acc + pr * p.DV, make_smem_desc(a + kk * 32, 16, 1024),
                        make_smem_desc(bsm + kk * 2048, FB_PANEL, 1024), idesc_o, (j | half | kk) ? 1u : 0u);
            umma_commit(v_empty + 8 * vs);
            if (half == 1 && pr == NPROD - 1) {
              umma_commit(t_empty);
              if (j == ntile - 1) umma_commit(o_full);
            }
          }
          __syncwarp();
          if (++vs == p.v_stages) { vs = 0; vph ^= 1u; }
        }
    }
  } else if (elect_one()) {
    // ===================== TMA issuer =====================
    int qs = 0, vs = 0;
    uint32_t qph = 0, vph = 0;
    auto load_g = [&](int j) {
      for (int gi = 0; gi < 2; ++gi)
        for (int c = 0; c < nkc; ++c) {
          mbar_wait(qk_empty + 8 * qs, qph ^ 1u);
          const uint32_t a = qk_smem + qs * FB_QK_STAGE_BYTES, bar = qk_full + 8 * qs;
          mbar_arrive_expect_tx(bar, FB_QK_STAGE_BYTES);
          tma_load_4d(a, gi == 0 ? &x1map : &x2map, bar, c * 64, h, x0, b);
          tma_load_4d(a + FB_BM * 128, gi == 0 ? &y1map : &y2map, bar, c * 64, h, j * FB_BN, b);
          if (++qs == p.qk_stages) { qs = 0; qph ^= 1u; }
        }
    };
    auto load_v = [&](int j) {
      for (int half = 0; half < 2; ++half)
        for (int pr = 0; pr < NPROD; ++pr) {
          mbar_wait(v_empty + 8 * vs, vph ^ 1u);
          const uint32_t dst = v_smem + vs * v_stage_bytes, bar = v_full + 8 * vs;
          mbar_arrive_expect_tx(bar, v_stage_bytes);
          const CUtensorMap* m = (MODE == 0 && pr == 0) ? &b1map : &b2map;
          for (int pn = 0; pn < p.DV / 64; ++pn)
            tma_load_4d(dst + pn * FB_PANEL, m, bar, slice * p.DV + pn * 64, h, j * FB_BN + half * 64, b);
          if (++vs == p.v_stages) { vs = 0; vph ^= 1u; }
        }
    };
    load_g(0);
    for (int j = 0; j < ntile; ++j) {
      if (j + 1 < ntile) load_g(j + 1);
      load_v(j);
    }
  }
  __syncthreads();
  if (warp == 4) {
    tcgen05_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// delta[bh][q] = sum_c dO[b,q,h*dh+c] * O[b,q,h*dh+c]: one warp per (b, q, h)
__global__ void __launch_bounds__(256) attn_delta_kernel(const __nv_bfloat16* __restrict__ o,
                                                         const __nv_bfloat16* __restrict__ d_o, float* __restrict__ delta,
                                                         int B, int H, int L, int dh) {
  const int lane = threadIdx.x & 31;
  const int64_t w = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (w >= (int64_t)B * L * H) return;
  const int h = (int)(w % H);
  const int64_t bq = w / H;
  const int64_t b = bq / L, q = bq - b * L;
  const __nv_bfloat16* po = o + bq * ((int64_t)H * dh) + (int64_t)h * dh;
  const __nv_bfloat16* pd = d_o + bq * ((int64_t)H * dh) + (int64_t)h * dh;
  float acc = 0.f;
  for (int c = lane * 8; c < dh; c += 256) {   // dh is a multiple of 64
    const uint4 a = *reinterpret_cast<const uint4*>(po + c), d = *reinterpret_cast<const uint4*>(pd + c);
    const __nv_bfloat162* a2 = reinterpret_cast<const __nv_bfloat162*>(&a);
    const __nv_bfloat162* d2 = reinterpret_cast<const __nv_bfloat162*>(&d);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 x = __bfloat1622float2(a2[e]), y = __bfloat1622float2(d2[e]);
      acc = fmaf(x.x, y.x, fmaf(x.y, y.y, acc));
    }
  }
  acc = warp_sum(acc);
  if (lane == 0) delta[(b * H + h) * L + q] = acc;
}

template <int MODE>
static int launch_flash_bwd(const CUtensorMap& x1, const CUtensorMap& y1, const CUtensorMap& x2, const CUtensorMap& y2,
                            const CUtensorMap& b1, const CUtensorMap& b2, FlashBwdParams p, dim3 grid, cudaStream_t st) {
  const int v_stage = (p.DV / 64) * FB_PANEL;
  p.v_stages = FB_V_RING_BYTES / v_stage > 4 ? 4 : FB_V_RING_BYTES / v_stage;
  auto bytes = [&](int qk_stages) { return qk_stages * FB_QK_STAGE_BYTES + 2 * FB_T_BYTES + p.v_stages * v_stage + 1024; };
  p.qk_stages = bytes(3) <= 227 * 1024 - 4096 ? 3 : 2;
  const int smem = bytes(p.qk_stages);
  static SmemOptIn optin;
  if (int rc = ensure_dynamic_smem(flash_bwd_kernel<MODE>, smem, optin, "flash_attention_bwd")) return rc;
  flash_bwd_kernel<MODE><<<grid, 192, smem, st>>>(x1, y1, x2, y2, b1, b2, p);
  return check_launch("flash_bwd_kernel");
}

static int slice_width(int dh, int cap) {
  for (int w = cap; w >= 64; w >>= 1)
    if (dh % w == 0) return w;
  return 0;
}

}  // namespace mig

using namespace mig;

extern "C" int mig_flash_attention_bwd(const void* q, const void* k, const void* v, const void* o, const void* d_o,
                                       const float* lse, float* delta, void* dq, void* dk, void* dv, int32_t B, int32_t H,
                                       int32_t Lq, int32_t Lk, int32_t dh, float scale, void* stream) {
  MIG_REQUIRE(q && k && v && o && d_o && lse && delta && dq && dk && dv, "flash_attention_bwd: null argument");
  MIG_REQUIRE(mig_has_tcgen05(), "flash_attention_bwd: needs an sm_100 device");
  MIG_REQUIRE(dh % 64 == 0 && dh >= 64, "flash_attention_bwd: head dim %d must be a multiple of 64", dh);
  MIG_REQUIRE(B > 0 && Lq > 0 && Lk > 0 && (int64_t)B * H < 65536, "flash_attention_bwd: bad sizes");
  const uintptr_t al = reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v) |
                       reinterpret_cast<uintptr_t>(o) | reinterpret_cast<uintptr_t>(d_o) | reinterpret_cast<uintptr_t>(dq) |
                       reinterpret_cast<uintptr_t>(dk) | reinterpret_cast<uintptr_t>(dv);
  MIG_REQUIRE((al & 15) == 0, "flash_attention_bwd: tensors must be 16-byte aligned");
  cudaStream_t st = as_stream(stream);
  {
    const int64_t warps = (int64_t)B * Lq * H;
    attn_delta_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, st>>>((const __nv_bfloat16*)o, (const __nv_bfloat16*)d_o, delta,
                                                                   B, H, Lq, dh);
    if (int rc = check_launch("attn_delta_kernel")) return rc;
  }
  CUtensorMap q128, k128, v128, do128, q64, k64, do64;
  const int64_t ld = (int64_t)H * dh;
  if (bhld_map(&q128, q, B, H, Lq, dh, 128, ld) || bhld_map(&k128, k, B, H, Lk, dh, 128, ld) ||
      bhld_map(&v128, v, B, H, Lk, dh, 128, ld) || bhld_map(&do128, d_o, B, H, Lq, dh, 128, ld) ||
      bhld_map(&q64, q, B, H, Lq, dh, 64, ld) || bhld_map(&k64, k, B, H, Lk, dh, 64, ld) ||
      bhld_map(&do64, d_o, B, H, Lq, dh, 64, ld))
    return 1;
  FlashBwdParams p{};
  p.B = B; p.H = H; p.Lq = Lq; p.Lk = Lk; p.dh = dh;
  p.scale = scale;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.lse = lse;
  p.delta = delta;
  // MODE 0: dK, dV per 128-key tile
  p.DV = slice_width(dh, 128);
  p.out1 = (__nv_bfloat16*)dv;
  p.out2 = (__nv_bfloat16*)dk;
  if (int rc = launch_flash_bwd<0>(k128, q128, v128, do128, do64, q64, p,
                                   dim3((Lk + FB_BM - 1) / FB_BM, dh / p.DV, B * H), st))
    return rc;
  // MODE 1: dQ per 128-query tile
  p.DV = slice_width(dh, 256);
  p.out1 = nullptr;
  p.out2 = (__nv_bfloat16*)dq;
  return launch_flash_bwd<1>(q128, k128, do128, v128, k64, k64, p, dim3((Lq + FB_BM - 1) / FB_BM, dh / p.DV, B * H), st);
}

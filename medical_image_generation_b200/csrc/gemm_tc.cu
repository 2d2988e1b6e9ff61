// tcgen05 / TMEM / TMA engine (sm_100a): bf16 operands, fp32 accumulation in tensor memory.
//
//  conv_tc_kernel   conv fwd + dgrad as implicit GEMM.  D[128 voxels][BN channels] per CTA.
//                   A (activations, K-major): im2col rows gathered on the fly from the NDHWC tensor by
//                   four producer warps with 16-byte cp.async (zero-fill = halo / stride holes / K tail),
//                   written straight into the 128B-swizzled UMMA layout.
//                   B (filters [Cout][tap][Cin], K-major): one TMA box per stage.
//                   Epilogue: TMEM -> registers -> (+bias, +time-embedding, +residual) -> bf16 NDHWC,
//                   or fp32 atomics into a workspace for split-K on the small deep levels.
//  wgrad_tc_kernel  dW[Cout][tap*Cin] += dY^T * im2col(X); both operands MN-major: dY tiles by TMA,
//                   im2col(X) tiles gathered with cp.async; voxel (K) dimension split across CTAs,
//                   fp32 reduction into dW with red.global.add.
//  gemm_tc_kernel   strided batched GEMM with both operands by TMA, either major (attention products).
//
// Warp roles (192 threads): warps 0-3 producers, then epilogue (TMEM lane quadrant = warp id);
// warp 4 = TMEM allocator + single-thread MMA issuer; warp 5 = TMA issuer.
#include <cuda.h>

#include <mutex>

#include "common.cuh"
#include "tc_common.cuh"
#include "tc_host.cuh"

namespace mig {

using namespace tc;

int filter_transpose(int dtype, const void* w, void* wt, int Cout, int Tn, int Cin, void* stream);
bool tc_wgrad_eligible(const mig_conv_geom* g);  // gemm_tc2.cu

constexpr int TBM = 128;        // UMMA M
constexpr int TBK = 64;         // K per stage (one 128-byte swizzle row of bf16)
constexpr int kProducerThreads = 128;
constexpr int kThreads = 192;
constexpr int kLag = 2;         // cp.async groups kept in flight per producer thread

__host__ __device__ constexpr int stages_for(int bn) {
  // stage = A 16 KB + B bn*128 B ; keep <= ~200 KB
  return bn >= 256 ? 4 : (bn >= 128 ? 6 : 8);
}
__host__ __device__ constexpr int tmem_cols_for(int bn) { return bn <= 32 ? 32 : (bn <= 64 ? 64 : (bn <= 128 ? 128 : 256)); }

struct ConvTcParams {
  Gather g;
  const __nv_bfloat16* src;
  const float* bias;
  const float* chan_bias;
  const __nv_bfloat16* residual;
  __nv_bfloat16* out;
  float* partial;     // split-K fp32 workspace [M][Cdst] (zeroed), or nullptr
  int num_kb;         // total K blocks
  int kb_per_split;
};

// ---------------------------------------------------------------------------------------------------
// conv fwd / dgrad
// ---------------------------------------------------------------------------------------------------
template <int BN>
__global__ void __launch_bounds__(kThreads, 1) conv_tc_kernel(const __grid_constant__ CUtensorMap wmap, ConvTcParams p) {
  constexpr int STAGES = stages_for(BN);
  constexpr int A_BYTES = TBM * 128, B_BYTES = BN * 128, STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr int TCOLS = tmem_cols_for(BN);
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  __shared__ __align__(8) uint64_t bars[2 * STAGES + 1];
  __shared__ uint32_t tmem_slot;
  const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[STAGES]), accbar = smem_u32(&bars[2 * STAGES]);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const Gather& g = p.g;
  const int64_t m0 = (int64_t)blockIdx.x * TBM;
  const int n0 = blockIdx.y * BN;
  const int kb_begin = blockIdx.z * p.kb_per_split;
  const int kb_end = min(p.num_kb, kb_begin + p.kb_per_split);
  const int nkb = kb_end - kb_begin;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full0 + 8 * s, kProducerThreads + 1);  // 128 gather threads + the TMA thread's expect_tx arrive
      mbar_init(empty0 + 8 * s, 1);                    // one tcgen05.commit
    }
    mbar_init(accbar, 1);
    fence_barrier_init();
  }
  if (warp == 4) tmem_alloc<TCOLS>(smem_u32(&tmem_slot));
  if (warp == 5 && lane == 0) tma_prefetch_desc(&wmap);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_acc = tmem_slot;

  if (warp < 4) {
    // ===================== producers: im2col gather of the A tile ======================
    const int t = threadIdx.x;
    const int j = t & 7;        // 16-byte chunk within the 128-byte K row
    const int rb = t >> 3;      // rows rb + 16*i
    int pz[8], py[8], px[8], pn[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int64_t m = m0 + rb + 16 * i;
      if (m < g.M) {
        int64_t r = m;
        int o2 = (int)(r % g.dst[2]); r /= g.dst[2];
        int o1 = (int)(r % g.dst[1]); r /= g.dst[1];
        int o0 = (int)(r % g.dst[0]);
        pn[i] = (int)(r / g.dst[0]);
        pz[i] = o0 * g.a[0] + g.c[0];
        py[i] = o1 * g.a[1] + g.c[1];
        px[i] = o2 * g.a[2] + g.c[2];
      } else {
        pn[i] = -1; pz[i] = py[i] = px[i] = 0;
      }
    }
    const bool unit = (g.d[0] == 1 && g.d[1] == 1 && g.d[2] == 1);
    for (int it = 0; it < nkb; ++it) {
      const int s = it % STAGES;
      const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
      mbar_wait(empty0 + 8 * s, ph ^ 1u);
      const uint32_t a_smem = smem_base + s * STAGE_BYTES;
      const int k = (kb_begin + it) * TBK + j * 8;
      const bool kok = k < g.K;
      int tap = kok ? k / g.Csrc : 0;
      const int ci = kok ? k - tap * g.Csrc : 0;
      const int t2 = tap % g.ks[2]; tap /= g.ks[2];
      const int t1 = tap % g.ks[1];
      const int t0 = tap / g.ks[1];
      const int dz = t0 * g.b[0], dy = t1 * g.b[1], dx = t2 * g.b[2];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = rb + 16 * i;
        int z = pz[i] + dz, y = py[i] + dy, x = px[i] + dx;
        bool ok = kok && pn[i] >= 0 && z >= 0 && y >= 0 && x >= 0;
        if (!unit) {
          int qz = z / g.d[0], qy = y / g.d[1], qx = x / g.d[2];
          ok = ok && (!g.exact || (qz * g.d[0] == z && qy * g.d[1] == y && qx * g.d[2] == x));
          z = qz; y = qy; x = qx;
        }
        ok = ok && z < g.src[0] && y < g.src[1] && x < g.src[2];
        const int64_t off = ok ? ((((int64_t)pn[i] * g.src[0] + z) * g.src[1] + y) * g.src[2] + x) * g.Csrc + ci : 0;
        cp_async16(a_smem + sw128_offset(r, j), p.src + off, ok ? 16u : 0u);
      }
      cp_async_commit();
      if (it >= kLag) {
        cp_async_wait<kLag>();
        fence_proxy_async();
        mbar_arrive(full0 + 8 * ((it - kLag) % STAGES));
      }
    }
    cp_async_wait<0>();
    fence_proxy_async();
    for (int it = max(0, nkb - kLag); it < nkb; ++it) mbar_arrive(full0 + 8 * (it % STAGES));

    // ===================== epilogue: TMEM -> registers -> global ======================
    mbar_wait(accbar, 0);
    tcgen05_fence_after();
    const int row = warp * 32 + lane;
    const int64_t m = m0 + row;
    const bool mok = m < g.M;
    const int nimg = mok ? (int)(m / g.Mo) : 0;
    const uint32_t trow = tmem_acc + ((uint32_t)(warp * 32) << 16);
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 16) {
      if (n0 + c0 >= g.Cdst) break;   // warp-uniform
      float v[16];
      tmem_ld16(trow + c0, v);
      if (!mok) continue;
      const int col0 = n0 + c0;
      if (p.partial) {
        red_add_16(p.partial + m * g.Cdst + col0, v, g.Cdst - col0);
        continue;
      }
      const bool full16 = (col0 + 16 <= g.Cdst) && ((g.Cdst & 7) == 0);
      if (p.bias) {
#pragma unroll
        for (int e = 0; e < 16; ++e) if (col0 + e < g.Cdst) v[e] += p.bias[col0 + e];
      }
      if (p.chan_bias) {
        const float* cb = p.chan_bias + (int64_t)nimg * g.Cdst + col0;
#pragma unroll
        for (int e = 0; e < 16; ++e) if (col0 + e < g.Cdst) v[e] += cb[e];
      }
      __nv_bfloat16* dst = p.out + m * g.Cdst + col0;
      if (full16) {
        if (p.residual) {
          const uint4* rp = reinterpret_cast<const uint4*>(p.residual + m * g.Cdst + col0);
          uint4 r0 = rp[0], r1 = rp[1];
          const __nv_bfloat16* rh0 = reinterpret_cast<const __nv_bfloat16*>(&r0);
          const __nv_bfloat16* rh1 = reinterpret_cast<const __nv_bfloat16*>(&r1);
#pragma unroll
          for (int e = 0; e < 8; ++e) { v[e] += __bfloat162float(rh0[e]); v[8 + e] += __bfloat162float(rh1[e]); }
        }
        uint4 o0, o1;
        __nv_bfloat162* h0 = reinterpret_cast<__nv_bfloat162*>(&o0);
        __nv_bfloat162* h1 = reinterpret_cast<__nv_bfloat162*>(&o1);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          h0[e] = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
          h1[e] = __floats2bfloat162_rn(v[8 + 2 * e], v[8 + 2 * e + 1]);
        }
        reinterpret_cast<uint4*>(dst)[0] = o0;
        reinterpret_cast<uint4*>(dst)[1] = o1;
      } else {
#pragma unroll
        for (int e = 0; e < 16; ++e)
          if (col0 + e < g.Cdst) {
            float r = p.residual ? __bfloat162float(p.residual[m * g.Cdst + col0 + e]) : 0.f;
            dst[e] = __float2bfloat16_rn(v[e] + r);
          }
      }
    }
    tcgen05_fence_before();
  } else if (warp == 4) {
    // ===================== MMA issuer ======================
    constexpr uint32_t idesc = make_idesc(TBM, BN, 0, 0);
    for (int it = 0; it < nkb; ++it) {
      const int s = it % STAGES;
      const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
      mbar_wait(full0 + 8 * s, ph);
      tcgen05_fence_after();
      if (elect_one()) {
        const uint32_t a_smem = smem_base + s * STAGE_BYTES, b_smem = a_smem + A_BYTES;
#pragma unroll
        for (int kk = 0; kk < TBK / 16; ++kk) {
          const uint64_t ad = make_smem_desc(a_smem + kk * 32, 16, 1024);
          const uint64_t bd = make_smem_desc(b_smem + kk * 32, 16, 1024);
          umma_bf16(tmem_acc, ad, bd, idesc, (it | kk) ? 1u : 0u);
        }
        umma_commit(empty0 + 8 * s);          // frees the smem stage when these MMAs retire
        if (it == nkb - 1) umma_commit(accbar);  // accumulator complete
      }
      __syncwarp();
    }
    if (nkb == 0 && lane == 0) mbar_arrive(accbar);
  } else {
    // ===================== TMA issuer (filters) ======================
    if (elect_one()) {
      for (int it = 0; it < nkb; ++it) {
        const int s = it % STAGES;
        const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
        mbar_wait(empty0 + 8 * s, ph ^ 1u);
        const uint32_t b_smem = smem_base + s * STAGE_BYTES + A_BYTES;
        mbar_arrive_expect_tx(full0 + 8 * s, B_BYTES);
        tma_load_2d(b_smem, &wmap, full0 + 8 * s, (kb_begin + it) * TBK, n0);
      }
    }
  }
  __syncthreads();
  if (warp == 4) {
    tcgen05_fence_after();
    tmem_dealloc<TCOLS>(tmem_acc);
  }
}

// split-K finish: out = bf16(partial + bias + chan_bias + residual)
__global__ void __launch_bounds__(256) splitk_finish_kernel(const float* __restrict__ partial,
                                                            const float* __restrict__ bias,
                                                            const float* __restrict__ chan_bias,
                                                            const __nv_bfloat16* __restrict__ residual,
                                                            __nv_bfloat16* __restrict__ out, int64_t M, int C,
                                                            int64_t Mo) {
  const int64_t total = M * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = i / C;
    const int c = (int)(i - m * C);
    float v = partial[i];
    if (bias) v += bias[c];
    if (chan_bias) v += chan_bias[(m / Mo) * C + c];
    if (residual) v += __bfloat162float(residual[i]);
    out[i] = __float2bfloat16_rn(v);
  }
}

// ---------------------------------------------------------------------------------------------------
// host: tensor maps
// ---------------------------------------------------------------------------------------------------
template <int BN>
static int launch_conv_tc(const CUtensorMap& wmap, const ConvTcParams& p, dim3 grid, cudaStream_t st) {
  constexpr int smem = stages_for(BN) * (TBM * 128 + BN * 128) + 1024;
  static SmemOptIn optin;
  if (int rc = ensure_dynamic_smem(conv_tc_kernel<BN>, smem, optin, "conv_tc")) return rc;
  conv_tc_kernel<BN><<<grid, kThreads, smem, st>>>(wmap, p);
  return check_launch("conv_tc_kernel");
}

// Csrc % 8 (16-byte gather chunks inside one tap) and 16-byte aligned rows are the hard requirements.
static bool gather_ok(const Gather& q) { return q.Csrc % 8 == 0 && q.K % 8 == 0 && q.M > 0; }

bool tc_conv_eligible(const mig_conv_geom* g, int dtype, int which) {
  if (dtype != MIG_BF16) return false;
  if (which == 0) return g->Cin % 8 == 0;
  if (which == 1) return g->Cout % 8 == 0;
  return tc_wgrad_eligible(g);
}

static int split_plan(const Gather& q, int bn, int* splits, int* kb_per) {
  const int num_kb = (q.K + TBK - 1) / TBK;
  const int64_t tiles = ((q.M + TBM - 1) / TBM) * ((q.Cdst + bn - 1) / bn);
  const int sms = device_info().sm_count;
  int s = 1;
  if (tiles * 2 <= sms) {  // less than half a wave: split K until the chip is covered
    s = (int)(sms / tiles);
    if (s > num_kb / 8) s = num_kb / 8;  // keep >= 8 K blocks per CTA
    if (s < 1) s = 1;
  }
  int per = (num_kb + s - 1) / s;
  s = (num_kb + per - 1) / per;
  *splits = s;
  *kb_per = per;
  return num_kb;
}

int64_t tc_conv_workspace(const mig_conv_geom* g, int which) {
  // dgrad: transposed filter copy; fwd/dgrad split-K: fp32 [M][Cdst]
  int T = g->ksize[0] * g->ksize[1] * g->ksize[2];
  int64_t wt = which == 1 ? (int64_t)g->Cin * T * g->Cout * 2 : 0;
  wt = (wt + 255) / 256 * 256;
  Gather q = which == 1 ? make_gather_dgrad(g) : make_gather_fwd(g);
  int64_t part = which <= 1 ? q.M * q.Cdst * 4 : 0;
  return wt + part;
}

static int run_conv_tc(const Gather& q, const void* src, const void* wk, const float* bias, const float* chan_bias,
                       const void* residual, void* out, void* ws, int64_t ws_bytes, void* stream) {
  MIG_REQUIRE(gather_ok(q), "conv_tc: shape not eligible (Csrc=%d)", q.Csrc);
  MIG_REQUIRE((reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(wk) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(out) & 15) == 0,
              "conv_tc: tensors must be 16-byte aligned");
  cudaStream_t st = as_stream(stream);
  const int bn = pick_bn(q.Cdst);
  CUtensorMap wmap;
  uint64_t dims[2] = {(uint64_t)q.K, (uint64_t)q.Cdst};
  uint64_t strides[1] = {(uint64_t)q.K * 2};
  uint32_t box[2] = {TBK, (uint32_t)bn};
  if (make_map(&wmap, wk, 2, dims, strides, box)) return 1;
  ConvTcParams p{};
  p.g = q;
  p.src = (const __nv_bfloat16*)src;
  p.bias = bias; p.chan_bias = chan_bias;
  p.residual = (const __nv_bfloat16*)residual;
  p.out = (__nv_bfloat16*)out;
  int splits, per;
  p.num_kb = split_plan(q, bn, &splits, &per);
  p.kb_per_split = per;
  if (splits > 1 && (ws == nullptr || ws_bytes < q.M * q.Cdst * 4)) { splits = 1; p.kb_per_split = p.num_kb; }
  if (splits > 1) {
    p.partial = (float*)ws;
    cudaMemsetAsync(ws, 0, (size_t)(q.M * q.Cdst * 4), st);
  }
  MIG_REQUIRE((q.M + TBM - 1) / TBM < (1ll << 31), "conv_tc: too many voxels");
  dim3 grid((unsigned)((q.M + TBM - 1) / TBM), (unsigned)((q.Cdst + bn - 1) / bn), (unsigned)splits);
  int rc;
  switch (bn) {
    case 256: rc = launch_conv_tc<256>(wmap, p, grid, st); break;
    case 128: rc = launch_conv_tc<128>(wmap, p, grid, st); break;
    case 64: rc = launch_conv_tc<64>(wmap, p, grid, st); break;
    default: rc = launch_conv_tc<32>(wmap, p, grid, st); break;
  }
  if (rc) return rc;
  if (splits > 1) {
    splitk_finish_kernel<<<bw_grid(q.M * q.Cdst, 256), 256, 0, st>>>((const float*)ws, bias, chan_bias,
                                                                    (const __nv_bfloat16*)residual,
                                                                    (__nv_bfloat16*)out, q.M, q.Cdst, q.Mo);
    return check_launch("splitk_finish");
  }
  return 0;
}

int tc_conv_fwd(const mig_conv_geom* g, const void* x, const void* w, const float* bias, const float* chan_bias,
                const void* residual, void* y, void* ws, int64_t ws_bytes, void* stream) {
  Gather q = make_gather_fwd(g);
  return run_conv_tc(q, x, w, bias, chan_bias, residual, y, ws, ws_bytes, stream);
}

int tc_conv_dgrad(const mig_conv_geom* g, const void* dy, const void* w, void* dx, void* ws, int64_t ws_bytes,
                  void* stream) {
  Gather q = make_gather_dgrad(g);
  const int T = g->ksize[0] * g->ksize[1] * g->ksize[2];
  int64_t wt_bytes = ((int64_t)g->Cin * T * g->Cout * 2 + 255) / 256 * 256;
  MIG_REQUIRE(ws && ws_bytes >= wt_bytes, "conv_dgrad(tc): workspace too small");
  if (filter_transpose(MIG_BF16, w, ws, g->Cout, T, g->Cin, stream)) return 2;
  return run_conv_tc(q, dy, ws, nullptr, nullptr, nullptr, dx, (uint8_t*)ws + wt_bytes, ws_bytes - wt_bytes, stream);
}

}  // namespace mig

// Fused flash-style attention forward on tcgen05 (replaces xformers.ops.memory_efficient_attention, unet:128-135,403;
// and the baddbmm -> softmax -> bmm chain unet:406-416 when no gradient is required).
//
//   O[b, q, h*dh + :] = softmax_k(scale * Q K^T) V        per (batch b, head h); heads live inside the channel dim.
//
// The L x L score matrix never goes to HBM.
// Head dim <= 256 (pixel-space U-Nets, 128-channel heads at 32768 tokens): ONE pass with an online softmax -- running
// row maximum / sum in registers, O accumulated in tensor memory and rescaled lazily (only when a key tile raises the
// maximum by more than 2^8), normalised by 1/sum in the epilogue.
// Head dim > 256: two passes, both with S = Q K^T accumulated in tensor memory:
//   pass 0 (stats)  : per row running max / sum over all key tiles  ->  lse[row] = max + log2(sum)  (log2 domain)
//   pass 1 (output) : P = exp2(S * scale*log2e - lse) is ALREADY normalised, so O += P V needs no rescaling of the
//                     accumulator (no TMEM read-modify-write, no correction warps); S is double-buffered in TMEM so
//                     the softmax of key tile j overlaps the Q K^T of tile j+1.
// Head dims above 256 (the LDM default uses single heads of 512 / 768 channels) do not fit TMEM next to S: the
// value/output dim is cut into 256-column slices, one CTA per slice (each recomputes S).
//
// Roles (192 threads): warps 0-3 softmax + epilogue (thread = query row = TMEM lane), warp 4 UMMA issuer + TMEM
// allocator, warp 5 TMA issuer. Shared memory: 3-stage ring for (Q chunk, K chunk) pairs, one P tile (bf16,
// K-major, 128B swizzle = the A operand of P V), 2-stage ring for V half-tiles (MN-major B operand).
#include <cuda.h>

#include <algorithm>

#include "common.cuh"
#include "tc_common.cuh"
#include "tc_host.cuh"

namespace mig {

using namespace tc;

constexpr int FA_MAX_THREADS = 320;
// softmax warps: 4 (thread = query row) in the two-pass kernels; 8 in the online kernel, where warps w and w+4 share
// the rows of TMEM lane quadrant w and each takes 64 of the 128 keys of a tile -- the softmax, not the tensor pipe, is
// the critical path at head dim 128 (128 exp2 + packing per row and tile against 1024 cycles of UMMA)
__host__ __device__ constexpr int fa_softmax_warps(int pass) { return pass == 2 ? 8 : 4; }
constexpr int FA_BM = 128, FA_BN = 128;         // query rows / keys per tile
constexpr int FA_QK_STAGES = 3, FA_V_STAGES = 2;
constexpr int FA_QK_STAGE_BYTES = 2 * FA_BM * 128;   // Q chunk + K chunk, 64 channels each
constexpr int FA_P_BYTES = 2 * FA_BM * 128;          // 128 x 128 bf16 as two 64-key panels
constexpr int FA_PANEL = 64 * 128;

__device__ __forceinline__ float fast_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

struct FlashParams {
  int B, H, Lq, Lk, dh, DV;   // DV = value/output columns handled by one CTA (<= 256)
  int qk_stages;              // (Q chunk, K chunk) ring depth: 3, or 2 when 256-wide V stages leave no room
  float scale_log2;           // softmax scale * log2(e)
  float* lse;                 // [B*H][Lq], log2 domain
  __nv_bfloat16* out;         // (B, Lq, H*dh)
};

// bars: qk_full[3] qk_empty[3] v_full[2] v_empty[2] s_full[2] s_empty[2] p_full[2] p_empty[2] o_full
// The P tile is DOUBLE-buffered: the softmax of key tile j+1 writes P[(j+1)&1] while P V of tile j still reads P[j&1];
// with a single buffer the exp2 work and the P V MMAs of consecutive tiles were serialised (3150 cycles per tile for
// 1024 cycles of UMMA).
template <int PASS>
__global__ void __launch_bounds__(FA_MAX_THREADS, 1) flash_fwd_kernel(const __grid_constant__ CUtensorMap qmap,
                                                                  const __grid_constant__ CUtensorMap kmap,
                                                                  const __grid_constant__ CUtensorMap vmap,
                                                                  FlashParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t qk_smem = smem_base;
  const uint32_t p_smem = qk_smem + p.qk_stages * FA_QK_STAGE_BYTES;
  const uint32_t v_smem = p_smem + 2 * FA_P_BYTES;
  constexpr int SW = fa_softmax_warps(PASS);
  __shared__ __align__(8) uint64_t bars[19];
  __shared__ uint32_t tmem_slot;
  __shared__ float xch[2][2][FA_BM];   // online kernel: row max / row sum exchange between the two key halves
  const uint32_t b0 = smem_u32(&bars[0]);
  const uint32_t qk_full = b0, qk_empty = b0 + 8 * 3, v_full = b0 + 8 * 6, v_empty = b0 + 8 * 8, s_full = b0 + 8 * 10,
                 s_empty = b0 + 8 * 12, p_full = b0 + 8 * 14, p_empty = b0 + 8 * 16, o_full = b0 + 8 * 18;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * FA_BM;
  const int slice = blockIdx.y;
  const int b = blockIdx.z / p.H, h = blockIdx.z - b * p.H;
  const int nkv = (p.Lk + FA_BN - 1) / FA_BN;
  const int nkc = p.dh / 64;
  const int v_stage_bytes = (p.DV / 64) * FA_PANEL;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 3; ++i) { mbar_init(qk_full + 8 * i, 1); mbar_init(qk_empty + 8 * i, 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(v_full + 8 * i, 1); mbar_init(v_empty + 8 * i, 1);
      mbar_init(s_full + 8 * i, 1); mbar_init(s_empty + 8 * i, SW * 32);
    }
    for (int i = 0; i < 2; ++i) { mbar_init(p_full + 8 * i, SW * 32); mbar_init(p_empty + 8 * i, 1); }
    mbar_init(o_full, 1);
    fence_barrier_init();
  }
  if (warp == SW) tmem_alloc<512>(smem_u32(&tmem_slot));
  if (warp == SW + 1 && lane == 0) { tma_prefetch_desc(&qmap); tma_prefetch_desc(&kmap); tma_prefetch_desc(&vmap); }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_slot;
  const uint32_t tmem_o = tmem_base + 256;   // S buffers at columns [0,128) and [128,256)

  if (warp < SW) {
    // ============================ softmax / epilogue: thread = query row (x key half in the online kernel) ===========
    const int r = (warp & 3) * 32 + lane;
    const int hs = warp >> 2;   // key half of this thread (always 0 in the two-pass kernels)
    const int q = q0 + r;
    const bool qok = q < p.Lq;
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    float m_run = -INFINITY, l_run = 0.f;
    float lse_r = 0.f;
    if (PASS == 1) lse_r = qok ? p.lse[(int64_t)blockIdx.z * p.Lq + q] : 0.f;
    for (int j = 0; j < nkv; ++j) {
      const int buf = j & 1;
      mbar_wait(s_full + 8 * buf, (uint32_t)(j >> 1) & 1u);
      tcgen05_fence_after();
      const uint32_t ts = tmem_base + lane_off + buf * FA_BN;
      const int kbase = j * FA_BN;
      // The S row is read in two 64-column TMEM loads (one round trip each): with 16-column loads the softmax warps
      // spent most of their time waiting for tcgen05.ld round trips (8-16 per tile), not computing.
      if (PASS == 0) {
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
          float v[64];
          tmem_ld64(ts + half * 64, v);
          const int kb = kbase + half * 64;
          if (kb + 64 > p.Lk) {   // ragged last key tile only
#pragma unroll
            for (int e = 0; e < 64; ++e) v[e] = (kb + e < p.Lk) ? v[e] : -INFINITY;
          }
          float t0 = fmaxf(v[0], v[1]), t1 = fmaxf(v[2], v[3]), t2 = fmaxf(v[4], v[5]), t3 = fmaxf(v[6], v[7]);
#pragma unroll
          for (int e = 8; e < 64; e += 8) {
            t0 = fmaxf(t0, fmaxf(v[e], v[e + 1]));
            t1 = fmaxf(t1, fmaxf(v[e + 2], v[e + 3]));
            t2 = fmaxf(t2, fmaxf(v[e + 4], v[e + 5]));
            t3 = fmaxf(t3, fmaxf(v[e + 6], v[e + 7]));
          }
          const float tmax = fmaxf(fmaxf(t0, t1), fmaxf(t2, t3)) * p.scale_log2;   // scale > 0 commutes with max
          if (tmax > -INFINITY) {   // online update per 64 keys
            const float m_new = fmaxf(m_run, tmax);
            float sum = 0.f, sum_b = 0.f;
#pragma unroll
            for (int e = 0; e < 64; e += 2) {
              sum += fast_ex2(fmaf(v[e], p.scale_log2, -m_new));
              sum_b += fast_ex2(fmaf(v[e + 1], p.scale_log2, -m_new));
            }
            l_run = l_run * fast_ex2(m_run - m_new) + (sum + sum_b);
            m_run = m_new;
          }
        }
        tcgen05_fence_before();
        mbar_arrive(s_empty + 8 * buf);
      } else if (PASS == 2) {
        // ---- single pass, online softmax (head dim <= 256: S x2 and the whole O fit tensor memory) ----
        // The running maximum is LAZY: the O accumulator is only rescaled when a tile raises the row maximum by more
        // than 2^8 (P stays <= 256, harmless in bf16 / fp32); the decision is warp-uniform because tcgen05.ld/st are
        // warp-collective. Rescaling waits for P V of the previous tile (p_empty), which every tile does anyway.
        float v[64];
        tmem_ld64(ts + hs * 64, v);                    // this thread's 64 keys of the tile
        tcgen05_fence_before();
        mbar_arrive(s_empty + 8 * buf);                // S is in registers: Q K^T of tile j+2 may overwrite it
        const int kb = kbase + hs * 64;
        // The scores stay UNSCALED in registers: scale > 0, so the row maximum commutes with the scaling and the
        // exponent becomes one FFMA (v * scale - m) feeding MUFU.EX2. Per element: FMNMX + FFMA + MUFU + FADD (+ half a
        // pack) instead of FMUL + compare + select + FMNMX + FADD + MUFU + FADD -- the softmax warps were issue-bound next
        // to the 1024 MUFU cycles of a tile. Only a ragged last key tile takes the masked form.
        const bool ragged = kb + 64 > p.Lk;
        if (ragged) {
#pragma unroll
          for (int e = 0; e < 64; ++e) v[e] = (kb + e < p.Lk) ? v[e] : -INFINITY;
        }
        // four independent maxima (a single running maximum is a 64-deep dependent FMNMX chain on the critical path)
        float t0 = fmaxf(v[0], v[1]), t1 = fmaxf(v[2], v[3]), t2 = fmaxf(v[4], v[5]), t3 = fmaxf(v[6], v[7]);
#pragma unroll
        for (int e = 8; e < 64; e += 8) {
          t0 = fmaxf(t0, fmaxf(v[e], v[e + 1]));
          t1 = fmaxf(t1, fmaxf(v[e + 2], v[e + 3]));
          t2 = fmaxf(t2, fmaxf(v[e + 4], v[e + 5]));
          t3 = fmaxf(t3, fmaxf(v[e + 6], v[e + 7]));
        }
        float tmax = fmaxf(fmaxf(t0, t1), fmaxf(t2, t3)) * p.scale_log2;   // (-inf stays -inf)
        // row maximum over both key halves: exchange through shared memory (double-buffered by tile parity)
        xch[j & 1][hs][r] = tmax;
        asm volatile("bar.sync 2, 256;" ::: "memory");
        tmax = fmaxf(tmax, xch[j & 1][hs ^ 1][r]);
        const int pb = j & 1;
        const float m_new = fmaxf(m_run, tmax);        // identical in both threads of a row
        if (j == 0) {
          m_run = m_new;
        } else if (__any_sync(0xffffffffu, m_new > m_run + 8.f)) {
          // O must be stable: P V of tile j-1 (the latest user of P[(j-1)&1]) has to be complete
          mbar_wait(p_empty + 8 * ((j - 1) & 1), (uint32_t)((j - 1) >> 1) & 1u);
          tcgen05_fence_after();
          const float f = fast_ex2(m_run - m_new);     // 1 for rows whose maximum did not move
          const uint32_t to = tmem_o + lane_off;
          // the two threads of a row split the O columns (whole 64-column loads; a 64-wide O stays with half 0)
          const int ncw = p.DV / 64, cbeg = ncw >= 2 ? hs * (ncw / 2) : 0, cend = ncw >= 2 ? (hs ? ncw : ncw / 2) : (hs ? 0 : 1);
#pragma unroll 1
          for (int cw = cbeg; cw < cend; ++cw) {
            float ow[64];
            tmem_ld64(to + cw * 64, ow);
#pragma unroll
            for (int e = 0; e < 64; ++e) ow[e] *= f;
            tmem_st64(to + cw * 64, ow);
          }
          l_run *= f;
          m_run = m_new;
        }
        float sum = 0.f, sum_b = 0.f;
        mbar_wait(p_empty + 8 * pb, ((uint32_t)(j >> 1) & 1u) ^ 1u);   // P V of tile j-2 has consumed this P buffer
        {
          const uint32_t base = p_smem + pb * FA_P_BYTES + hs * (FA_BM * 128);   // P panel of this key half
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            uint32_t o[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int k0 = c * 8 + 2 * e;
              const float p0 = fast_ex2(fmaf(v[k0], p.scale_log2, -m_run)), p1 = fast_ex2(fmaf(v[k0 + 1], p.scale_log2, -m_run));
              if (e & 1) sum_b += p0 + p1;
              else sum += p0 + p1;
              __nv_bfloat162 q2 = __floats2bfloat162_rn(p0, p1);
              o[e] = *reinterpret_cast<uint32_t*>(&q2);
            }
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(base + sw128_offset(r, c)), "r"(o[0]), "r"(o[1]),
                         "r"(o[2]), "r"(o[3]) : "memory");
          }
        }
        l_run += sum + sum_b;                          // partial sum of this key half; combined in the epilogue
        tcgen05_fence_before();
        fence_proxy_async();
        mbar_arrive(p_full + 8 * pb);
      } else {
        const int pb = j & 1;
        mbar_wait(p_empty + 8 * pb, ((uint32_t)(j >> 1) & 1u) ^ 1u);   // P V of tile j-2 has consumed this P buffer
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
          float v[64];
          tmem_ld64(ts + half * 64, v);
          const int kb = kbase + half * 64;
          const uint32_t base = p_smem + pb * FA_P_BYTES + half * (FA_BM * 128);   // one 64-key panel per half
          const bool ragged1 = kb + 64 > p.Lk;
#pragma unroll
          for (int c = 0; c < 8; ++c) {                          // 16-byte chunks of the 128-byte row
            uint32_t o[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int k0 = c * 8 + 2 * e;
              float p0 = fast_ex2(fmaf(v[k0], p.scale_log2, -lse_r)), p1 = fast_ex2(fmaf(v[k0 + 1], p.scale_log2, -lse_r));
              if (ragged1) {
                p0 = (kb + k0 < p.Lk) ? p0 : 0.f;
                p1 = (kb + k0 + 1 < p.Lk) ? p1 : 0.f;
              }
              __nv_bfloat162 q2 = __floats2bfloat162_rn(p0, p1);
              o[e] = *reinterpret_cast<uint32_t*>(&q2);
            }
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(base + sw128_offset(r, c)), "r"(o[0]), "r"(o[1]),
                         "r"(o[2]), "r"(o[3]) : "memory");
          }
        }
        tcgen05_fence_before();
        mbar_arrive(s_empty + 8 * buf);
        fence_proxy_async();          // generic-proxy smem writes -> visible to the UMMA (async proxy)
        mbar_arrive(p_full + 8 * pb);
      }
    }
    if (PASS == 0) {
      if (qok) p.lse[(int64_t)blockIdx.z * p.Lq + q] = m_run + log2f(l_run);
    } else {
      float inv_l = 1.f;
      int cw_beg = 0, cw_end = p.DV;
      if (PASS == 2) {
        // both key halves hold a partial row sum under the same running maximum: combine, then split the O columns
        xch[0][hs][r] = l_run;
        asm volatile("bar.sync 2, 256;" ::: "memory");
        l_run += xch[0][hs ^ 1][r];
        inv_l = 1.f / l_run;
        if (qok && hs == 0) p.lse[(int64_t)blockIdx.z * p.Lq + q] = m_run + log2f(l_run);
        const int ncw = p.DV / 64;
        cw_beg = (ncw >= 2 ? hs * (ncw / 2) : 0) * 64;
        cw_end = (ncw >= 2 ? (hs ? ncw : ncw / 2) : (hs ? 0 : 1)) * 64;
      }
      mbar_wait(o_full, 0);
      tcgen05_fence_after();
      const uint32_t to = tmem_o + lane_off;
      __nv_bfloat16* orow = p.out + ((int64_t)b * p.Lq + q) * ((int64_t)p.H * p.dh) + (int64_t)h * p.dh + slice * p.DV;
#pragma unroll 1
      for (int cw = cw_beg; cw < cw_end; cw += 64) {
        float vw[64];
        tmem_ld64(to + cw, vw);
        if (!qok) continue;
#pragma unroll
      for (int c0 = cw; c0 < cw + 64; c0 += 16) {
        const float* v = vw + (c0 - cw);
        uint4 o0, o1;
        __nv_bfloat162* h0 = reinterpret_cast<__nv_bfloat162*>(&o0);
        __nv_bfloat162* h1 = reinterpret_cast<__nv_bfloat162*>(&o1);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          h0[e] = __floats2bfloat162_rn(v[2 * e] * inv_l, v[2 * e + 1] * inv_l);
          h1[e] = __floats2bfloat162_rn(v[8 + 2 * e] * inv_l, v[8 + 2 * e + 1] * inv_l);
        }
        reinterpret_cast<uint4*>(orow + c0)[0] = o0;
        reinterpret_cast<uint4*>(orow + c0)[1] = o1;
      }
      }
    }
    tcgen05_fence_before();
  } else if (warp == SW) {
    // ============================ UMMA issuer ============================
    const uint32_t idesc_s = make_idesc(FA_BM, FA_BN, 0, 0);
    const uint32_t idesc_o = make_idesc(FA_BM, p.DV, 0, 1);
    int qs = 0;      // QK ring position
    uint32_t qph = 0;
    int vs = 0;
    uint32_t vph = 0;
    auto issue_qk = [&](int j) {
      const int buf = j & 1;
      mbar_wait(s_empty + 8 * buf, ((uint32_t)(j >> 1) & 1u) ^ 1u);
      tcgen05_fence_after();
      for (int c = 0; c < nkc; ++c) {
        mbar_wait(qk_full + 8 * qs, qph);
        tcgen05_fence_after();
        if (elect_one()) {
          const uint32_t a = qk_smem + qs * FA_QK_STAGE_BYTES, bsm = a + FA_BM * 128;
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            umma_bf16(tmem_base + buf * FA_BN, make_smem_desc(a + kk * 32, 16, 1024), make_smem_desc(bsm + kk * 32, 16, 1024),
                      idesc_s, (c | kk) ? 1u : 0u);
          umma_commit(qk_empty + 8 * qs);
          if (c == nkc - 1) umma_commit(s_full + 8 * buf);
        }
        __syncwarp();
        if (++qs == p.qk_stages) { qs = 0; qph ^= 1u; }
      }
    };
    issue_qk(0);
    for (int j = 0; j < nkv; ++j) {
      if (j + 1 < nkv) issue_qk(j + 1);
      if (PASS >= 1) {
        mbar_wait(p_full + 8 * (j & 1), (uint32_t)(j >> 1) & 1u);
        tcgen05_fence_after();
        for (int half = 0; half < 2; ++half) {
          mbar_wait(v_full + 8 * vs, vph);
          tcgen05_fence_after();
          if (elect_one()) {
            const uint32_t a = p_smem + (j & 1) * FA_P_BYTES + half * (FA_BM * 128), bsm = v_smem + vs * v_stage_bytes;
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
              umma_bf16(tmem_o, make_smem_desc(a + kk * 32, 16, 1024), make_smem_desc(bsm + kk * 2048, FA_PANEL, 1024),
                        idesc_o, (j | half | kk) ? 1u : 0u);
            umma_commit(v_empty + 8 * vs);
            if (half == 1) {
              umma_commit(p_empty + 8 * (j & 1));
              if (j == nkv - 1) umma_commit(o_full);
            }
          }
          __syncwarp();
          if (++vs == FA_V_STAGES) { vs = 0; vph ^= 1u; }
        }
      }
    }
  } else if (elect_one()) {
    // ============================ TMA issuer ============================
    int qs = 0, vs = 0;
    uint32_t qph = 0, vph = 0;
    auto load_qk = [&](int j) {
      for (int c = 0; c < nkc; ++c) {
        mbar_wait(qk_empty + 8 * qs, qph ^ 1u);
        const uint32_t a = qk_smem + qs * FA_QK_STAGE_BYTES, bar = qk_full + 8 * qs;
        mbar_arrive_expect_tx(bar, FA_QK_STAGE_BYTES);
        tma_load_4d(a, &qmap, bar, c * 64, h, q0, b);
        tma_load_4d(a + FA_BM * 128, &kmap, bar, c * 64, h, j * FA_BN, b);
        if (++qs == p.qk_stages) { qs = 0; qph ^= 1u; }
      }
    };
    auto load_v = [&](int j) {
      for (int half = 0; half < 2; ++half) {
        mbar_wait(v_empty + 8 * vs, vph ^ 1u);
        const uint32_t dst = v_smem + vs * v_stage_bytes, bar = v_full + 8 * vs;
        mbar_arrive_expect_tx(bar, v_stage_bytes);
        for (int pn = 0; pn < p.DV / 64; ++pn)
          tma_load_4d(dst + pn * FA_PANEL, &vmap, bar, slice * p.DV + pn * 64, h, j * FA_BN + half * 64, b);
        if (++vs == FA_V_STAGES) { vs = 0; vph ^= 1u; }
      }
    };
    load_qk(0);
    for (int j = 0; j < nkv; ++j) {
      if (j + 1 < nkv) load_qk(j + 1);
      if (PASS >= 1) load_v(j);
    }
  }
  __syncthreads();
  if (warp == SW) {
    tcgen05_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// -----------------------------------------------------------------------------------------------------------------
// Head dim 64 / 128: the PAIR kernel. ncu on flash_fwd_kernel<2> at the config-4 sampling shape (L = 32768, d = 128)
// showed the tensor pipe 40 % active with neither MUFU nor issue slots saturated: the limit was SHARED-MEMORY traffic.
// Per 128 x 128 score tile that kernel moves 256 KB through shared memory (Q and K chunks re-streamed 32 + 32 KB, V
// 32 KB, P written 32 KB and read back 32 KB, the UMMA operand reads of Q / K / V 96 KB) = 2048 cycles at 128 B/clk
// against 1024 cycles of UMMA. This kernel cuts it to 128 KB per tile:
//   * one CTA owns TWO 128-row query tiles; Q (2 x 128 x dh) is loaded once and stays resident;
//   * every K / V tile is loaded once and used by both query tiles;
//   * P never touches shared memory: the softmax threads write it as packed bf16 into tensor memory over the first 64
//     columns of the S tile they have just read (tcgen05.st), and P V is issued with the A operand IN tensor memory
//     (tcgen05.mma [d], [a_tmem], b_desc). tcgen05.mma executes in issue order, so Q K^T of tile j+1 (which overwrites
//     S / P) is simply issued after P V of tile j.
// The two query tiles ping-pong: while softmax group g works on S_g the tensor pipe runs the other tile's MMAs.
// Tensor memory: S0 [0,128) S1 [128,256) O0 [256,384) O1 [384,512).
// Roles (384 threads): warps 0-3 softmax of query tile 0 (thread = row, all 128 keys of a tile in registers: no
// exchange between key halves), warps 4-7 of query tile 1, warp 8 UMMA issuer + TMEM allocator, warp 9 TMA issuer,
// warps 10-11 idle (they complete the third warpgroup for setmaxnreg).
// -----------------------------------------------------------------------------------------------------------------
// 384 threads = three warpgroups, because setmaxnreg moves registers between WHOLE warpgroups: the softmax threads keep a
// 128-value score row plus the packed P row in registers (the 168 registers a 384-thread CTA starts with spill half the
// row to local memory), the issuer warpgroup (UMMA warp, TMA warp, two idle warps) needs almost none.
constexpr int FP_THREADS = 384, FP_KV_STAGES = 2;

__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// 32 packed words -> 32 consecutive TMEM columns of this thread's lane; completion is awaited by tmem_wait_st()
__device__ __forceinline__ void tmem_st32_nowait(uint32_t taddr, const uint32_t w[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      :
      : "r"(taddr), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]), "r"(w[8]),
        "r"(w[9]), "r"(w[10]), "r"(w[11]), "r"(w[12]), "r"(w[13]), "r"(w[14]), "r"(w[15]), "r"(w[16]), "r"(w[17]),
        "r"(w[18]), "r"(w[19]), "r"(w[20]), "r"(w[21]), "r"(w[22]), "r"(w[23]), "r"(w[24]), "r"(w[25]), "r"(w[26]),
        "r"(w[27]), "r"(w[28]), "r"(w[29]), "r"(w[30]), "r"(w[31])
      : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 128 consecutive columns as two 64-column loads in flight together and ONE wait (a second round trip costs ~100 cycles
// on the softmax critical path). The empty volatile asm statements pin every use of the registers behind the wait.
__device__ __forceinline__ void tmem_ld128(uint32_t taddr, float v[128]) {
  uint32_t r[128];
#pragma unroll
  for (int hlf = 0; hlf < 2; ++hlf) {
    uint32_t* q = r + 64 * hlf;
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, %48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
        : "=r"(q[0]), "=r"(q[1]), "=r"(q[2]), "=r"(q[3]), "=r"(q[4]), "=r"(q[5]), "=r"(q[6]), "=r"(q[7]), "=r"(q[8]), "=r"(q[9]), "=r"(q[10]), "=r"(q[11]), "=r"(q[12]), "=r"(q[13]), "=r"(q[14]), "=r"(q[15]), "=r"(q[16]), "=r"(q[17]), "=r"(q[18]), "=r"(q[19]), "=r"(q[20]), "=r"(q[21]), "=r"(q[22]), "=r"(q[23]), "=r"(q[24]), "=r"(q[25]), "=r"(q[26]), "=r"(q[27]), "=r"(q[28]), "=r"(q[29]), "=r"(q[30]), "=r"(q[31]), "=r"(q[32]), "=r"(q[33]), "=r"(q[34]), "=r"(q[35]), "=r"(q[36]), "=r"(q[37]), "=r"(q[38]), "=r"(q[39]), "=r"(q[40]), "=r"(q[41]), "=r"(q[42]), "=r"(q[43]), "=r"(q[44]), "=r"(q[45]), "=r"(q[46]), "=r"(q[47]), "=r"(q[48]), "=r"(q[49]), "=r"(q[50]), "=r"(q[51]), "=r"(q[52]), "=r"(q[53]), "=r"(q[54]), "=r"(q[55]), "=r"(q[56]), "=r"(q[57]), "=r"(q[58]), "=r"(q[59]), "=r"(q[60]), "=r"(q[61]), "=r"(q[62]), "=r"(q[63])
        : "r"(taddr + 64 * hlf)
        : "memory");
  }
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 128; ++i) {
    asm volatile("" : "+r"(r[i]));
    v[i] = __uint_as_float(r[i]);
  }
}

// 2^x on the FMA pipe (Cody-Waite: x = n + f, |f| <= 0.5; degree-3 minimax polynomial for 2^f, relative error 7.5e-5 --
// far below the bf16 rounding of P). The 16 MUFU lanes of an SM need 2048 cycles for the 2 x 128 x 128 exponentials of
// one key tile, exactly the UMMA time of that tile; with POLY one exponential in four goes through here instead
// (optional, off by default: see launch_flash_pair).
__device__ __forceinline__ float poly_ex2(float x) {
  x = fmaxf(x, -125.f);
  const float t = x + 12582912.f;          // 1.5 * 2^23: round-to-nearest leaves n in the low mantissa bits
  const float f = x - (t - 12582912.f);
  float y = fmaf(f, 0.0551716648f, 0.2426111251f);
  y = fmaf(y, f, 0.6932609677f);
  y = fmaf(y, f, 0.9999280572f);
  return __int_as_float(__float_as_int(y) + (__float_as_int(t) << 23));
}

// bars: q_full k_full[2] k_empty[2] v_full[2] v_empty[2] s_full[2] p_full[2][2] pv_done[2]
// P is handed to the UMMA issuer in two 64-key halves: P V of the first half runs while the softmax threads still
// exponentiate the second half (the softmax latency, not its throughput, sets the pace of a query tile's
// S -> P -> P V -> next S chain).
template <int DH, bool POLY>
__global__ void __launch_bounds__(FP_THREADS, 1) flash_pair_kernel(const __grid_constant__ CUtensorMap qmap,   // 128-row boxes
                                                               const __grid_constant__ CUtensorMap kmap,   // 128-row boxes
                                                               const __grid_constant__ CUtensorMap vmap,   // 64-row boxes
                                                               FlashParams p) {
  constexpr int NC = DH / 64;                       // 64-channel chunks of the head dim
  constexpr int TILE_BYTES = NC * FA_BM * 128;      // one 128-row tile of Q / K / V
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t q_smem = smem_base;
  const uint32_t k_smem = q_smem + 2 * TILE_BYTES;
  const uint32_t v_smem = k_smem + FP_KV_STAGES * TILE_BYTES;
  __shared__ __align__(8) uint64_t bars[17];
  __shared__ uint32_t tmem_slot;
  const uint32_t b0 = smem_u32(&bars[0]);
  const uint32_t q_full = b0, k_full = b0 + 8 * 1, k_empty = b0 + 8 * 3, v_full = b0 + 8 * 5, v_empty = b0 + 8 * 7,
                 s_full = b0 + 8 * 9, p_full = b0 + 8 * 11 /* [g][half] */, pv_done = b0 + 8 * 15;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * (2 * FA_BM);
  const int b = blockIdx.z / p.H, h = blockIdx.z - b * p.H;
  const int nkv = (p.Lk + FA_BN - 1) / FA_BN;

  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(k_full + 8 * i, 1); mbar_init(k_empty + 8 * i, 1);
      mbar_init(v_full + 8 * i, 1); mbar_init(v_empty + 8 * i, 1);
      mbar_init(s_full + 8 * i, 1); mbar_init(pv_done + 8 * i, 1);
      mbar_init(p_full + 16 * i, 128); mbar_init(p_full + 16 * i + 8, 128);
    }
    fence_barrier_init();
  }
  if (warp == 8) tmem_alloc<512>(smem_u32(&tmem_slot));
  if (warp == 9 && lane == 0) { tma_prefetch_desc(&qmap); tma_prefetch_desc(&kmap); tma_prefetch_desc(&vmap); }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_slot;

  if (warp < 8) {
    // ============================ softmax / epilogue: thread = query row of tile g ============================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
    const int g = warp >> 2;
    const int r = (warp & 3) * 32 + lane;
    const int q = q0 + g * FA_BM + r;
    const bool qok = q < p.Lq;
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t ts = tmem_base + lane_off + g * FA_BN;          // S_g; P_g = its first 64 columns, packed bf16
    const uint32_t to = tmem_base + lane_off + 256 + g * 128;      // O_g
    float m_run = -INFINITY, l_run = 0.f;
    for (int j = 0; j < nkv; ++j) {
      mbar_wait(s_full + 8 * g, (uint32_t)j & 1u);
      tcgen05_fence_after();
      float v[128];
      tmem_ld128(ts, v);
      const int kbase = j * FA_BN;
      if (kbase + FA_BN > p.Lk) {   // ragged last key tile only
#pragma unroll
        for (int e = 0; e < 128; ++e) v[e] = (kbase + e < p.Lk) ? v[e] : -INFINITY;
      }
      // scores stay unscaled (scale > 0 commutes with the maximum); four independent maxima
      float t0 = fmaxf(v[0], v[1]), t1 = fmaxf(v[2], v[3]), t2 = fmaxf(v[4], v[5]), t3 = fmaxf(v[6], v[7]);
#pragma unroll
      for (int e = 8; e < 128; e += 8) {
        t0 = fmaxf(t0, fmaxf(v[e], v[e + 1]));
        t1 = fmaxf(t1, fmaxf(v[e + 2], v[e + 3]));
        t2 = fmaxf(t2, fmaxf(v[e + 4], v[e + 5]));
        t3 = fmaxf(t3, fmaxf(v[e + 6], v[e + 7]));
      }
      const float tmax = fmaxf(fmaxf(t0, t1), fmaxf(t2, t3)) * p.scale_log2;
      const float m_new = fmaxf(m_run, tmax);
      if (j == 0) {
        m_run = m_new;
      } else if (__any_sync(0xffffffffu, m_new > m_run + 8.f)) {
        // LAZY rescale (P stays <= 2^8): O_g must be stable, i.e. P V of tile j-1 complete
        mbar_wait(pv_done + 8 * g, (uint32_t)(j - 1) & 1u);
        tcgen05_fence_after();
        const float f = fast_ex2(m_run - m_new);   // 1 for rows whose maximum did not move
#pragma unroll 1
        for (int cw = 0; cw < DH; cw += 64) {
          float ow[64];
          tmem_ld64(to + cw, ow);
#pragma unroll
          for (int e = 0; e < 64; ++e) ow[e] *= f;
          tmem_st64(to + cw, ow);
        }
        l_run *= f;
        m_run = m_new;
      }
      float sum = 0.f, sum_b = 0.f;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t w[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const int k0 = half * 64 + 2 * i;
          const float x1 = fmaf(v[k0 + 1], p.scale_log2, -m_run);
          const float p0 = fast_ex2(fmaf(v[k0], p.scale_log2, -m_run));
          const float p1 = (POLY && (i & 1)) ? poly_ex2(x1) : fast_ex2(x1);
          if (i & 1) sum_b += p0 + p1;
          else sum += p0 + p1;
          __nv_bfloat162 q2 = __floats2bfloat162_rn(p0, p1);
          w[i] = *reinterpret_cast<uint32_t*>(&q2);
        }
        tmem_st32_nowait(ts + half * 32, w);
        tmem_wait_st();
        tcgen05_fence_before();
        mbar_arrive(p_full + 16 * g + 8 * half);
      }
      l_run += sum + sum_b;
    }
    // ---- epilogue ----
    const float inv_l = 1.f / l_run;
    if (qok) p.lse[(int64_t)blockIdx.z * p.Lq + q] = m_run + log2f(l_run);
    mbar_wait(pv_done + 8 * g, (uint32_t)(nkv - 1) & 1u);
    tcgen05_fence_after();
    __nv_bfloat16* orow = p.out + ((int64_t)b * p.Lq + q) * ((int64_t)p.H * DH) + (int64_t)h * DH;
#pragma unroll 1
    for (int cw = 0; cw < DH; cw += 64) {
      float vw[64];
      tmem_ld64(to + cw, vw);
      if (!qok) continue;
#pragma unroll
      for (int c0 = 0; c0 < 64; c0 += 8) {
        uint4 o;
        __nv_bfloat162* hh = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
        for (int e = 0; e < 4; ++e) hh[e] = __floats2bfloat162_rn(vw[c0 + 2 * e] * inv_l, vw[c0 + 2 * e + 1] * inv_l);
        *reinterpret_cast<uint4*>(orow + cw + c0) = o;
      }
    }
    tcgen05_fence_before();
  } else if (warp == 8) {
    // ============================ UMMA issuer (one elected thread) ============================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
    if (elect_one()) {
      constexpr uint32_t idesc_s = make_idesc(FA_BM, FA_BN, 0, 0);
      constexpr uint32_t idesc_o = make_idesc(FA_BM, DH, 0, 1);
      auto issue_s = [&](int g, int j) {   // S_g = Q_g K_j^T
        const uint32_t a = q_smem + g * TILE_BYTES, bsm = k_smem + (j % FP_KV_STAGES) * TILE_BYTES;
#pragma unroll
        for (int c = 0; c < NC; ++c)
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            umma_bf16(tmem_base + g * FA_BN, make_smem_desc(a + c * (FA_BM * 128) + kk * 32, 16, 1024),
                      make_smem_desc(bsm + c * (FA_BN * 128) + kk * 32, 16, 1024), idesc_s, (c | kk) ? 1u : 0u);
        umma_commit(s_full + 8 * g);
      };
      mbar_wait(q_full, 0);
      mbar_wait(k_full, 0);
      tcgen05_fence_after();
      issue_s(0, 0);
      issue_s(1, 0);
      umma_commit(k_empty);
      for (int j = 0; j < nkv; ++j) {
        const int vs = j % FP_KV_STAGES;
        const uint32_t vph = (uint32_t)(j / FP_KV_STAGES) & 1u;
        mbar_wait(v_full + 8 * vs, vph);
        for (int g = 0; g < 2; ++g) {
          const uint32_t bsm = v_smem + vs * TILE_BYTES;
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            mbar_wait(p_full + 16 * g + 8 * half, (uint32_t)j & 1u);
            tcgen05_fence_after();
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)   // A = P_g (tensor memory, 8 columns per 16 keys); B = 16 key rows of every 64-channel panel
              umma_bf16_ts(tmem_base + 256 + g * 128, tmem_base + g * FA_BN + half * 32 + kk * 8,
                           make_smem_desc(bsm + half * (NC * FA_PANEL) + kk * 2048, FA_PANEL, 1024), idesc_o,
                           (j | half | kk) ? 1u : 0u);
          }
          umma_commit(pv_done + 8 * g);
          if (g == 1) umma_commit(v_empty + 8 * vs);
          if (j + 1 < nkv) {
            const int ks = (j + 1) % FP_KV_STAGES;
            if (g == 0) {
              mbar_wait(k_full + 8 * ks, (uint32_t)((j + 1) / FP_KV_STAGES) & 1u);
              tcgen05_fence_after();
            }
            issue_s(g, j + 1);
            if (g == 1) umma_commit(k_empty + 8 * ks);
          }
        }
      }
    }
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
    if (warp == 9 && elect_one()) {
    // ============================ TMA issuer ============================
    mbar_arrive_expect_tx(q_full, 2 * TILE_BYTES);
    for (int g = 0; g < 2; ++g)
      for (int c = 0; c < NC; ++c)
        tma_load_4d(q_smem + g * TILE_BYTES + c * (FA_BM * 128), &qmap, q_full, c * 64, h, q0 + g * FA_BM, b);
    for (int j = 0; j < nkv; ++j) {
      const int s = j % FP_KV_STAGES;
      const uint32_t ph = (uint32_t)(j / FP_KV_STAGES) & 1u;
      mbar_wait(k_empty + 8 * s, ph ^ 1u);
      mbar_arrive_expect_tx(k_full + 8 * s, TILE_BYTES);
      for (int c = 0; c < NC; ++c)
        tma_load_4d(k_smem + s * TILE_BYTES + c * (FA_BN * 128), &kmap, k_full + 8 * s, c * 64, h, j * FA_BN, b);
      mbar_wait(v_empty + 8 * s, ph ^ 1u);
      mbar_arrive_expect_tx(v_full + 8 * s, TILE_BYTES);
      for (int half = 0; half < 2; ++half)
        for (int pn = 0; pn < NC; ++pn)
          tma_load_4d(v_smem + s * TILE_BYTES + half * (NC * FA_PANEL) + pn * FA_PANEL, &vmap, v_full + 8 * s, pn * 64, h,
                      j * FA_BN + half * 64, b);
    }
    }
  }
  __syncthreads();
  if (warp == 8) {
    tcgen05_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

bool flash_eligible(int H, int dh) {
  if (dh % 64 != 0) return false;
  if (dh > 256 && dh % 256 != 0) return false;
  return H >= 1;
}

template <int PASS>
static int launch_flash(const CUtensorMap& qm, const CUtensorMap& km, const CUtensorMap& vm, FlashParams p,
                        dim3 grid, cudaStream_t st) {
  auto bytes = [&](int qk_stages) {
    return qk_stages * FA_QK_STAGE_BYTES + 2 * FA_P_BYTES + FA_V_STAGES * (p.DV / 64) * FA_PANEL + 1024;
  };
  p.qk_stages = bytes(FA_QK_STAGES) <= 227 * 1024 - 4096 ? FA_QK_STAGES : 2;   // 4 KB left for static shared memory
  const int smem = bytes(p.qk_stages);
  static SmemOptIn optin;
  if (int rc = ensure_dynamic_smem(flash_fwd_kernel<PASS>, smem, optin, "flash_attention")) return rc;
  flash_fwd_kernel<PASS><<<grid, (fa_softmax_warps(PASS) + 2) * 32, smem, st>>>(qm, km, vm, p);
  return check_launch("flash_fwd_kernel");
}

template <int DH>
static int launch_flash_pair(const CUtensorMap& qm, const CUtensorMap& km, const CUtensorMap& vm, const FlashParams& p,
                             cudaStream_t st) {
  const int smem = (2 + 2 * FP_KV_STAGES) * (DH / 64) * FA_BM * 128 + 1024;
  // polynomial exp2 for one exponential in four: measured no faster than MUFU alone (the kernel is not MUFU-bound), so
  // the exact path is the default; MIG_FLASH_POLY=1 keeps the variant available for A/B runs
  static const bool poly = [] {
    const char* e = getenv("MIG_FLASH_POLY");
    return e && e[0] == '1';
  }();
  const dim3 grid((p.Lq + 2 * FA_BM - 1) / (2 * FA_BM), 1, p.B * p.H);
  if (poly) {
    static SmemOptIn optin;
    if (int rc = ensure_dynamic_smem(flash_pair_kernel<DH, true>, smem, optin, "flash_attention (pair)")) return rc;
    flash_pair_kernel<DH, true><<<grid, FP_THREADS, smem, st>>>(qm, km, vm, p);
  } else {
    static SmemOptIn optin;
    if (int rc = ensure_dynamic_smem(flash_pair_kernel<DH, false>, smem, optin, "flash_attention (pair)")) return rc;
    flash_pair_kernel<DH, false><<<grid, FP_THREADS, smem, st>>>(qm, km, vm, p);
  }
  return check_launch("flash_pair_kernel");
}

static bool flash_pair_enabled() {
  static const bool on = [] {
    const char* e = getenv("MIG_FLASH_PAIR");
    return !(e && e[0] == '0');
  }();
  return on;
}

}  // namespace mig

using namespace mig;

extern "C" int mig_flash_attention_fwd_ld(const void* q, const void* k, const void* v, void* out, float* lse, int32_t B,
                                          int32_t H, int32_t Lq, int32_t Lk, int32_t dh, int64_t ldq, int64_t ldk,
                                          int64_t ldv, float scale, void* stream) {
  MIG_REQUIRE(q && k && v && out && lse, "flash_attention: null argument");
  MIG_REQUIRE(mig_has_tcgen05(), "flash_attention: needs an sm_100 device");
  MIG_REQUIRE(flash_eligible(H, dh), "flash_attention: head dim %d not supported (multiple of 64; above 256 a multiple of 256)", dh);
  MIG_REQUIRE(B > 0 && Lq > 0 && Lk > 0 && (int64_t)B * H < 65536, "flash_attention: bad sizes");
  MIG_REQUIRE(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v) |
                reinterpret_cast<uintptr_t>(out)) & 15) == 0, "flash_attention: tensors must be 16-byte aligned");
  const int64_t C = (int64_t)H * dh;
  MIG_REQUIRE(ldq >= C && ldk >= C && ldv >= C && ((ldq | ldk | ldv) & 7) == 0,
              "flash_attention: row pitches must be >= H*dh and multiples of 8 elements");
  CUtensorMap qm, km, vm;
  if (bhld_map(&qm, q, B, H, Lq, dh, FA_BM, ldq)) return 1;
  if (bhld_map(&km, k, B, H, Lk, dh, FA_BN, ldk)) return 1;
  if (bhld_map(&vm, v, B, H, Lk, dh, 64, ldv)) return 1;
  FlashParams p{};
  p.B = B; p.H = H; p.Lq = Lq; p.Lk = Lk; p.dh = dh;
  p.DV = dh > 256 ? 256 : dh;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.lse = lse;
  p.out = (__nv_bfloat16*)out;
  cudaStream_t st = as_stream(stream);
  const unsigned mt = (Lq + FA_BM - 1) / FA_BM;
  if (flash_pair_enabled() && dh == 128) return launch_flash_pair<128>(qm, km, vm, p, st);
  if (flash_pair_enabled() && dh == 64) return launch_flash_pair<64>(qm, km, vm, p, st);
  if (dh <= 256) return launch_flash<2>(qm, km, vm, p, dim3(mt, 1, B * H), st);   // single pass, online softmax
  if (launch_flash<0>(qm, km, vm, p, dim3(mt, 1, B * H), st)) return 2;
  return launch_flash<1>(qm, km, vm, p, dim3(mt, dh / p.DV, B * H), st);
}

extern "C" int mig_flash_attention_fwd(const void* q, const void* k, const void* v, void* out, float* lse, int32_t B,
                                       int32_t H, int32_t Lq, int32_t Lk, int32_t dh, float scale, void* stream) {
  const int64_t C = (int64_t)H * dh;
  return mig_flash_attention_fwd_ld(q, k, v, out, lse, B, H, Lq, Lk, dh, C, C, C, scale, stream);
}

// tcgen05 engine, part 3: all-TMA implicit-GEMM convolution (fwd / dgrad: source channels >= 48, multiple of 8; wgrad:
// multiple of 64; stride 1, or stride 2 through tensor-map element strides / stride-residue classes).
//
// The im2col matrix is never gathered by threads. The NDHWC activation tensor is described to the TMA unit as a
// 5-d tensor (C, W, H, D, N); a GEMM row tile is a BOX of voxels (bw x bh x bd voxels in a 64- or 128-row slot) and
// the K loop walks (filter tap, 64-channel chunk). For tap (tz,ty,tx) the A tile is simply the same box shifted by the
// tap offset; coordinates that fall outside the tensor are filled with zeros by the TMA unit, which IS the
// convolution's zero padding (the halo). ONE elected thread issues the TMA loads (odometer indexing, warp-uniform
// arithmetic), one thread issues the UMMAs, four warps only run the epilogue -- there is no address arithmetic and no
// load instruction in the main loop at all, and up to STAGES-1 whole stages (~130 KB) are in flight per SM.
//
// The CTA tile is made as large as TMEM allows: MT = 2 stacks two 128-row UMMA accumulators that share every B stage
// (256 x 256 per tile = all 512 TMEM columns); narrower layers keep two accumulator sets so that the epilogue of one
// tile overlaps the main loop of the next. What was learnt from ncu on the way (DESIGN.md section 4.1): the producer
// THREAD, not the TMA unit, limited the first versions (one lane per box, divisions per stage); the 24^3-level layers
// now run at the same rate as cuBLAS bf16 GEMMs on this pool.
//
//   conv_tma_kernel   persistent; fwd and dgrad (dgrad = same kernel on dY with mirrored taps and the transposed filter)
//   wgrad_tma_kernel  dW[Cout][tap*Cin] += dY^T * im2col(X): both operands MN-major, voxel reduction walks boxes,
//                     split across CTAs, fp32 red.global.add into the gradient.
#include <cuda.h>

#include <mutex>

#include "common.cuh"
#include "residue_classes.cuh"
#include "tc_common.cuh"
#include "tc_host.cuh"

namespace mig {

using namespace tc;

int filter_transpose(int dtype, const void* w, void* wt, int Cout, int Tn, int Cin, void* stream);

constexpr int TBM = 128, TBK = 64, kThreads = 192, PANEL = 64 * 128;
// conv_tma_kernel: warps 0-3 and 6-9 are TWO epilogue groups (a warp reads the TMEM lane quadrant warp % 4; the groups
// split the accumulator columns in 64-column chunks), warp 4 issues the UMMAs, warp 5 the TMA loads. With one group the
// epilogue of a 256 x 256 tile (all 512 TMEM columns, so nothing to overlap it with) cost ~6 k cycles next to a ~55 k
// cycle main loop; the second group halves that and pays for the GroupNorm statistics the epilogue now also produces.
constexpr int kConvThreads = 320;
constexpr int kSmemBudget = 200 * 1024;
__host__ __device__ constexpr int stages_of(int stage_bytes) {
  return kSmemBudget / stage_bytes > 8 ? 8 : kSmemBudget / stage_bytes;
}
__host__ __device__ constexpr int tmem_cols(int c) { return c <= 32 ? 32 : (c <= 64 ? 64 : (c <= 128 ? 128 : (c <= 256 ? 256 : 512))); }

__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::
          "r"(dst),
      "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

struct BoxGeom {
  int N, D, H, W;        // extent of the GEMM-row side (conv output for fwd, conv input for dgrad)
  int bd, bh, bw;        // box; boxes may overhang the tensor
  int rb, nb;            // rows per shared-memory slot (64 or 128) and valid rows per box (bd*bh*bw <= rb);
                         // wgrad: rb = 64 and nb a multiple of 16 (the box is one K stage of nb/16 UMMAs)
  int nbd, nbh, nbw;     // boxes per axis (ceil)
  uint32_t dmul[3], dshr[3];   // division by nbw / nbh / nbd as multiply-high + shift (set_box_counts); dividends < 2^31
  int64_t num_boxes;     // N*nbd*nbh*nbw
  int ks[3];             // kernel
  int off[3];            // source coordinate = row coordinate + tap*sign + off   (fwd: +1, -pad; dgrad: -1, +pad)
  int sign;
  int ss[3];             // source stride: source coordinate = row*ss + tap*sign + off (2 for a stride-2 forward conv /
                         // wgrad, where the TMA tensor map walks the source with the same element stride)
  int Csrc, Cdst, K;     // K = taps*Csrc
  int cchunks;           // ceil(Csrc / 64): the last chunk of a 96-channel source reads 32 channels past the end, which
                         // TMA zero-fills in the activation box (so whatever the filter box holds there is multiplied by 0)
  // where a row lands in the output tensor: coordinate = row*os + oo inside an (OD,OH,OW) volume. Identity except
  // for strided dgrad, where each stride-residue class of input voxels is its own dense stride-1 problem.
  int os[3], oo[3], OD, OH, OW;
};

// box index -> (sample, box origin). Every tile of every role decodes several boxes; with plain 64-bit / and % (a
// reciprocal + correction sequence each) the epilogue of a small-K tile (1x1x1 convs on 32/64 channels) spent most of its
// ~2000 instructions per tile dividing -- ncu: 8700 cycles per tile on a layer whose main loop is four UMMAs.
__device__ __forceinline__ uint32_t fast_div(uint32_t x, int d, uint32_t mul, uint32_t shr) {
  return d == 1 ? x : __umulhi(x, mul) >> shr;
}
__device__ __forceinline__ void box_origin(const BoxGeom& g, int64_t box, int& n, int& d0, int& h0, int& w0) {
  uint32_t r = (uint32_t)box;
  uint32_t q = fast_div(r, g.nbw, g.dmul[0], g.dshr[0]);
  w0 = (int)(r - q * (uint32_t)g.nbw) * g.bw; r = q;
  q = fast_div(r, g.nbh, g.dmul[1], g.dshr[1]);
  h0 = (int)(r - q * (uint32_t)g.nbh) * g.bh; r = q;
  q = fast_div(r, g.nbd, g.dmul[2], g.dshr[2]);
  d0 = (int)(r - q * (uint32_t)g.nbd) * g.bd;
  n = (int)q;
}

// Dynamic tile scheduler state of one launch. A CTA's first tile is blockIdx.x; every further tile is
// gridDim.x + atomicAdd(next, 1). The last CTA to finish zeroes the pair again, so a slot is reusable by the next launch
// that picks it (and by every replay of a CUDA graph that captured it) without a memset node per convolution.
struct TileCounter {
  unsigned int next, done;
};

struct ConvTmaParams {
  BoxGeom g;
  const float* bias;
  const float* chan_bias;
  const __nv_bfloat16* residual;
  __nv_bfloat16* out;
  float* partial;
  int num_kb, kb_per_split;
  int mtiles, ntiles, splits;   // tile grid; tile index = (split * ntiles + ntile) * mtiles + mtile
  // GroupNorm statistics of the OUTPUT, accumulated by the epilogue (forward, no split-K): sums[n][g][2] (fp64) +=
  // (sum y, sum y^2) of the bf16-rounded values, for the GroupNorm that consumes this convolution (unet:648,698 / ae:167)
  double* gn_sums;
  int gn_cpg, gn_G;
  int epi_groups;   // 1 or 2 epilogue warp groups (A/B switch MIG_CONV_EPI_GROUPS; default 2)
  TileCounter* sched;   // dynamic tile counter of this launch (nullptr: static round-robin)
};

// Sum eight per-thread values over the 32 lanes of a warp with 7 + 2 shuffles (recursive halving: after step k every
// lane keeps 8 / 2^k values). Returns, in every lane, the warp total of value index ((lane>>4)&1)*4 + ((lane>>3)&1)*2 +
// ((lane>>2)&1).
__device__ __forceinline__ float warp_sum8(const float v[8], int lane) {
  float a[4], b[2], c;
  const bool h16 = lane & 16, h8 = lane & 8, h4 = lane & 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float keep = h16 ? v[i + 4] : v[i], send = h16 ? v[i] : v[i + 4];
    a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const float keep = h8 ? a[i + 2] : a[i], send = h8 ? a[i] : a[i + 2];
    b[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
  {
    const float keep = h4 ? b[1] : b[0], send = h4 ? b[0] : b[1];
    c = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  c += __shfl_xor_sync(0xffffffffu, c, 2);
  c += __shfl_xor_sync(0xffffffffu, c, 1);
  return c;
}

// BN: output-channel tile; MT: number of stacked 128-row accumulators (tile = MT*128 voxels x BN channels).
//
// PERSISTENT: one CTA per SM walks a sequence of tiles: blockIdx.x, blockIdx.x + gridDim.x, ... by default, or -- with a
// TileCounter (p.sched) -- drawn dynamically: the TMA thread draws the next tile index while it loads the current one.
// Either way the TMA thread hands the indices to the UMMA warp and the epilogue threads through a small shared-memory
// ring. (Why dynamic: with the static round-robin a CTA that starts late does its whole share late, e.g. when an NCCL
// kernel of the overlapped gradient exchange holds its SM. See next_tile_counter() for what was measured.)
// The shared-memory ring and its
// barriers run straight through tile boundaries, so the producer prefetches the next tile's operands while the
// current tile is still in the tensor pipe; when two accumulator sets fit in tensor memory (2*MT*BN <= 512 columns)
// the epilogue of tile i also overlaps the main loop of tile i+1. ncu on the one-tile-per-CTA version showed ~15 k
// cycles of launch / TMEM allocation / pipeline fill / drain around every tile: 12 % of a 256x256x6912 tile, and four
// times the 3.5 k-cycle main loop of a 64-channel layer.
// BMN: the B operand (filter) is MN-major -- the UNTRANSPOSED filter [Csrc][tap][Cdst] read through a 3-d tensor map as
// 64 x 64 panels. This is how dgrad runs on the forward filter layout without a per-step transposed copy.
template <int BN, int MT, bool BMN = false>
__global__ void __launch_bounds__(kConvThreads, 1) conv_tma_kernel(const __grid_constant__ CUtensorMap xmap,
                                                               const __grid_constant__ CUtensorMap wmap,
                                                               ConvTmaParams p) {
  constexpr int A_BYTES = MT * TBM * 128, B_BYTES = BN * 128, STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr int STAGES = stages_of(STAGE_BYTES);
  constexpr int NACC = (2 * MT * BN <= 512) ? 2 : 1;   // accumulator sets in tensor memory
  constexpr int TCOLS = tmem_cols(NACC * MT * BN);
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  constexpr int SQ = 4;   // depth of the tile-index ring
  __shared__ __align__(8) uint64_t bars[2 * STAGES + 4 + 2 * SQ];
  __shared__ uint32_t tmem_slot;
  __shared__ int tile_ring[SQ];   // tile index, or -1: no more tiles
  __shared__ __align__(16) float add_s[2 * MT][BN];
  const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[STAGES]), acc_full = smem_u32(&bars[2 * STAGES]),
                 acc_empty = smem_u32(&bars[2 * STAGES + 2]), sq_full = smem_u32(&bars[2 * STAGES + 4]),
                 sq_empty = smem_u32(&bars[2 * STAGES + 4 + SQ]);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const BoxGeom& g = p.g;
  const int spt = TBM / g.rb;            // boxes per 128-row accumulator
  const int nslot = MT * spt;
  const int64_t total_tiles = (int64_t)p.mtiles * p.ntiles * p.splits;

  // tile -> (first box, first output channel, k-block range)
  auto decode = [&](int64_t tile, int64_t& box0, int& n0, int& kb_begin, int& nkb) {
    const int64_t rest = tile / p.mtiles;
    box0 = (tile - rest * p.mtiles) * nslot;
    const int sp = (int)(rest / p.ntiles);
    n0 = (int)(rest - (int64_t)sp * p.ntiles) * BN;
    kb_begin = sp * p.kb_per_split;
    nkb = min(p.num_kb, kb_begin + p.kb_per_split) - kb_begin;
  };

  // consumer side of the tile ring: the ti-th tile of this CTA (-1 when the sequence has ended)
  auto next_tile = [&](int ti) -> int64_t {
    const int q = ti % SQ;
    mbar_wait(sq_full + 8 * q, (uint32_t)(ti / SQ) & 1u);
    const int t = tile_ring[q];
    mbar_arrive(sq_empty + 8 * q);
    return t;
  };

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full0 + 8 * s, 1);
      mbar_init(empty0 + 8 * s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(acc_full + 8 * a, 1);
      mbar_init(acc_empty + 8 * a, 128 * p.epi_groups);
    }
    for (int a = 0; a < SQ; ++a) {
      mbar_init(sq_full + 8 * a, 1);
      mbar_init(sq_empty + 8 * a, 32 + 128 * p.epi_groups);   // consumers: the UMMA warp and the epilogue threads
    }
    fence_barrier_init();
  }
  if (warp == 4) tmem_alloc<TCOLS>(smem_u32(&tmem_slot));
  if (warp == 5 && lane == 0) { tma_prefetch_desc(&xmap); tma_prefetch_desc(&wmap); }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_acc = tmem_slot;

  if (warp < 4 || (warp >= 6 && p.epi_groups == 2)) {
    // ===================== epilogue: two groups of four warps =====================
    const int eg = warp >= 6 ? 1 : 0;          // column group
    const int egroups = p.epi_groups, ethreads = 128 * egroups;
    const int quad = warp & 3;                 // TMEM lane quadrant this warp may read (warps 6..9 -> 2,3,0,1)
    const int row = quad * 32 + lane;
    const int etid = eg * 128 + row;
    const int r = row & (g.rb - 1), slot = row / g.rb;
    const int lw = r % g.bw, lh = (r / g.bw) % g.bh, ld = r / (g.bw * g.bh);
    int staged_n0 = -1;
    for (int ti = 0;; ++ti) {
      const int64_t tile = next_tile(ti);
      if (tile < 0) break;
      int64_t box0;
      int n0, kb_begin, nkb;
      decode(tile, box0, n0, kb_begin, nkb);
      const int ab = ti % NACC;
      // while the main loop runs: bias + per-sample channel bias of this tile's columns, one row per box (a box lies
      // inside one sample), so that the epilogue adds them with broadcast shared-memory reads. Without a per-sample
      // bias the rows only depend on the column block: staged once, not per tile.
      if (!p.partial && (p.chan_bias != nullptr || n0 != staged_n0)) {
        staged_n0 = n0;
        asm volatile("bar.sync 1, %0;" ::"r"(ethreads) : "memory");   // the previous tile's readers are done with add_s
        for (int j = 0; j < nslot; ++j) {
          int n = 0, d0, h0, w0;
          if (box0 + j < g.num_boxes) box_origin(g, box0 + j, n, d0, h0, w0);
          for (int c = etid; c < BN; c += ethreads) {
            const int col = n0 + c;
            float a = 0.f;
            if (col < g.Cdst) {
              if (p.bias) a += p.bias[col];
              if (p.chan_bias) a += p.chan_bias[(int64_t)n * g.Cdst + col];
            }
            add_s[j][c] = a;
          }
        }
        asm volatile("bar.sync 1, %0;" ::"r"(ethreads) : "memory");
      }
      mbar_wait(acc_full + 8 * ab, (uint32_t)(ti / NACC) & 1u);
      tcgen05_fence_after();
#pragma unroll 1
      for (int mt = 0; mt < MT; ++mt) {
        const int64_t box = box0 + mt * spt + slot;
        const bool bok = box < g.num_boxes;        // warp-uniform: a warp's 32 rows lie in one box
        int n = 0, d0 = 0, h0 = 0, w0 = 0;
        if (bok) box_origin(g, box, n, d0, h0, w0);
        const bool mok = bok && r < g.nb && (d0 + ld < g.D) && (h0 + lh < g.H) && (w0 + lw < g.W);   // boxes may overhang
        const bool st = p.gn_sums != nullptr && bok;
        const int64_t m = (((int64_t)n * g.OD + (d0 + ld) * g.os[0] + g.oo[0]) * g.OH + (h0 + lh) * g.os[1] + g.oo[1]) *
                              g.OW + (w0 + lw) * g.os[2] + g.oo[2];
        const uint32_t trow = tmem_acc + ((uint32_t)(quad * 32) << 16) + ab * (MT * BN) + mt * BN;
        constexpr int LDW = BN >= 64 ? 64 : 16;   // columns per TMEM load (one round trip each)
#pragma unroll 1
        for (int cw = eg * LDW; cw < BN; cw += egroups * LDW) {
          if (n0 + cw >= g.Cdst) break;
          // residual of this row's LDW columns: all 16-byte loads issued up front, in flight during the TMEM load
          // (one dependent global load per 16 columns cost the forward kernels ~6 % against dgrad on the same shape)
          uint4 rres[LDW / 8];
          const bool pre_res = p.residual != nullptr && mok && !p.partial && (g.Cdst & 7) == 0;
          if (pre_res) {
            const uint4* rp = reinterpret_cast<const uint4*>(p.residual + m * g.Cdst + n0 + cw);
#pragma unroll
            for (int e = 0; e < LDW / 8; ++e)
              if (n0 + cw + 8 * e + 8 <= g.Cdst) rres[e] = rp[e];
          }
          float vw[LDW];
          if constexpr (LDW == 64) tmem_ld64(trow + cw, vw);
          else tmem_ld16(trow + cw, vw);
          if (!mok && !st) continue;
          float us[LDW / 8], uq[LDW / 8];   // GroupNorm partials per 8-column unit of this row
#pragma unroll
          for (int u = 0; u < LDW / 8; ++u) us[u] = uq[u] = 0.f;
#pragma unroll
          for (int c0 = cw; c0 < cw + LDW; c0 += 16) {
            if (n0 + c0 >= g.Cdst) break;
            float* v = vw + (c0 - cw);
            const int col0 = n0 + c0;
            if (p.partial) {
              if (mok) red_add_16(p.partial + m * g.Cdst + col0, v, g.Cdst - col0);
              continue;
            }
            const bool full16 = (col0 + 16 <= g.Cdst) && ((g.Cdst & 7) == 0);
            const float4* ap = reinterpret_cast<const float4*>(&add_s[mt * spt + slot][c0]);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float4 b4 = ap[e];
              v[4 * e] += b4.x; v[4 * e + 1] += b4.y; v[4 * e + 2] += b4.z; v[4 * e + 3] += b4.w;
            }
            __nv_bfloat16* dst = p.out + m * g.Cdst + col0;
            if (full16) {
              if (pre_res) {
                const uint4 r0 = rres[(c0 - cw) >> 3], r1 = rres[((c0 - cw) >> 3) + 1];
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
              if (mok) {
                reinterpret_cast<uint4*>(dst)[0] = o0;
                reinterpret_cast<uint4*>(dst)[1] = o1;
              }
              if (st && mok) {   // statistics of what the consumer will read: the ROUNDED values
                const int u = (c0 - cw) >> 3;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float2 f0 = __bfloat1622float2(q0[e]), f1 = __bfloat1622float2(q1[e]);
                  us[u] += f0.x + f0.y;
                  uq[u] = fmaf(f0.x, f0.x, fmaf(f0.y, f0.y, uq[u]));
                  us[u + 1] += f1.x + f1.y;
                  uq[u + 1] = fmaf(f1.x, f1.x, fmaf(f1.y, f1.y, uq[u + 1]));
                }
              }
            } else if (mok) {
#pragma unroll
              for (int e = 0; e < 16; ++e)
                if (col0 + e < g.Cdst) {
                  float rr = p.residual ? __bfloat162float(p.residual[m * g.Cdst + col0 + e]) : 0.f;
                  dst[e] = __float2bfloat16_rn(v[e] + rr);
                }
            }
          }
          if constexpr (LDW == 64) {
            if (st) {
              // 32 columns at a time: at most four groups (cpg >= 8) -> one 8-value warp reduction, 8 fp64 atomics
#pragma unroll
              for (int hf = 0; hf < 2; ++hf) {
                const int cbase = n0 + cw + 32 * hf;
                if (cbase >= g.Cdst) break;
                const int gfirst = cbase / p.gn_cpg;
                float acc[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) acc[i] = 0.f;
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  const int slot = (cbase + 8 * u) / p.gn_cpg - gfirst;
#pragma unroll
                  for (int sl = 0; sl < 4; ++sl)
                    if (slot == sl) { acc[2 * sl] += us[4 * hf + u]; acc[2 * sl + 1] += uq[4 * hf + u]; }
                }
                const float tot = warp_sum8(acc, lane);
                const int idx = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
                const int grp = gfirst + (idx >> 1);
                const int cend = cbase + 32 < g.Cdst ? cbase + 32 : g.Cdst;
                if ((lane & 3) == 0 && grp < p.gn_G && grp * p.gn_cpg < cend)
                  atomicAdd(p.gn_sums + ((int64_t)n * p.gn_G + grp) * 2 + (idx & 1), (double)tot);
              }
            }
          }
        }
      }
      tcgen05_fence_before();
      mbar_arrive(acc_empty + 8 * ab);   // this accumulator set may be overwritten by a later tile
    }
  } else if (warp >= 6) {
    // second epilogue group switched off
  } else if (warp == 4) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc = make_idesc(TBM, BN, 0, BMN ? 1 : 0);
    int s = 0;
    uint32_t ph = 0;
    for (int ti = 0;; ++ti) {
      const int64_t tile = next_tile(ti);
      if (tile < 0) break;
      int64_t box0;
      int n0, kb_begin, nkb;
      decode(tile, box0, n0, kb_begin, nkb);
      const int ab = ti % NACC;
      mbar_wait(acc_empty + 8 * ab, ((uint32_t)(ti / NACC) & 1u) ^ 1u);   // epilogue has drained this accumulator set
      tcgen05_fence_after();
      const uint32_t acc = tmem_acc + ab * (MT * BN);
      for (int it = 0; it < nkb; ++it) {
        mbar_wait(full0 + 8 * s, ph);
        tcgen05_fence_after();
        if (elect_one()) {
          const uint32_t a_smem = smem_base + s * STAGE_BYTES, b_smem = a_smem + A_BYTES;
#pragma unroll
          for (int kk = 0; kk < TBK / 16; ++kk) {
            const uint64_t bd = BMN ? make_smem_desc(b_smem + kk * 2048, PANEL, 1024)   // 16 K rows of every 64-column panel
                                    : make_smem_desc(b_smem + kk * 32, 16, 1024);
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
              umma_bf16(acc + mt * BN, make_smem_desc(a_smem + mt * (TBM * 128) + kk * 32, 16, 1024), bd, idesc,
                        (it | kk) ? 1u : 0u);
          }
          umma_commit(empty0 + 8 * s);
          if (it == nkb - 1) umma_commit(acc_full + 8 * ab);
        }
        __syncwarp();
        if (++s == STAGES) { s = 0; ph ^= 1u; }
      }
    }
  } else {
    // ============ TMA issuer: ONE elected thread, all address arithmetic warp-uniform ============
    // (The earlier one-lane-per-box scheme made ptxas wrap every UTMALDG in a divergence "waterfall" loop and redid the
    // tap / box index divisions every stage; this thread is the producer's critical path, so the k-block -> (tap,
    // channel chunk) mapping is an odometer and the box origins are computed once per tile.)
    if (elect_one()) {
      const uint32_t tx_bytes = (uint32_t)(nslot * g.nb) * 128u + B_BYTES;   // a box transfers its nb rows (zero-filled when out of bounds)
      const uint32_t slot_bytes = (uint32_t)g.rb * 128u;
      int s = 0;
      uint32_t ph = 0;
      int64_t tile = blockIdx.x;
      for (int ti = 0;; ++ti) {
        // publish the ti-th tile of this CTA (or the end marker) to the UMMA warp and the epilogue threads
        const bool more = tile < total_tiles;
        const int q = ti % SQ;
        mbar_wait(sq_empty + 8 * q, ((uint32_t)(ti / SQ) & 1u) ^ 1u);
        tile_ring[q] = more ? (int)tile : -1;
        mbar_arrive(sq_full + 8 * q);
        if (!more) break;
        // draw the next index now: the atomic's round trip hides behind this tile's loads
        unsigned int drawn = 0;
        if (p.sched) drawn = atomicAdd(&p.sched->next, 1u);
        int64_t box0;
        int n0, kb_begin, nkb;
        decode(tile, box0, n0, kb_begin, nkb);
        int bn_[2 * MT], bd_[2 * MT], bh_[2 * MT], bw_[2 * MT];
#pragma unroll
        for (int j = 0; j < 2 * MT; ++j) {
          bn_[j] = g.N; bd_[j] = 0; bh_[j] = 0; bw_[j] = 0;   // default: fully out of bounds -> zero rows (tile tail)
          if (j < nslot && box0 + j < g.num_boxes) box_origin(g, box0 + j, bn_[j], bd_[j], bh_[j], bw_[j]);
        }
        int tap = kb_begin / g.cchunks;
        int cch = kb_begin - tap * g.cchunks;
        int kcol = tap * g.Csrc;   // filter column of (tap, channel 0)
        int tapi = tap;            // linear tap index (BMN: coordinate 1 of the 3-d filter map)
        int t2 = tap % g.ks[2]; tap /= g.ks[2];
        int t1 = tap % g.ks[1];
        int t0 = tap / g.ks[1];
        for (int it = 0; it < nkb; ++it) {
          const uint32_t a_smem = smem_base + s * STAGE_BYTES, b_smem = a_smem + A_BYTES, bar = full0 + 8 * s;
          mbar_wait(empty0 + 8 * s, ph ^ 1u);
          mbar_arrive_expect_tx(bar, tx_bytes);
          const int dz = t0 * g.sign + g.off[0], dy = t1 * g.sign + g.off[1], dx = t2 * g.sign + g.off[2];
          const int c0 = cch * 64;
#pragma unroll
          for (int j = 0; j < 2 * MT; ++j)
            if (j < nslot)
              tma_load_5d(a_smem + j * slot_bytes, &xmap, bar, c0, bw_[j] * g.ss[2] + dx, bh_[j] * g.ss[1] + dy,
                          bd_[j] * g.ss[0] + dz, bn_[j]);
          if constexpr (BMN) {
#pragma unroll
            for (int q = 0; q < BN / 64; ++q)   // panels past Cdst are out of bounds -> zero-filled, byte count unchanged
              tma_load_3d(b_smem + q * PANEL, &wmap, bar, n0 + q * 64, tapi, c0);
          } else {
            tma_load_2d(b_smem, &wmap, bar, kcol + c0, n0);
          }
          if (++cch == g.cchunks) {
            cch = 0;
            kcol += g.Csrc;
            ++tapi;
            if (++t2 == g.ks[2]) { t2 = 0; if (++t1 == g.ks[1]) { t1 = 0; ++t0; } }
          }
          if (++s == STAGES) { s = 0; ph ^= 1u; }
        }
        tile = p.sched ? (int64_t)gridDim.x + drawn : tile + gridDim.x;
      }
      if (p.sched) {   // the last CTA to get here re-arms the counter for the next launch / graph replay
        __threadfence();
        if (atomicAdd(&p.sched->done, 1u) == gridDim.x - 1) {
          p.sched->next = 0;
          p.sched->done = 0;
          __threadfence();
        }
      }
    }
  }
  __syncthreads();
  if (warp == 4) {
    tcgen05_fence_after();
    tmem_dealloc<TCOLS>(tmem_acc);
  }
}

// split-K finish: out = bf16(partial + bias + chan_bias + residual); `partial` is indexed by plain voxel index
__global__ void __launch_bounds__(256) tma_splitk_finish(const float* __restrict__ partial, const float* __restrict__ bias,
                                                         const float* __restrict__ chan_bias,
                                                         const __nv_bfloat16* __restrict__ residual,
                                                         __nv_bfloat16* __restrict__ out, int64_t M, int C, int64_t Mo) {
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
// the same, 8 channels per thread (C % 8 == 0, all pointers 16-byte aligned)
__global__ void __launch_bounds__(256) tma_splitk_finish8(const float* __restrict__ partial, const float* __restrict__ bias,
                                                          const float* __restrict__ chan_bias,
                                                          const __nv_bfloat16* __restrict__ residual,
                                                          __nv_bfloat16* __restrict__ out, int64_t M, int C, int64_t Mo) {
  const int C8 = C >> 3;
  const int64_t total = M * C8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = i / C8;
    const int c = (int)(i - m * C8) * 8;
    const float4* pp = reinterpret_cast<const float4*>(partial + i * 8);
    float4 a = pp[0], b = pp[1];
    float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    if (bias) {
      const float4* q = reinterpret_cast<const float4*>(bias + c);
      a = q[0]; b = q[1];
      v[0] += a.x; v[1] += a.y; v[2] += a.z; v[3] += a.w; v[4] += b.x; v[5] += b.y; v[6] += b.z; v[7] += b.w;
    }
    if (chan_bias) {
      const float4* q = reinterpret_cast<const float4*>(chan_bias + (m / Mo) * C + c);
      a = q[0]; b = q[1];
      v[0] += a.x; v[1] += a.y; v[2] += a.z; v[3] += a.w; v[4] += b.x; v[5] += b.y; v[6] += b.z; v[7] += b.w;
    }
    if (residual) {
      const uint4 r = *reinterpret_cast<const uint4*>(residual + i * 8);
      const __nv_bfloat16* rb = reinterpret_cast<const __nv_bfloat16*>(&r);
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] += __bfloat162float(rb[e]);
    }
    uint4 o;
    __nv_bfloat162* q = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
    for (int e = 0; e < 4; ++e) q[e] = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
    *reinterpret_cast<uint4*>(out + i * 8) = o;
  }
}

// ---------------------------------------------------------------------------------------------------
// wgrad
// ---------------------------------------------------------------------------------------------------
struct WgradTmaParams {
  BoxGeom g;        // rows = conv OUTPUT voxels (dY); source = X; sign +1, off = -pad; Csrc = Cin, Cdst = Cout
  float* dw;
  int64_t boxes_per_split;
};

// CTA tile: MT*128 output channels x BN filter columns; reduction over voxel boxes
template <int BN, int MT>
__global__ void __launch_bounds__(kThreads, 1) wgrad_tma_kernel(const __grid_constant__ CUtensorMap dymap,
                                                                const __grid_constant__ CUtensorMap xmap,
                                                                WgradTmaParams p) {
  constexpr int NPAN = BN / 64, APAN = 2 * MT;
  constexpr int A_BYTES = APAN * PANEL, B_BYTES = NPAN * PANEL, STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr int STAGES = stages_of(STAGE_BYTES);
  constexpr int TCOLS = tmem_cols(MT * BN);
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  __shared__ __align__(8) uint64_t bars[2 * STAGES + 1];
  __shared__ uint32_t tmem_slot;
  const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[STAGES]), accbar = smem_u32(&bars[2 * STAGES]);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const BoxGeom& g = p.g;
  const int co0 = blockIdx.x * (TBM * MT);
  const int n0 = blockIdx.y * BN;     // column offset in K = tap*Cin + ci
  const int64_t bb = (int64_t)blockIdx.z * p.boxes_per_split;
  const int nst = (int)(min(g.num_boxes, bb + p.boxes_per_split) - bb);

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full0 + 8 * s, 1);
      mbar_init(empty0 + 8 * s, 1);
    }
    mbar_init(accbar, 1);
    fence_barrier_init();
  }
  if (warp == 4) tmem_alloc<TCOLS>(smem_u32(&tmem_slot));
  if (warp == 5 && lane == 0) { tma_prefetch_desc(&dymap); tma_prefetch_desc(&xmap); }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_acc = tmem_slot;

  if (warp < 4) {
    mbar_wait(accbar, 0);
    tcgen05_fence_after();
#pragma unroll 1
    for (int mt = 0; mt < MT; ++mt) {
      const int co = co0 + mt * TBM + warp * 32 + lane;
      const bool cok = co < g.Cdst && nst > 0;
      const uint32_t trow = tmem_acc + ((uint32_t)(warp * 32) << 16) + mt * BN;
#pragma unroll 1
      for (int cw = 0; cw < BN; cw += 64) {
        if (n0 + cw >= g.K) break;
        float vw[64];
        tmem_ld64(trow + cw, vw);
        if (!cok) continue;
#pragma unroll
        for (int c0 = cw; c0 < cw + 64; c0 += 16) {
          if (n0 + c0 >= g.K) break;
          red_add_16(p.dw + (int64_t)co * g.K + n0 + c0, vw + (c0 - cw), g.K - n0 - c0);
        }
      }
    }
    tcgen05_fence_before();
  } else if (warp == 4) {
    constexpr uint32_t idesc = make_idesc(TBM, BN, 1, 1);
    for (int it = 0; it < nst; ++it) {
      const int s = it % STAGES;
      mbar_wait(full0 + 8 * s, (uint32_t)(it / STAGES) & 1u);
      tcgen05_fence_after();
      if (elect_one()) {
        const uint32_t a_smem = smem_base + s * STAGE_BYTES, b_smem = a_smem + A_BYTES;
#pragma unroll
        for (int kk = 0; kk < TBK / 16; ++kk) {
          if (kk * 16 >= g.nb) break;   // boxes of 16/32/48 voxels use the first rows of each 64-row panel
          const uint64_t bd = make_smem_desc(b_smem + kk * 2048, PANEL, 1024);
#pragma unroll
          for (int mt = 0; mt < MT; ++mt)
            umma_bf16(tmem_acc + mt * BN, make_smem_desc(a_smem + mt * 2 * PANEL + kk * 2048, PANEL, 1024), bd, idesc,
                      (it | kk) ? 1u : 0u);
        }
        umma_commit(empty0 + 8 * s);
        if (it == nst - 1) umma_commit(accbar);
      }
      __syncwarp();
    }
    if (nst <= 0 && lane == 0) mbar_arrive(accbar);
  } else {
    // TMA issuer: one elected thread, warp-uniform arithmetic (see the forward kernel). Each im2col(X) panel is one
    // fixed (tap, 64-channel chunk) for the whole kernel; the voxel box walks the volume as an odometer.
    if (elect_one()) {
      int dz[NPAN], dy[NPAN], dx[NPAN], cc[NPAN];
#pragma unroll
      for (int q = 0; q < NPAN; ++q) {
        const int k = n0 + q * 64;
        int tap = k / g.Csrc;
        cc[q] = k < g.K ? k - tap * g.Csrc : -1;
        const int t2 = tap % g.ks[2]; tap /= g.ks[2];
        const int t1 = tap % g.ks[1];
        const int t0 = tap / g.ks[1];
        dz[q] = t0 + g.off[0]; dy[q] = t1 + g.off[1]; dx[q] = t2 + g.off[2];
      }
      int n = 0, d0 = 0, h0 = 0, w0 = 0;
      if (nst > 0) box_origin(g, bb, n, d0, h0, w0);
      const int wend = g.nbw * g.bw, hend = g.nbh * g.bh, dend = g.nbd * g.bd;
      const uint32_t tx_bytes = (uint32_t)((APAN + NPAN) * g.nb) * 128u;
      for (int it = 0; it < nst; ++it) {
        const int s = it % STAGES;
        const uint32_t a_smem = smem_base + s * STAGE_BYTES, b_smem = a_smem + A_BYTES, bar = full0 + 8 * s;
        mbar_wait(empty0 + 8 * s, ((uint32_t)(it / STAGES) & 1u) ^ 1u);
        mbar_arrive_expect_tx(bar, tx_bytes);
#pragma unroll
        for (int a = 0; a < APAN; ++a) tma_load_5d(a_smem + a * PANEL, &dymap, bar, co0 + a * 64, w0, h0, d0, n);
#pragma unroll
        for (int q = 0; q < NPAN; ++q) {
          if (cc[q] >= 0)
            tma_load_5d(b_smem + q * PANEL, &xmap, bar, cc[q], w0 * g.ss[2] + dx[q], h0 * g.ss[1] + dy[q], d0 * g.ss[0] + dz[q], n);
          // a panel past the end of K is loaded fully out of bounds (n = N) -> zeros, keeps the byte count fixed
          else tma_load_5d(b_smem + q * PANEL, &xmap, bar, 0, 0, 0, 0, g.N);
        }
        w0 += g.bw;
        if (w0 >= wend) {
          w0 = 0; h0 += g.bh;
          if (h0 >= hend) { h0 = 0; d0 += g.bd; if (d0 >= dend) { d0 = 0; ++n; } }
        }
      }
    }
  }
  __syncthreads();
  if (warp == 4) {
    tcgen05_fence_after();
    tmem_dealloc<TCOLS>(tmem_acc);
  }
}

// ---------------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------------
// boxes per axis, their product, and the multiply-high constants of the divisions box_origin performs
// (q = umulhi(x, mul) >> shr for x < 2^31: mul = ceil(2^(31 + ceil(log2 d)) / d), shr = ceil(log2 d) - 1)
static void set_box_counts(BoxGeom& b) {
  b.nbd = (b.D + b.bd - 1) / b.bd; b.nbh = (b.H + b.bh - 1) / b.bh; b.nbw = (b.W + b.bw - 1) / b.bw;
  b.num_boxes = (int64_t)b.N * b.nbd * b.nbh * b.nbw;
  const int div[3] = {b.nbw, b.nbh, b.nbd};
  for (int i = 0; i < 3; ++i) {
    const uint32_t d = (uint32_t)div[i];
    b.dmul[i] = 0; b.dshr[i] = 0;
    if (d <= 1) continue;
    int lg = 0;
    while ((1u << lg) < d) ++lg;   // ceil(log2 d)
    const int pw = 31 + lg;
    b.dmul[i] = (uint32_t)((((uint64_t)1 << pw) + d - 1) / d);
    b.dshr[i] = (uint32_t)(pw - 32);
  }
}

static bool pick_box(int D, int H, int W, int* bd, int* bh, int* bw) {
  // 64 voxels per box, power-of-two factors; prefer wide W (contiguous rows in memory)
  static const int cand[][3] = {{1, 8, 8}, {2, 4, 8}, {4, 2, 8}, {8, 1, 8}, {1, 4, 16}, {2, 2, 16}, {4, 1, 16},
                                {4, 4, 4}, {2, 8, 4}, {8, 2, 4}, {1, 16, 4}, {16, 1, 4}, {1, 2, 32}, {2, 1, 32},
                                {1, 1, 64}, {8, 4, 2}, {4, 8, 2}, {16, 2, 2}, {2, 16, 2}, {8, 8, 1}, {16, 4, 1},
                                {4, 16, 1}};
  // Boxes may overhang the tensor (TMA zero-fills out-of-bounds voxels, the epilogue masks them): pick the shape
  // that wastes the fewest rows; exact tilings (efficiency 1) win, e.g. 24^3 -> 1x8x8, 12^3 -> 4x4x4. On a tie the
  // earlier candidate wins: 6^3 -> 1x8x8 (2x4x8 wastes as many rows).
  double best = 0.0;
  for (auto& c : cand) {
    const double cover = (double)((D + c[0] - 1) / c[0] * c[0]) * ((H + c[1] - 1) / c[1] * c[1]) *
                         ((W + c[2] - 1) / c[2] * c[2]);
    const double eff = (double)D * H * W / cover;
    if (eff > best + 1e-9) {
      best = eff;
      *bd = c[0]; *bh = c[1]; *bw = c[2];
    }
  }
  return best >= 0.5;   // below that the cp.async gather kernels are the better choice
}

// wgrad: a box is one K stage, so its voxel count only has to be a multiple of 16 (the UMMA K). Besides the 64-voxel
// shapes, 48/32/16-voxel boxes are tried for volumes the 64-voxel boxes tile badly (6^3: 2x4x6 boxes, 75 % instead of
// 56 % useful rows); smaller stages pay relatively more per-stage overhead, hence the discount.
static bool pick_box_k(int D, int H, int W, int* bd, int* bh, int* bw) {
  bool ok = pick_box(D, H, W, bd, bh, bw);
  double best = 0.0;
  if (ok) {
    const double cover = (double)((D + *bd - 1) / *bd * *bd) * ((H + *bh - 1) / *bh * *bh) * ((W + *bw - 1) / *bw * *bw);
    best = (double)D * H * W / cover;
  }
  if (best >= 0.8) return true;
  double best_s = best * 64.0 / 72.0;
  for (int d = 1; d <= D && d <= 64; ++d)
    for (int h = 1; h <= H && d * h <= 64; ++h)
      for (int w = 1; w <= W && d * h * w <= 64; ++w) {
        const int nb = d * h * w;
        if (nb % 16 != 0) continue;
        const double boxes = (double)((D + d - 1) / d) * ((H + h - 1) / h) * ((W + w - 1) / w);
        const double sc = (double)D * H * W / (boxes * nb) * nb / (nb + 8.0);
        if (sc > best_s + 0.05) { best_s = sc; *bd = d; *bh = h; *bw = w; ok = true; }
      }
  return ok && best_s * 72.0 / 64.0 >= 0.5;
}

// fwd / dgrad only: a box may also fill one whole 128-row slot with FEWER than 128 voxels (the unused rows compute
// garbage accumulator rows that the epilogue never reads), which tiles small odd volumes much better than overhanging
// 64-voxel boxes: 6^3 -> two 3x6x6 boxes per sample (84 % useful rows instead of 56 %).
static bool pick_box_rows(int D, int H, int W, int* bd, int* bh, int* bw, int* rb) {
  *rb = 64;
  double best = 0.0;
  bool ok = pick_box(D, H, W, bd, bh, bw);
  if (ok) {
    const double cover = (double)((D + *bd - 1) / *bd * *bd) * ((H + *bh - 1) / *bh * *bh) * ((W + *bw - 1) / *bw * *bw);
    best = (double)D * H * W / cover;
  }
  if (best >= 0.8) return true;
  double best128 = 0.0;
  int c[3] = {0, 0, 0};
  for (int d = 1; d <= D && d <= 128; ++d)
    for (int h = 1; h <= H && d * h <= 128; ++h)
      for (int w = 1; w <= W && d * h * w <= 128; ++w) {
        const double boxes = (double)((D + d - 1) / d) * ((H + h - 1) / h) * ((W + w - 1) / w);
        const double eff = (double)D * H * W / (boxes * 128.0);
        if (eff > best128 + 1e-9 || (eff > best128 - 1e-9 && w > c[2])) { best128 = eff; c[0] = d; c[1] = h; c[2] = w; }
      }
  if (best128 > best + 0.1) {
    *bd = c[0]; *bh = c[1]; *bw = c[2]; *rb = 128;
    return best128 >= 0.5;
  }
  return ok;
}

// which: 0 fwd, 1 dgrad, 2 wgrad
bool tma_conv_eligible(const mig_conv_geom* g, int which) {
  bool strided = false;
  for (int i = 0; i < 3; ++i) {
    if (g->stride[i] < 1 || g->stride[i] > 2) return false;
    strided = strided || g->stride[i] != 1;
  }
  if (strided && which == 1) return false;   // strided dgrad: stride-residue classes (tma_conv_dgrad_strided)
  const int csrc = which == 1 ? g->Cout : g->Cin;
  // wgrad panels must not straddle taps; a strided forward conv takes 32 channels too (half-empty chunk, still far
  // ahead of the gather kernel)
  if (which == 2 ? csrc % 64 != 0 : (csrc % 8 != 0 || csrc < (strided ? 32 : 48))) return false;
  if (which == 2 && g->Cout % 8 != 0) return false;
  const int32_t* dims = which == 1 ? g->in_dims : g->out_dims;
  // box indices are 31-bit in the kernels (fast_div); a box holds at least 16 voxels
  if ((double)g->N * dims[0] * dims[1] * dims[2] > 16.0 * 2147483647.0) return false;
  int bd, bh, bw, rb;
  if (which != 2) return pick_box_rows(dims[0], dims[1], dims[2], &bd, &bh, &bw, &rb);
  return pick_box_k(dims[0], dims[1], dims[2], &bd, &bh, &bw);
}

static int make_act_map(CUtensorMap* m, const void* base, int N, const int32_t dims[3], int C, int bd, int bh, int bw,
                        const int* estride = nullptr) {
  // 5-d (C, W, H, D, N) with a 64-channel x box window
  const uint64_t gd[5] = {(uint64_t)C, (uint64_t)dims[2], (uint64_t)dims[1], (uint64_t)dims[0], (uint64_t)N};
  const uint64_t gs[4] = {(uint64_t)C * 2, (uint64_t)dims[2] * C * 2, (uint64_t)dims[1] * dims[2] * C * 2,
                          (uint64_t)dims[0] * dims[1] * dims[2] * C * 2};
  // With an element stride s the box SPANS bw*s tensor elements and delivers every s-th one: bw voxels reach shared
  // memory, exactly the source voxels of bw consecutive outputs of a stride-s convolution.
  const int sd = estride ? estride[0] : 1, sh = estride ? estride[1] : 1, sw = estride ? estride[2] : 1;
  const uint32_t bx[5] = {64, (uint32_t)(bw * sw), (uint32_t)(bh * sh), (uint32_t)(bd * sd), 1};
  const uint32_t es[5] = {1, (uint32_t)sw, (uint32_t)sh, (uint32_t)sd, 1};
  MIG_REQUIRE(bx[1] <= 256 && bx[2] <= 256 && bx[3] <= 256, "conv_tma: strided box exceeds the TMA box limit");
  return make_map(m, base, 5, gd, gs, bx, "conv_tma activation map", CU_TENSOR_MAP_SWIZZLE_128B, es);
}

enum BoxPicker { kBox64, kBoxRows, kBoxStage };   // pick_box, pick_box_rows (fwd / dgrad), pick_box_k (wgrad)

// One box-conv problem: rows over ext[] (N samples), source coordinate = row*ss + tap*sign + off over ks[] taps, and
// row j lands at j*os + oo inside out[]. Returns whether the picker found a box worth using.
static bool box_geom(BoxGeom& b, BoxPicker pick, int N, const int ext[3], const int ks[3], const int off[3], int sign,
                     const int ss[3], const int os[3], const int oo[3], const int out[3], int Csrc, int Cdst) {
  b = BoxGeom{};
  b.N = N; b.D = ext[0]; b.H = ext[1]; b.W = ext[2];
  b.rb = 64;
  const bool ok = pick == kBoxRows    ? pick_box_rows(b.D, b.H, b.W, &b.bd, &b.bh, &b.bw, &b.rb)
                  : pick == kBoxStage ? pick_box_k(b.D, b.H, b.W, &b.bd, &b.bh, &b.bw)
                                      : pick_box(b.D, b.H, b.W, &b.bd, &b.bh, &b.bw);
  b.nb = b.bd * b.bh * b.bw;
  set_box_counts(b);
  int taps = 1;
  for (int i = 0; i < 3; ++i) {
    b.ks[i] = ks[i]; b.off[i] = off[i]; b.ss[i] = ss[i]; b.os[i] = os[i]; b.oo[i] = oo[i];
    taps *= ks[i];
  }
  b.sign = sign;
  b.Csrc = Csrc; b.Cdst = Cdst;
  b.K = taps * Csrc;
  b.cchunks = (Csrc + 63) / 64;
  b.OD = out[0]; b.OH = out[1]; b.OW = out[2];
  return ok;
}

static const int kOnes[3] = {1, 1, 1}, kZeros[3] = {0, 0, 0};

// which: 0 fwd, 1 dgrad, 2 wgrad of a convolution; rows are the tensor being produced (wgrad: the conv output)
static BoxGeom make_box_geom(const mig_conv_geom* g, int which) {
  const int32_t* rows = which == 1 ? g->in_dims : g->out_dims;
  int off[3];
  for (int i = 0; i < 3; ++i) off[i] = which == 1 ? g->pad[i] : -g->pad[i];
  BoxGeom b;
  box_geom(b, which == 2 ? kBoxStage : kBoxRows, g->N, rows, g->ksize, off, which == 1 ? -1 : 1,
           which == 1 ? kOnes : g->stride, kOnes, kZeros, rows, which == 1 ? g->Cout : g->Cin,
           which == 1 ? g->Cin : g->Cout);
  return b;
}

template <int BN, int MT, bool BMN = false>
static int launch_conv_tma(const CUtensorMap& xm, const CUtensorMap& wm, const ConvTmaParams& p, dim3 grid,
                           cudaStream_t st) {
  constexpr int stage = MT * TBM * 128 + BN * 128;
  constexpr int smem = stages_of(stage) * stage + 1024;
  static SmemOptIn optin;
  if (int rc = ensure_dynamic_smem(conv_tma_kernel<BN, MT, BMN>, smem, optin, "conv_tma")) return rc;
  conv_tma_kernel<BN, MT, BMN><<<grid, kConvThreads, smem, st>>>(xm, wm, p);
  return check_launch("conv_tma_kernel");
}

// Optional extras of a launch: GroupNorm statistics of the output (forward) and the MN-major filter operand (dgrad on
// the untransposed filter).
struct BoxExtras {
  double* gn_sums = nullptr;   // [N][G][2], accumulated into (caller zeroes)
  int gn_groups = 0;
  bool stats_done = false;     // out: the epilogue produced the statistics (false: split-K plan, caller falls back)
  bool bmn = false;            // filter is [Csrc][taps][Cdst] (the forward layout seen from dgrad)
};

static int launch_box_conv(const BoxGeom& b, int N, const int32_t* sdims, const void* src, const void* wk,
                           const float* bias, const float* chan_bias, const void* residual, void* out, void* ws,
                           int64_t ws_bytes, void* stream, BoxExtras* ex = nullptr);

// Tile / split-K plan from a small cost model (cycles): a stage costs the larger of its UMMA time and its operand
// fill time (ncu: the L2 -> SM path sustains ~60-85 B/clk/SM); a CTA adds a fixed launch / pipeline-fill / drain cost
// (ncu on 64-channel layers: ~15 k cycles around a 3.5 k-cycle main loop, which is why narrow layers also get
// 256-row tiles); the grid runs in ceil(CTAs / SMs) waves; split-K fills the chip on the small deep levels.
// Split-K needs an fp32 [M][Cdst] workspace: ws_bytes is what the launch has (0: none, as for the class launches).
struct BoxPlan {
  int bn, mt;              // output-channel tile, stacked 128-row accumulators
  int num_kb;              // k-blocks: taps x 64-channel chunks
  int splits, kb_per_split;
};
static BoxPlan plan_box(const BoxGeom& b, int64_t ws_bytes) {
  const int sms = device_info().sm_count;
  BoxPlan pl;
  pl.bn = pick_bn(b.Cdst);
  pl.num_kb = (b.K / b.Csrc) * b.cchunks;
  const int bn = pl.bn, num_kb = pl.num_kb;
  const int64_t ntiles = (b.Cdst + bn - 1) / bn;
  const int64_t M = (int64_t)b.N * b.D * b.H * b.W;
  const bool ws_ok = ws_bytes >= M * b.Cdst * 4;
  double best = 1e30;
  static const int cand_s[] = {1, 2, 3, 4, 6, 8, 12, 16};
  pl.mt = 1; pl.splits = 1;
  for (int m_ = 1; m_ <= 2; ++m_) {
    const int nslot_ = m_ * (TBM / b.rb);
    const int64_t mtiles_ = (b.num_boxes + nslot_ - 1) / nslot_;
    const double t_stage = fmax(512.0 * m_ * bn / 256.0, ((double)nslot_ * b.nb + bn) * 128.0 / 70.0);
    for (int s_ : cand_s) {
      if (s_ > 1 && (!ws_ok || num_kb / s_ < 4)) continue;
      const double waves = (double)((mtiles_ * ntiles * s_ + sms - 1) / sms);
      const double kb = (double)((num_kb + s_ - 1) / s_);
      const double t_epi = 2500.0 + m_ * (bn / 16) * (s_ > 1 ? 160.0 : 110.0);
      double t = waves * (kb * t_stage + t_epi + 9000.0);
      if (s_ > 1) t += (double)M * b.Cdst * 14.0 / 3000.0 + 8000.0;   // memset + fp32 reductions + finish pass
      if (t < best) { best = t; pl.mt = m_; pl.splits = s_; }
    }
  }
  pl.kb_per_split = (num_kb + pl.splits - 1) / pl.splits;
  pl.splits = (num_kb + pl.kb_per_split - 1) / pl.kb_per_split;
  return pl;
}

// One TileCounter per launch out of a per-device pool, handed out round-robin: launches in flight (and the kernel nodes
// of a captured graph) never share a slot unless more than kTileSlots convolutions are in flight at once. The pool is
// allocated on first use; if that first use happens inside a stream capture (no allocation allowed) the launch keeps the
// static schedule.
// OFF by default (MIG_CONV_SCHED=dynamic switches it on). Measured on 2 B200s, same box, back to back
// (bench.py --gpus 2, sharded optimiser): in the eager instrumented steps the dynamic schedule does what it was built for
// (dgrad 1105 -> 1145 TFLOP/s while reduce-scatter kernels hold SMs, step 42.1 -> 41.7 ms), but the CUDA-graph step --
// the one that is timed and shipped -- is 2 % SLOWER with it (39.7 / 39.8 vs 38.9 ms); at N = 1 it is neutral
// (36.9 vs 36.8 ms). The static round-robin therefore stays the default.
static TileCounter* next_tile_counter(cudaStream_t st) {
  constexpr unsigned kTileSlots = 2048;
  static std::mutex mu;
  static TileCounter* pool[16] = {};
  static unsigned cursor[16] = {};
  static int mode = -1;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return nullptr;
  std::lock_guard<std::mutex> lk(mu);
  if (mode < 0) {
    const char* e = getenv("MIG_CONV_SCHED");
    mode = (e && e[0] == 'd') ? 1 : 0;
  }
  if (!mode) return nullptr;
  if (!pool[dev]) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) {
      cudaGetLastError();
      return nullptr;
    }
    TileCounter* ptr = nullptr;
    if (cudaMalloc(&ptr, kTileSlots * sizeof(TileCounter)) != cudaSuccess ||
        cudaMemset(ptr, 0, kTileSlots * sizeof(TileCounter)) != cudaSuccess) {
      cudaGetLastError();
      return nullptr;
    }
    pool[dev] = ptr;
  }
  return pool[dev] + (cursor[dev]++ % kTileSlots);
}

// The epilogue can only deliver the statistics when it sees final values (no split-K) and whole 8-channel units of one
// group. It is USED when it is free: with two accumulator sets in tensor memory (2*MT*BN <= 512 columns) the epilogue of
// tile i overlaps the main loop of tile i+1. For the 256 x 256 tile the epilogue is exposed, and measured on the
// config-3 step the extra reduction work cost 0.8 ms of convolution time per step to save 0.16 ms of (L2-resident)
// statistics passes -- there the separate pass is the faster design. MIG_GN_EPILOGUE=always / never overrides (tests).
static bool epilogue_stats_ok(const BoxGeom& b, const BoxPlan& pl, int groups) {
  if (!(pl.splits == 1 && pl.bn >= 64 && b.Cdst % 16 == 0 && groups > 0 && b.Cdst % groups == 0 &&
        (b.Cdst / groups) % 8 == 0))
    return false;
  const char* e = getenv("MIG_GN_EPILOGUE");
  if (e && e[0] == 'a') return true;
  if (e && e[0] == 'n') return false;
  return 2 * pl.mt * pl.bn <= 512;
}

// src: activation being convolved (x for fwd, dy for dgrad); wk: filter as [Cdst][taps][Csrc] (or, with ex->bmn, as
// [Csrc][taps][Cdst])
static int run_conv_tma(const mig_conv_geom* g, int which, const void* src, const void* wk, const float* bias,
                        const float* chan_bias, const void* residual, void* out, void* ws, int64_t ws_bytes,
                        void* stream, BoxExtras* ex = nullptr) {
  BoxGeom b = make_box_geom(g, which);
  const int32_t* sdims = which == 1 ? g->out_dims : g->in_dims;   // extent of the SOURCE tensor
  return launch_box_conv(b, g->N, sdims, src, wk, bias, chan_bias, residual, out, ws, ws_bytes, stream, ex);
}

// Launch the kernel for a prepared geometry. Split-K (needs `ws`) is only legal when rows map 1:1 to the output.
static int launch_box_conv(const BoxGeom& b, int N, const int32_t* sdims, const void* src, const void* wk,
                           const float* bias, const float* chan_bias, const void* residual, void* out, void* ws,
                           int64_t ws_bytes, void* stream, BoxExtras* ex) {
  cudaStream_t st = as_stream(stream);
  CUtensorMap xm, wm;
  if (make_act_map(&xm, src, N, sdims, b.Csrc, b.bd, b.bh, b.bw, b.ss)) return 1;
  const BoxPlan pl = plan_box(b, ws ? ws_bytes : 0);
  const int bn = pl.bn, mt = pl.mt, splits = pl.splits;
  const bool bmn = ex && ex->bmn;
  if (bmn) {
    MIG_REQUIRE(bn >= 64, "conv_tma: the MN-major filter operand needs at least 64 output channels");
    const int T = b.K / b.Csrc;
    uint64_t dims[3] = {(uint64_t)b.Cdst, (uint64_t)T, (uint64_t)b.Csrc};
    uint64_t strides[2] = {(uint64_t)b.Cdst * 2, (uint64_t)T * b.Cdst * 2};
    uint32_t box[3] = {64, 1, 64};
    if (make_map(&wm, wk, 3, dims, strides, box)) return 1;
  } else {
    uint64_t dims[2] = {(uint64_t)b.K, (uint64_t)b.Cdst};
    uint64_t strides[1] = {(uint64_t)b.K * 2};
    uint32_t box[2] = {TBK, (uint32_t)bn};
    if (make_map(&wm, wk, 2, dims, strides, box)) return 1;
  }
  ConvTmaParams p{};
  p.g = b;
  p.bias = bias; p.chan_bias = chan_bias;
  p.residual = (const __nv_bfloat16*)residual;
  p.out = (__nv_bfloat16*)out;
  p.num_kb = pl.num_kb;
  p.kb_per_split = pl.kb_per_split;
  const int sms = device_info().sm_count;
  const int64_t ntiles = (b.Cdst + bn - 1) / bn;
  const int64_t M = (int64_t)b.N * b.D * b.H * b.W;
  const int nslot = mt * (TBM / b.rb);
  const int64_t mtiles = (b.num_boxes + nslot - 1) / nslot;
  if (splits > 1) {
    p.partial = (float*)ws;
    cudaMemsetAsync(ws, 0, (size_t)(M * b.Cdst * 4), st);
  }
  if (ex && ex->gn_sums && epilogue_stats_ok(b, pl, ex->gn_groups)) {
    p.gn_sums = ex->gn_sums;
    p.gn_G = ex->gn_groups;
    p.gn_cpg = b.Cdst / ex->gn_groups;
    ex->stats_done = true;
  }
  p.mtiles = (int)mtiles; p.ntiles = (int)ntiles; p.splits = splits;
  {
    static int groups = 0;
    if (groups == 0) {
      const char* e = getenv("MIG_CONV_EPI_GROUPS");
      groups = (e && e[0] == '1') ? 1 : 2;
    }
    p.epi_groups = groups;
  }
  int64_t nct = mtiles * ntiles * splits;
  static int one_tile_per_cta = -1;   // A/B switch: static round-robin persistence vs. hardware CTA scheduling
  if (one_tile_per_cta < 0) {
    const char* e = getenv("MIG_CONV_NONPERSISTENT");
    one_tile_per_cta = (e && e[0] == '1') ? 1 : 0;
  }
  const int64_t all_tiles = nct;
  if (nct > sms && !one_tile_per_cta) nct = sms;
  dim3 grid((unsigned)nct);   // persistent: one CTA per SM walks the tiles
  p.sched = all_tiles > nct ? next_tile_counter(st) : nullptr;
  int rc;
  if (bmn) {
    if (mt == 2 && bn == 256) rc = launch_conv_tma<256, 2, true>(xm, wm, p, grid, st);
    else if (mt == 2 && bn == 128) rc = launch_conv_tma<128, 2, true>(xm, wm, p, grid, st);
    else if (mt == 2) rc = launch_conv_tma<64, 2, true>(xm, wm, p, grid, st);
    else if (bn == 256) rc = launch_conv_tma<256, 1, true>(xm, wm, p, grid, st);
    else if (bn == 128) rc = launch_conv_tma<128, 1, true>(xm, wm, p, grid, st);
    else rc = launch_conv_tma<64, 1, true>(xm, wm, p, grid, st);
  } else
  if (mt == 2 && bn == 256) rc = launch_conv_tma<256, 2>(xm, wm, p, grid, st);
  else if (mt == 2 && bn == 128) rc = launch_conv_tma<128, 2>(xm, wm, p, grid, st);
  else if (mt == 2 && bn == 64) rc = launch_conv_tma<64, 2>(xm, wm, p, grid, st);
  else if (mt == 2) rc = launch_conv_tma<32, 2>(xm, wm, p, grid, st);
  else if (bn == 256) rc = launch_conv_tma<256, 1>(xm, wm, p, grid, st);
  else if (bn == 128) rc = launch_conv_tma<128, 1>(xm, wm, p, grid, st);
  else if (bn == 64) rc = launch_conv_tma<64, 1>(xm, wm, p, grid, st);
  else rc = launch_conv_tma<32, 1>(xm, wm, p, grid, st);
  if (rc) return rc;
  if (splits > 1) {
    if (b.Cdst % 8 == 0 && aligned16(ws) && aligned16(bias) && aligned16(chan_bias) && aligned16(residual) &&
        aligned16(out))
      tma_splitk_finish8<<<bw_grid(M * b.Cdst / 8, 256), 256, 0, st>>>((const float*)ws, bias, chan_bias,
                                                                       (const __nv_bfloat16*)residual,
                                                                       (__nv_bfloat16*)out, M, b.Cdst,
                                                                       (int64_t)b.D * b.H * b.W);
    else
      tma_splitk_finish<<<bw_grid(M * b.Cdst, 256), 256, 0, st>>>((const float*)ws, bias, chan_bias,
                                                                  (const __nv_bfloat16*)residual, (__nv_bfloat16*)out, M,
                                                                  b.Cdst, (int64_t)b.D * b.H * b.W);
    return check_launch("tma_splitk_finish");
  }
  return 0;
}

// gn_sums / gn_groups (optional): GroupNorm statistics of y from the epilogue; *stats_done tells whether they were
// produced (a split-K plan cannot: its epilogue only sees partial sums).
int tma_conv_fwd(const mig_conv_geom* g, const void* x, const void* w, const float* bias, const float* chan_bias,
                 const void* residual, void* y, void* ws, int64_t ws_bytes, void* stream, double* gn_sums,
                 int gn_groups, int* stats_done) {
  BoxExtras ex;
  ex.gn_sums = gn_sums;
  ex.gn_groups = gn_groups;
  int rc = run_conv_tma(g, 0, x, w, bias, chan_bias, residual, y, ws, ws_bytes, stream, &ex);
  if (stats_done) *stats_done = ex.stats_done ? 1 : 0;
  return rc;
}

// would tma_conv_fwd's epilogue produce the GroupNorm statistics for this geometry / workspace?
bool tma_conv_fwd_stats_in_epilogue(const mig_conv_geom* g, int gn_groups, int64_t ws_bytes) {
  const BoxGeom b = make_box_geom(g, 0);
  return epilogue_stats_ok(b, plan_box(b, ws_bytes), gn_groups);
}

int tma_conv_dgrad(const mig_conv_geom* g, const void* dy, const void* w, void* dx, void* ws, int64_t ws_bytes,
                   void* stream) {
  static int bmn_ok = -1;   // A/B switch: MIG_DGRAD_TRANSPOSE=1 restores the per-call transposed filter copy
  if (bmn_ok < 0) {
    const char* e = getenv("MIG_DGRAD_TRANSPOSE");
    bmn_ok = (e && e[0] == '1') ? 0 : 1;
  }
  if (bmn_ok && g->Cin % 64 == 0) {
    // the forward filter [Cout][taps][Cin] IS an MN-major B operand for dX = dY * W: no transposed copy, no workspace
    BoxExtras ex;
    ex.bmn = true;
    return run_conv_tma(g, 1, dy, w, nullptr, nullptr, nullptr, dx, ws, ws_bytes, stream, &ex);
  }
  const int T = g->ksize[0] * g->ksize[1] * g->ksize[2];
  int64_t wt_bytes = ((int64_t)g->Cin * T * g->Cout * 2 + 255) / 256 * 256;
  MIG_REQUIRE(ws && ws_bytes >= wt_bytes, "conv_dgrad(tma): workspace too small");
  if (filter_transpose(MIG_BF16, w, ws, g->Cout, T, g->Cin, stream)) return 2;
  return run_conv_tma(g, 1, dy, ws, nullptr, nullptr, nullptr, dx, (uint8_t*)ws + wt_bytes, ws_bytes - wt_bytes, stream);
}

// ---------------------------------------------------------------------------------------------------
// strided dgrad by stride-residue classes
// ---------------------------------------------------------------------------------------------------
// Every class (residue_classes.cuh) runs as a dense stride-1 box problem on the conv kernel, without split-K.
bool tma_dgrad_strided_eligible(const mig_conv_geom* g) {
  bool any = false;
  for (int i = 0; i < 3; ++i) {
    if (g->stride[i] < 1 || g->stride[i] > 2) return false;
    any = any || g->stride[i] == 2;
  }
  if (!any || g->Cout % 64 != 0 || g->Cin < 8) return false;
  ResidueClass cls[kMaxClasses];
  const int n = residue_classes(g, cls);
  for (int i = 0; i < n; ++i) {
    const AxisClass* a = cls[i].a;
    int bd, bh, bw;
    if (cls[i].ntaps > kMaxClassTaps || !pick_box(a[0].ext, a[1].ext, a[2].ext, &bd, &bh, &bw)) return false;
  }
  return true;
}

int tma_conv_dgrad_strided(const mig_conv_geom* g, const void* dy, const void* w, void* dx, void* ws, int64_t ws_bytes,
                           void* stream) {
  auto launch_class = [&](const ResidueClass& c, const void* wsub) {
    int ext[3], nu[3], base[3], o[3];
    for (int i = 0; i < 3; ++i) { ext[i] = c.a[i].ext; nu[i] = c.a[i].nu; base[i] = c.a[i].base; o[i] = c.a[i].o; }
    BoxGeom b;
    box_geom(b, kBox64, g->N, ext, nu, base, -1, kOnes, g->stride, o, g->in_dims, g->Cout, g->Cin);
    return launch_box_conv(b, g->N, g->out_dims, dy, wsub, nullptr, nullptr, nullptr, dx, nullptr, 0, stream);
  };
  return dgrad_by_residue_classes(g, w, dx, ws, ws_bytes, stream, "conv_dgrad(tma, strided)", launch_class);
}

// ---------------------------------------------------------------------------------------------------
// folded upsample convolution, forward: one residue class written straight into the full-resolution output
// ---------------------------------------------------------------------------------------------------
// Class r of "nearest x f + conv" (upconv.cu) is a dense stride-1 convolution of the low-resolution tensor whose rows
// land at f*j + r of the output: the row mapping (os, oo, OD/OH/OW) the strided dgrad above uses, with sign = +1.
bool tma_upconv_class_eligible(int N, const int32_t low[3], int Cin, int Cout) {
  if (Cin % 8 != 0 || Cin < 48 || Cout % 8 != 0) return false;
  if ((double)N * low[0] * low[1] * low[2] > 16.0 * 2147483647.0) return false;
  int bd, bh, bw;
  return pick_box(low[0], low[1], low[2], &bd, &bh, &bw);
}

int tma_upconv_class_fwd(int N, const int32_t low[3], const int32_t factor[3], const int32_t res[3], const int32_t nu[3],
                         const int32_t base[3], int Cin, int Cout, const void* x, const void* wc, const float* bias,
                         void* y, void* stream) {
  const int out[3] = {low[0] * factor[0], low[1] * factor[1], low[2] * factor[2]};
  BoxGeom b;
  MIG_REQUIRE(box_geom(b, kBox64, N, low, nu, base, 1, kOnes, factor, res, out, Cin, Cout),
              "upconv_fwd: no TMA box for this volume");
  return launch_box_conv(b, N, low, x, wc, bias, nullptr, nullptr, y, nullptr, 0, stream);
}

template <int BN, int MT>
static int launch_wgrad_tma(const CUtensorMap& dym, const CUtensorMap& xm, const WgradTmaParams& p, dim3 grid,
                            cudaStream_t st) {
  constexpr int stage = (2 * MT + BN / 64) * PANEL;
  constexpr int smem = stages_of(stage) * stage + 1024;
  static SmemOptIn optin;
  if (int rc = ensure_dynamic_smem(wgrad_tma_kernel<BN, MT>, smem, optin, "wgrad_tma")) return rc;
  wgrad_tma_kernel<BN, MT><<<grid, kThreads, smem, st>>>(dym, xm, p);
  return check_launch("wgrad_tma_kernel");
}

int tma_conv_wgrad(const mig_conv_geom* g, const void* x, const void* dy, float* dw, void* stream) {
  BoxGeom b = make_box_geom(g, 2);
  cudaStream_t st = as_stream(stream);
  CUtensorMap dym, xm;
  if (make_act_map(&dym, dy, g->N, g->out_dims, g->Cout, b.bd, b.bh, b.bw)) return 1;
  if (make_act_map(&xm, x, g->N, g->in_dims, g->Cin, b.bd, b.bh, b.bw, b.ss)) return 1;
  // Tile / split plan from the same kind of cost model as the forward kernel: stage = max(UMMA, TMA row issue),
  // CTA = stages + prologue + fp32 reduction epilogue (16-byte red ops), grid = ceil(CTAs / SMs) waves.
  int bn = 64, mt = 1;
  int64_t splits = 1;
  {
    const int sms = device_info().sm_count;
    static const int cand_t[][2] = {{256, 2}, {256, 1}, {128, 1}, {64, 1}};
    double best = 1e30;
    for (auto& c : cand_t) {
      const int bn_ = c[0], mt_ = c[1];
      if (bn_ > 64 && b.K <= bn_ / 2) continue;
      if (mt_ == 2 && g->Cout <= 128) continue;
      const int64_t tiles = (int64_t)((g->Cout + TBM * mt_ - 1) / (TBM * mt_)) * ((b.K + bn_ - 1) / bn_);
      const double t_stage = fmax(512.0 * mt_ * bn_ / 256.0 * b.nb / 64.0, b.nb * 3.5 * (2 * mt_ + bn_ / 64));
      const double t_epi = 2500.0 + mt_ * 128.0 * bn_ / 5.0;
      for (int64_t s_ = 1; s_ <= b.num_boxes && s_ <= 4096; s_ = s_ < 8 ? s_ + 1 : s_ + s_ / 4) {
        const double waves = (double)((tiles * s_ + sms - 1) / sms);
        const double st = (double)((b.num_boxes + s_ - 1) / s_);
        const double t = waves * (st * t_stage + t_epi + 2500.0);
        if (t < best) { best = t; bn = bn_; mt = mt_; splits = s_; }
      }
    }
  }
  WgradTmaParams p{};
  p.g = b;
  p.dw = dw;
  const int mrows = TBM * mt;
  if (splits > 65535) splits = 65535;
  p.boxes_per_split = (b.num_boxes + splits - 1) / splits;
  splits = (b.num_boxes + p.boxes_per_split - 1) / p.boxes_per_split;
  dim3 grid((unsigned)((g->Cout + mrows - 1) / mrows), (unsigned)((b.K + bn - 1) / bn), (unsigned)splits);
  MIG_REQUIRE(grid.y < 65536, "conv_wgrad(tma): filter too large");
  if (mt == 2) return launch_wgrad_tma<256, 2>(dym, xm, p, grid, st);
  if (bn == 256) return launch_wgrad_tma<256, 1>(dym, xm, p, grid, st);
  if (bn == 128) return launch_wgrad_tma<128, 1>(dym, xm, p, grid, st);
  return launch_wgrad_tma<64, 1>(dym, xm, p, grid, st);
}

}  // namespace mig

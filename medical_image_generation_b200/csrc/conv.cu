// C-ABI entry points for convolution and strided GEMM: engine selection between
//   * the all-TMA tcgen05 kernels (conv_tma.cu)        -- stride 1, channel counts multiple of 64
//   * the cp.async-gather tcgen05 kernels (gemm_tc*.cu) -- any stride, channel counts multiple of 8
//   * the SIMT family (gemm_simt.cu)                    -- everything, and the fp32 parity mode
//   * skinny-linear kernels (small_ops.cu)              -- <= 32 rows (time-embedding path)
// Convolutions with 1/3-channel ends (conv_in, out) are zero-padded to 8 channels in workspace so they can use
// the tensor-core kernels as well.
#include <cstdlib>

#include "common.cuh"

namespace mig {
// gemm_simt.cu
int simt_conv_fwd(const mig_conv_geom* g, int dtype, const void* x, const void* w, const float* bias,
                  const float* chan_bias, const void* residual, void* y, void* stream);
int simt_conv_dgrad(const mig_conv_geom* g, int dtype, const void* dy, const void* wt, void* dx, void* stream);
int simt_conv_wgrad(const mig_conv_geom* g, int dtype, const void* x, const void* dy, float* dw, void* stream);
int simt_gemm_strided(const mig_gemm_desc* d, int dtype_ab, int dtype_c, const void* A, const void* B, void* C,
                      void* stream);
int filter_transpose(int dtype, const void* w, void* wt, int Cout, int Tn, int Cin, void* stream);
// gemm_tc.cu / gemm_tc2.cu
bool tc_conv_eligible(const mig_conv_geom* g, int dtype, int which);
int tc_conv_fwd(const mig_conv_geom* g, const void* x, const void* w, const float* bias, const float* chan_bias,
                const void* residual, void* y, void* ws, int64_t ws_bytes, void* stream);
int tc_conv_dgrad(const mig_conv_geom* g, const void* dy, const void* w, void* dx, void* ws, int64_t ws_bytes,
                  void* stream);
int tc_conv_wgrad(const mig_conv_geom* g, const void* x, const void* dy, float* dw, void* ws, int64_t ws_bytes,
                  void* stream);
int64_t tc_conv_workspace(const mig_conv_geom* g, int which);
bool tc_gemm_eligible(const mig_gemm_desc* d, int dtype_ab, int dtype_c);
int tc_gemm_strided(const mig_gemm_desc* d, int dtype_c, const void* A, const void* B, void* C, void* stream);
// conv_tma.cu
bool tma_conv_eligible(const mig_conv_geom* g, int which);
int tma_conv_fwd(const mig_conv_geom* g, const void* x, const void* w, const float* bias, const float* chan_bias,
                 const void* residual, void* y, void* ws, int64_t ws_bytes, void* stream, double* gn_sums = nullptr,
                 int gn_groups = 0, int* stats_done = nullptr);
bool tma_conv_fwd_stats_in_epilogue(const mig_conv_geom* g, int gn_groups, int64_t ws_bytes);
// groupnorm_tma.cu
bool gt_eligible(int N, int64_t S, int C, int G);
int gt_stats(const void* x, double* sums, int N, int64_t S, int C, int G, void* stream);
int tma_conv_dgrad(const mig_conv_geom* g, const void* dy, const void* w, void* dx, void* ws, int64_t ws_bytes,
                   void* stream);
int tma_conv_wgrad(const mig_conv_geom* g, const void* x, const void* dy, float* dw, void* stream);
bool tma_dgrad_strided_eligible(const mig_conv_geom* g);
bool halo_dgrad_strided_eligible(const mig_conv_geom* g);
int halo_conv_dgrad_strided(const mig_conv_geom* g, const void* dy, const void* w, void* dx, void* ws, int64_t ws_bytes,
                            void* stream);
int tma_conv_dgrad_strided(const mig_conv_geom* g, const void* dy, const void* w, void* dx, void* ws, int64_t ws_bytes,
                           void* stream);
// small_ops.cu
bool skinny_eligible(const mig_conv_geom* g);
int skinny_fwd(const mig_conv_geom* g, int dtype, const void* x, const void* w, const float* bias,
               const float* chan_bias, const void* residual, void* y, void* stream);
int skinny_dgrad(const mig_conv_geom* g, int dtype, const void* dy, const void* w, void* dx, void* stream);
int skinny_wgrad(const mig_conv_geom* g, int dtype, const void* x, const void* dy, float* dw, void* stream);
int pad_channels(int dtype, const void* src, void* dst, int64_t rows, int C, int Cp, void* stream);
int unpad_add(const float* src, float* dst, int64_t rows, int C, int Cp, void* stream);

static bool tma_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MIG_DISABLE_TMA_CONV");
    v = (e && e[0] == '1') ? 0 : 1;
  }
  return v == 1;
}
static int taps(const mig_conv_geom* g) { return g->ksize[0] * g->ksize[1] * g->ksize[2]; }
static int64_t esize(int dtype) { return dtype == MIG_BF16 ? 2 : 4; }
static int64_t in_vox(const mig_conv_geom* g) { return (int64_t)g->N * g->in_dims[0] * g->in_dims[1] * g->in_dims[2]; }
static int64_t out_vox(const mig_conv_geom* g) {
  return (int64_t)g->N * g->out_dims[0] * g->out_dims[1] * g->out_dims[2];
}
static int64_t up256(int64_t v) { return (v + 255) / 256 * 256; }
static int pad8(int c) { return (c + 7) / 8 * 8; }

static bool tc_device(int dtype, int engine) { return engine != 1 && dtype == MIG_BF16 && mig_has_tcgen05(); }
static bool use_tc(const mig_conv_geom* g, int dtype, int which, int engine) {
  return tc_device(dtype, engine) && tc_conv_eligible(g, dtype, which);
}
// pad 1/3/..-channel ends to 8 so the tcgen05 kernels apply (only worth it for real volumes)
static bool want_pad(const mig_conv_geom* g, int dtype, int which, int engine) {
  if (!tc_device(dtype, engine) || tc_conv_eligible(g, dtype, which)) return false;
  if (out_vox(g) < 4096) return false;
  if (which == 0) return g->Cin % 8 != 0;                       // fwd only needs Cin % 8
  if (which == 1) return g->Cout % 8 != 0;                      // dgrad only needs Cout % 8
  return g->Cin % 8 != 0 || g->Cout % 8 != 0;                   // wgrad needs both
}

// conv_halo.cu: 32-channel layers with a smem-resident halo tile
bool halo_conv_eligible(const mig_conv_geom* g, int which);
int halo_conv_fwd(const mig_conv_geom* g, const void* x, const void* w, const float* bias, const float* chan_bias,
                  const void* residual, void* y, void* stream);
int halo_conv_dgrad(const mig_conv_geom* g, const void* dy, const void* w, void* dx, void* ws, int64_t ws_bytes,
                    void* stream);
bool halo_wgrad_eligible(const mig_conv_geom* g);
int halo_conv_wgrad(const mig_conv_geom* g, const void* x, const void* dy, float* dw, void* stream);
// conv_thin.cu: CUDA-core kernels for the 1..4-channel ends (conv_in / out conv at full resolution)
bool thin_conv_eligible(const mig_conv_geom* g, int which);
int thin_conv(const mig_conv_geom* g, int which, const void* thin, const void* w, const float* bias,
              const float* chan_bias, const void* residual, void* out, void* stream);
int thin_conv_wgrad(const mig_conv_geom* g, const void* x, const void* dy, float* dw, void* stream);
static bool thin_ok(const mig_conv_geom* g, int dtype, int which, int engine) {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MIG_DISABLE_THIN_CONV");
    v = (e && e[0] == '1') ? 0 : 1;
  }
  return v == 1 && dtype == MIG_BF16 && engine != 1 && thin_conv_eligible(g, which);
}
static bool halo_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MIG_DISABLE_HALO_CONV");
    v = (e && e[0] == '1') ? 0 : 1;
  }
  return v == 1;
}

static int run_fwd(const mig_conv_geom* g, const void* x, const void* w, const float* bias, const float* chan_bias,
                   const void* residual, void* y, void* ws, int64_t wsb, void* stream, double* gn_sums = nullptr,
                   int gn_groups = 0, int* stats_done = nullptr) {
  if (halo_enabled() && halo_conv_eligible(g, 0) && aligned16(x) && aligned16(w) && aligned16(y) &&
      (!residual || aligned16(residual)))
    return halo_conv_fwd(g, x, w, bias, chan_bias, residual, y, stream);
  if (tma_enabled() && tma_conv_eligible(g, 0) && aligned16(x) && aligned16(w) && aligned16(y) &&
      (!residual || aligned16(residual)))
    return tma_conv_fwd(g, x, w, bias, chan_bias, residual, y, ws, wsb, stream, gn_sums, gn_groups, stats_done);
  return tc_conv_fwd(g, x, w, bias, chan_bias, residual, y, ws, wsb, stream);
}
static int run_dgrad(const mig_conv_geom* g, const void* dy, const void* w, void* dx, void* ws, int64_t wsb,
                     void* stream) {
  if (halo_enabled() && halo_conv_eligible(g, 1) && aligned16(dy) && aligned16(w) && aligned16(dx))
    return halo_conv_dgrad(g, dy, w, dx, ws, wsb, stream);
  if (halo_enabled() && halo_dgrad_strided_eligible(g) && aligned16(dy) && aligned16(w) && aligned16(dx))
    return halo_conv_dgrad_strided(g, dy, w, dx, ws, wsb, stream);
  if (tma_enabled() && aligned16(dy) && aligned16(w) && aligned16(dx)) {
    if (tma_conv_eligible(g, 1)) return tma_conv_dgrad(g, dy, w, dx, ws, wsb, stream);
    if (tma_dgrad_strided_eligible(g)) return tma_conv_dgrad_strided(g, dy, w, dx, ws, wsb, stream);
  }
  return tc_conv_dgrad(g, dy, w, dx, ws, wsb, stream);
}
static int run_wgrad(const mig_conv_geom* g, const void* x, const void* dy, float* dw, void* ws, int64_t wsb,
                     void* stream) {
  if (halo_enabled() && halo_wgrad_eligible(g) && aligned16(x) && aligned16(dy) && aligned16(dw))
    return halo_conv_wgrad(g, x, dy, dw, stream);
  if (tma_enabled() && tma_conv_eligible(g, 2) && aligned16(x) && aligned16(dy)) return tma_conv_wgrad(g, x, dy, dw, stream);
  return tc_conv_wgrad(g, x, dy, dw, ws, wsb, stream);
}

// workspace needed by the padded variants (on top of the inner call's own workspace)
static int64_t pad_workspace(const mig_conv_geom* g, int which) {
  const int cin = pad8(g->Cin), cout = pad8(g->Cout), T = taps(g);
  if (which == 0) return up256(in_vox(g) * cin * 2) + up256((int64_t)g->Cout * T * cin * 2);
  if (which == 1) return up256(out_vox(g) * cout * 2) + up256((int64_t)cout * T * g->Cin * 2);
  return up256(in_vox(g) * cin * 2) + up256(out_vox(g) * cout * 2) + up256((int64_t)cout * T * cin * 4);
}
static mig_conv_geom padded_geom(const mig_conv_geom* g, bool pin, bool pout) {
  mig_conv_geom q = *g;
  if (pin) q.Cin = pad8(g->Cin);
  if (pout) q.Cout = pad8(g->Cout);
  return q;
}
}  // namespace mig

using namespace mig;

extern "C" int64_t mig_conv_workspace_bytes(const mig_conv_geom* g, int dtype, int which, int engine) {
  if (!g) return 0;
  int64_t simt = which == 1 ? (int64_t)g->Cin * taps(g) * g->Cout * esize(dtype) : 0;
  if (engine == 1 || dtype != MIG_BF16) return simt;
  int64_t tc = tc_conv_workspace(g, which);
  if (want_pad(g, dtype, which, engine)) {
    mig_conv_geom q = padded_geom(g, which != 1, which != 0);
    tc = pad_workspace(g, which) + tc_conv_workspace(&q, which);
  }
  return simt > tc ? simt : tc;
}

static int conv_fwd_impl(const mig_conv_geom* g, int dtype, const void* x, const void* w, const float* bias,
                         const float* chan_bias, const void* residual, void* y, int engine, void* workspace,
                         int64_t workspace_bytes, void* stream, double* gn_sums, int gn_groups, int* stats_done);

extern "C" int mig_conv_fwd(const mig_conv_geom* g, int dtype, const void* x, const void* w, const float* bias,
                            const float* chan_bias, const void* residual, void* y, int engine, void* workspace,
                            int64_t workspace_bytes, void* stream) {
  return conv_fwd_impl(g, dtype, x, w, bias, chan_bias, residual, y, engine, workspace, workspace_bytes, stream, nullptr,
                       0, nullptr);
}

// mig_conv_fwd that ALSO delivers the GroupNorm statistics of its output: gn_sums[n][g][2] (fp64) = (sum y, sum y^2) per
// (sample, group) of the bf16-rounded result, for the GroupNorm that consumes it (unet:648,698; ae:167): from the
// epilogue of the tcgen05 kernel where the plan allows it, otherwise by one statistics pass over y. Requires
// mig_groupnorm_can_split(dtype, N, out voxels, Cout, gn_groups).
extern "C" int mig_conv_fwd_stats(const mig_conv_geom* g, int dtype, const void* x, const void* w, const float* bias,
                                  const float* chan_bias, const void* residual, void* y, double* gn_sums,
                                  int32_t gn_groups, int engine, void* workspace, int64_t workspace_bytes,
                                  void* stream) {
  MIG_REQUIRE(g && gn_sums && gn_groups > 0, "conv_fwd_stats: null argument");
  const int64_t S = (int64_t)g->out_dims[0] * g->out_dims[1] * g->out_dims[2];
  MIG_REQUIRE(dtype == MIG_BF16 && gt_eligible(g->N, S, g->Cout, gn_groups),
              "conv_fwd_stats: output is not eligible for split GroupNorm (bf16, Cout a multiple of 32)");
  cudaMemsetAsync(gn_sums, 0, sizeof(double) * (size_t)g->N * gn_groups * 2, as_stream(stream));
  int done = 0;
  if (int rc = conv_fwd_impl(g, dtype, x, w, bias, chan_bias, residual, y, engine, workspace, workspace_bytes, stream,
                             gn_sums, gn_groups, &done))
    return rc;
  if (done) return 0;
  return gt_stats(y, gn_sums, g->N, S, g->Cout, gn_groups, stream);
}

// 1 when mig_conv_fwd_stats takes the statistics from the tcgen05 epilogue for this geometry (0: statistics pass over y)
extern "C" int mig_conv_fwd_stats_in_epilogue(const mig_conv_geom* g, int dtype, int32_t gn_groups, int engine,
                                              int64_t workspace_bytes) {
  if (!g || !use_tc(g, dtype, 0, engine) || !tma_enabled() || !tma_conv_eligible(g, 0)) return 0;
  if (halo_enabled() && halo_conv_eligible(g, 0)) return 0;
  if (skinny_eligible(g) || thin_ok(g, dtype, 0, engine)) return 0;
  return tma_conv_fwd_stats_in_epilogue(g, gn_groups, workspace_bytes) ? 1 : 0;
}

static int conv_fwd_impl(const mig_conv_geom* g, int dtype, const void* x, const void* w, const float* bias,
                         const float* chan_bias, const void* residual, void* y, int engine, void* workspace,
                         int64_t workspace_bytes, void* stream, double* gn_sums, int gn_groups, int* stats_done) {
  MIG_REQUIRE(g && x && w && y, "conv_fwd: null argument");
  if (skinny_eligible(g) && !chan_bias && !residual) return skinny_fwd(g, dtype, x, w, bias, nullptr, nullptr, y, stream);
  if (thin_ok(g, dtype, 0, engine) && aligned16(y) && (!residual || aligned16(residual)))
    return thin_conv(g, 0, x, w, bias, chan_bias, residual, y, stream);
  if (use_tc(g, dtype, 0, engine))
    return run_fwd(g, x, w, bias, chan_bias, residual, y, workspace, workspace_bytes, stream, gn_sums, gn_groups, stats_done);
  if (want_pad(g, dtype, 0, engine) && workspace && workspace_bytes >= mig_conv_workspace_bytes(g, dtype, 0, engine)) {
    // pad the input channels of x and of the filter to a multiple of 8 (zeros), then the normal tensor-core path
    const int cp = pad8(g->Cin), T = taps(g);
    uint8_t* p = (uint8_t*)workspace;
    void* xp = p; p += up256(in_vox(g) * cp * 2);
    void* wp = p; p += up256((int64_t)g->Cout * T * cp * 2);
    if (pad_channels(dtype, x, xp, in_vox(g), g->Cin, cp, stream)) return 2;
    if (pad_channels(dtype, w, wp, (int64_t)g->Cout * T, g->Cin, cp, stream)) return 2;
    mig_conv_geom q = padded_geom(g, true, false);
    return run_fwd(&q, xp, wp, bias, chan_bias, residual, y, p, workspace_bytes - (p - (uint8_t*)workspace), stream);
  }
  MIG_REQUIRE(engine != 2, "conv_fwd: tcgen05 engine requested but shape/dtype/device not eligible");
  return simt_conv_fwd(g, dtype, x, w, bias, chan_bias, residual, y, stream);
}

extern "C" int mig_conv_dgrad(const mig_conv_geom* g, int dtype, const void* dy, const void* w, void* dx, int engine,
                              void* workspace, int64_t workspace_bytes, void* stream) {
  MIG_REQUIRE(g && dy && w && dx, "conv_dgrad: null argument");
  if (skinny_eligible(g)) return skinny_dgrad(g, dtype, dy, w, dx, stream);
  if (thin_ok(g, dtype, 1, engine) && aligned16(dx)) return thin_conv(g, 1, dy, w, nullptr, nullptr, nullptr, dx, stream);
  if (use_tc(g, dtype, 1, engine)) return run_dgrad(g, dy, w, dx, workspace, workspace_bytes, stream);
  if (want_pad(g, dtype, 1, engine) && workspace && workspace_bytes >= mig_conv_workspace_bytes(g, dtype, 1, engine)) {
    // pad the output channels: dy gets zero channels, the filter gets zero rows
    const int cp = pad8(g->Cout), T = taps(g);
    uint8_t* p = (uint8_t*)workspace;
    void* dyp = p; p += up256(out_vox(g) * cp * 2);
    void* wp = p; p += up256((int64_t)cp * T * g->Cin * 2);
    if (pad_channels(dtype, dy, dyp, out_vox(g), g->Cout, cp, stream)) return 2;
    const size_t wbytes = (size_t)g->Cout * T * g->Cin * 2;
    cudaMemsetAsync((uint8_t*)wp + wbytes, 0, (size_t)(cp - g->Cout) * T * g->Cin * 2, as_stream(stream));
    cudaMemcpyAsync(wp, w, wbytes, cudaMemcpyDeviceToDevice, as_stream(stream));
    mig_conv_geom q = padded_geom(g, false, true);
    return run_dgrad(&q, dyp, wp, dx, p, workspace_bytes - (p - (uint8_t*)workspace), stream);
  }
  MIG_REQUIRE(engine != 2, "conv_dgrad: tcgen05 engine requested but shape/dtype/device not eligible");
  int64_t need = (int64_t)g->Cin * taps(g) * g->Cout * esize(dtype);
  MIG_REQUIRE(workspace && workspace_bytes >= need, "conv_dgrad: workspace too small (%lld < %lld)",
              (long long)workspace_bytes, (long long)need);
  if (filter_transpose(dtype, w, workspace, g->Cout, taps(g), g->Cin, stream)) return 2;
  return simt_conv_dgrad(g, dtype, dy, workspace, dx, stream);
}

extern "C" int mig_conv_wgrad(const mig_conv_geom* g, int dtype, const void* x, const void* dy, float* dw,
                              float* dbias, int engine, void* workspace, int64_t workspace_bytes, void* stream) {
  MIG_REQUIRE(g && x && dy, "conv_wgrad: null argument");
  if (dbias) {
    if (mig_colsum(dtype, dy, dbias, out_vox(g), g->Cout, 1, stream)) return 2;
  }
  if (!dw) return 0;
  if (skinny_eligible(g)) return skinny_wgrad(g, dtype, x, dy, dw, stream);
  if (thin_ok(g, dtype, 2, engine)) return thin_conv_wgrad(g, x, dy, dw, stream);
  if (use_tc(g, dtype, 2, engine)) return run_wgrad(g, x, dy, dw, workspace, workspace_bytes, stream);
  if (want_pad(g, dtype, 2, engine) && workspace && workspace_bytes >= mig_conv_workspace_bytes(g, dtype, 2, engine)) {
    const int cin = pad8(g->Cin), cout = pad8(g->Cout), T = taps(g);
    uint8_t* p = (uint8_t*)workspace;
    const void* xs = x;
    const void* dys = dy;
    if (cin != g->Cin) {
      void* xp = p; p += up256(in_vox(g) * cin * 2);
      if (pad_channels(dtype, x, xp, in_vox(g), g->Cin, cin, stream)) return 2;
      xs = xp;
    }
    if (cout != g->Cout) {
      void* dyp = p; p += up256(out_vox(g) * cout * 2);
      if (pad_channels(dtype, dy, dyp, out_vox(g), g->Cout, cout, stream)) return 2;
      dys = dyp;
    }
    float* dwp = (float*)p; p += up256((int64_t)cout * T * cin * 4);
    cudaMemsetAsync(dwp, 0, (size_t)cout * T * cin * 4, as_stream(stream));
    mig_conv_geom q = padded_geom(g, true, true);
    int rc = run_wgrad(&q, xs, dys, dwp, p, workspace_bytes - (p - (uint8_t*)workspace), stream);
    if (rc) return rc;
    // dw[co][tap][ci] += dwp[co][tap][ci] for co < Cout, ci < Cin (the first Cout*T rows of the padded gradient)
    return unpad_add(dwp, dw, (int64_t)g->Cout * T, g->Cin, cin, stream);
  }
  MIG_REQUIRE(engine != 2, "conv_wgrad: tcgen05 engine requested but shape/dtype/device not eligible");
  return simt_conv_wgrad(g, dtype, x, dy, dw, stream);
}

extern "C" int mig_gemm_strided(const mig_gemm_desc* d, int dtype_ab, int dtype_c, const void* A, const void* B,
                                void* C, int engine, void* stream) {
  MIG_REQUIRE(d && A && B && C, "gemm: null argument");
  if (engine != 1 && mig_has_tcgen05() && tc_gemm_eligible(d, dtype_ab, dtype_c))
    return tc_gemm_strided(d, dtype_c, A, B, C, stream);
  MIG_REQUIRE(engine != 2, "gemm: tcgen05 engine requested but shape/dtype/device not eligible");
  return simt_gemm_strided(d, dtype_ab, dtype_c, A, B, C, stream);
}

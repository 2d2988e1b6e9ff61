// Strided convolution dgrad by stride-residue classes (host only), shared by the TMA box engine (conv_tma.cu) and the
// halo engine (conv_halo.cu).
//
// dx[i] = sum_t dy[(i + p - t)/s] w[t] over the taps with (i + p - t) % s == 0. Input voxels with the same residue
// rho = (i + p) mod s (per axis) see the same tap subset {rho, rho+s, ...}; writing i = s*j + o and t = rho + s*u
// gives dx_class[j] = sum_u dy[j - u + base] w[rho + s*u]: a dense stride-1 problem per class (2^d classes for
// stride 2), whose rows scatter back to dx with stride s. Total work = the useful work (no zero taps).
#pragma once
#include "common.cuh"

namespace mig {

int filter_transpose_taps(int dtype, const void* w, void* wt, int Cout, int Tn, int Cin, int ntaps, const int* taps,
                          void* stream);

// one axis of one class
struct AxisClass {
  int rho;    // residue: the first tap of the class
  int o;      // first input coordinate of the class
  int ext;    // how many input coordinates it holds
  int nu;     // taps rho, rho+s, ...
  int base;   // dy coordinate of (class row 0, tap rho)
};
inline AxisClass axis_class(int in, int k, int s, int p, int rho) {
  AxisClass a;
  a.rho = rho;
  a.o = ((rho - p) % s + s) % s;
  a.ext = in > a.o ? (in - a.o + s - 1) / s : 0;
  a.nu = rho < k ? (k - rho + s - 1) / s : 0;
  a.base = (a.o + p - rho) / s;
  return a;
}

constexpr int kMaxClasses = 8;      // strides 1 or 2 on three axes
constexpr int kMaxClassTaps = 32;   // filter_transpose_taps' limit

struct ResidueClass {
  AxisClass a[3];
  int ntaps;                  // a[0].nu * a[1].nu * a[2].nu; 0: these input voxels receive no gradient
  int taps[kMaxClassTaps];    // the class's filter taps, u2 fastest; filled when ntaps <= kMaxClassTaps
};

// The classes holding at least one input voxel, in (r0, r1, r2) order. Every stride must be 1 or 2.
inline int residue_classes(const mig_conv_geom* g, ResidueClass cls[kMaxClasses]) {
  int n = 0;
  for (int r0 = 0; r0 < g->stride[0]; ++r0)
    for (int r1 = 0; r1 < g->stride[1]; ++r1)
      for (int r2 = 0; r2 < g->stride[2]; ++r2) {
        ResidueClass& c = cls[n];
        const int r[3] = {r0, r1, r2};
        for (int i = 0; i < 3; ++i) c.a[i] = axis_class(g->in_dims[i], g->ksize[i], g->stride[i], g->pad[i], r[i]);
        if (c.a[0].ext == 0 || c.a[1].ext == 0 || c.a[2].ext == 0) continue;
        c.ntaps = c.a[0].nu * c.a[1].nu * c.a[2].nu;
        if (c.ntaps <= kMaxClassTaps) {
          int nt = 0;
          for (int u0 = 0; u0 < c.a[0].nu; ++u0)
            for (int u1 = 0; u1 < c.a[1].nu; ++u1)
              for (int u2 = 0; u2 < c.a[2].nu; ++u2)
                c.taps[nt++] = ((r0 + g->stride[0] * u0) * g->ksize[1] + (r1 + g->stride[1] * u1)) * g->ksize[2] +
                               (r2 + g->stride[2] * u2);
        }
        ++n;
      }
  return n;
}

// One strided dgrad (bf16). The workspace holds every class's transposed sub-filter [Cin][ntaps][Cout], each at a
// 256-byte boundary. When some class has no taps, dx is zeroed before any class runs. Then, per class with taps, the
// sub-filter is transposed and launch(cls, subfilter) runs the class as a dense stride-1 problem.
template <class LaunchClass>
int dgrad_by_residue_classes(const mig_conv_geom* g, const void* w, void* dx, void* ws, int64_t ws_bytes, void* stream,
                             const char* what, LaunchClass&& launch) {
  auto subfilter_bytes = [&](int ntaps) { return ((int64_t)g->Cin * ntaps * g->Cout * 2 + 255) / 256 * 256; };
  ResidueClass cls[kMaxClasses];
  const int n = residue_classes(g, cls);
  int64_t need = 0;
  bool need_zero = false;
  for (int i = 0; i < n; ++i) {
    need += subfilter_bytes(cls[i].ntaps);
    need_zero = need_zero || cls[i].ntaps == 0;
  }
  MIG_REQUIRE(ws && ws_bytes >= need, "%s: workspace too small", what);
  if (need_zero) {   // some input voxels receive no tap at all (e.g. kernel 1 with stride 2)
    const int64_t elems = (int64_t)g->N * g->in_dims[0] * g->in_dims[1] * g->in_dims[2] * g->Cin;
    cudaMemsetAsync(dx, 0, (size_t)elems * 2, as_stream(stream));
  }
  const int T = g->ksize[0] * g->ksize[1] * g->ksize[2];
  uint8_t* wp = (uint8_t*)ws;
  for (int i = 0; i < n; ++i) {
    if (cls[i].ntaps == 0) continue;
    if (filter_transpose_taps(MIG_BF16, w, wp, g->Cout, T, g->Cin, cls[i].ntaps, cls[i].taps, stream)) return 2;
    if (int rc = launch(cls[i], (const void*)wp)) return rc;
    wp += subfilter_bytes(cls[i].ntaps);
  }
  return 0;
}

}  // namespace mig

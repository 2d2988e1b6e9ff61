// Host-side helpers of the tcgen05 engine: TMA tensor-map construction through the driver entry point
// (resolved at run time with cudaGetDriverEntryPoint, so the library does not link against libcuda).
#pragma once
#include <cuda.h>

#include <mutex>

#include "common.cuh"

namespace mig {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// up to 5-d bf16 map; dims[0] is the contiguous one; strides in BYTES for dims 1..rank-1; `estrides` are per-dimension
// element strides (nullptr: all 1); `what` names the map in the error message. Out-of-bounds box elements are filled
// with zeros (K tails, M/N tails, halo rows).
inline int make_map(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box, const char* what = "tensor map",
                    CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B, const uint32_t* estrides = nullptr) {
  EncodeTiledFn enc = get_encode();
  MIG_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled unavailable (driver too old?)");
  cuuint64_t gd[5];
  cuuint64_t gs[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; es[i] = estrides ? estrides[i] : 1; }
  for (int i = 0; i + 1 < rank; ++i) gs[i] = strides_bytes[i];
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  MIG_REQUIRE(r == CUDA_SUCCESS, "%s: cuTensorMapEncodeTiled failed with %d (rank %d, dims %llu x %llu)", what, (int)r,
              rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0));
  return 0;
}

// 4-d map over a (B, L, H*dh) bf16 tensor with row pitch ld >= H*dh elements (contiguous: ld = H*dh):
// dims (dh, H, L, B); box (64, 1, rows, 1)
inline int bhld_map(CUtensorMap* m, const void* base, int B, int H, int L, int dh, uint32_t box_rows, int64_t ld) {
  uint64_t dims[4] = {(uint64_t)dh, (uint64_t)H, (uint64_t)L, (uint64_t)B};
  uint64_t strides[3] = {(uint64_t)dh * 2, (uint64_t)ld * 2, (uint64_t)L * (uint64_t)ld * 2};
  uint32_t box[4] = {64, 1, box_rows, 1};
  return make_map(m, base, 4, dims, strides, box, "attention map");
}

// output-channel tile of the tcgen05 convolution kernels: the smallest of 32 / 64 / 128 / 256 that covers cdst (capped)
inline int pick_bn(int cdst) { return cdst > 128 ? 256 : (cdst > 64 ? 128 : (cdst > 32 ? 64 : 32)); }

}  // namespace mig

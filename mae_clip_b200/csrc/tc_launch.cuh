// Host side of launching the tcgen05 engines (clip_loss_tc.cu, head_tc.cu, gemm_tc.cu): TMA tensor maps and CTA-pair
// cluster launches.
#pragma once

#include <cuda.h>
#include <type_traits>

#include "common.cuh"

namespace mc {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// cuTensorMapEncodeTiled from the driver, resolved once per process (null when the driver does not have it)
inline EncodeTiledFn encode_fn() {
  static const EncodeTiledFn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
                    q == cudaDriverEntryPointSuccess;
    return ok ? reinterpret_cast<EncodeTiledFn>(f) : nullptr;
  }();
  return fn;
}

// 2-D tensor [rows][cols] with `pitch_bytes` between rows, box {box_cols, box_rows}; out-of-range parts of a box read
// as zero
inline int make_map(CUtensorMap* m, CUtensorMapDataType dt, const void* ptr, uint64_t rows, uint64_t cols,
                    uint64_t pitch_bytes, uint32_t box_cols, uint32_t box_rows, CUtensorMapSwizzle sw) {
  EncodeTiledFn fn = encode_fn();
  MC_REQUIRE(fn != nullptr, MC_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  MC_REQUIRE(aligned(ptr, 16) && pitch_bytes % 16 == 0, MC_ERR_ALIGN, "TMA needs 16-byte aligned rows");
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {pitch_bytes};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, dt, 2, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  MC_REQUIRE(r == CUDA_SUCCESS, MC_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return MC_OK;
}

// dense fp16 [rows][cols], box {64 cols, box_rows}, 128-byte swizzle: the operand planes of the loss sweeps
inline int make_map_f16(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  return make_map(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, ptr, rows, cols, cols * 2, 64, box_rows, CU_TENSOR_MAP_SWIZZLE_128B);
}

// CTA pairs for `jobs` independent jobs: at most one pair per job, at most one pair per two SMs
inline int pairs_for(long jobs) {
  const int np = num_sms() / 2;
  return jobs < np ? (int)jobs : np;
}

// `npairs` clusters of two CTAs with `smem` bytes of dynamic shared memory each.  OPT_IN (when non-zero) is the opt-in
// for a kernel whose launch size varies between calls: the largest size it is ever launched with.
template <auto Kern, int OPT_IN = 0, typename... Args>
int launch_pairs(int npairs, int threads, int smem, cudaStream_t st, Args... args) {
  MC_CUDA(ensure_dynamic_smem<Kern>(OPT_IN ? OPT_IN : smem));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * npairs);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim = {2, 1, 1};
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  MC_CUDA(cudaLaunchKernelEx(&cfg, Kern, args...));
  count_launch();
  return MC_OK;
}

// f(std::integral_constant<int, 3>) for the three-pass (fp16x3) instantiation of a kernel, f(..., 1>) for one pass
template <typename F>
int with_passes(bool three, F&& f) {
  return three ? f(std::integral_constant<int, 3>{}) : f(std::integral_constant<int, 1>{});
}

}  // namespace mc

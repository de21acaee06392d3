// fp32-class tcgen05 GEMM for the ProjectionHead: see gemm_tc.cuh.  One CTA per 128 x 128 output
// tile (cta_group::1, M = 128, N = 128), persistent over (tile, K-split) jobs:
//   warp 0  TMA producer: per 64-wide K chunk the hi and lo planes of the A and B row blocks (4 x 16 KB)
//   warp 1  MMA issuer (one elected lane) + TMEM allocator: hi*hi + hi*lo + lo*hi into an fp32 TMEM tile
//   warps 2-5  epilogue: tcgen05.ld -> scale (+ bias, + exact-erf GELU second output) -> global
// Two TMEM tile buffers overlap the epilogue of one job with the MMAs of the next.
#include <stdlib.h>

#include "gemm_tc.cuh"
#include "tc_launch.cuh"
#include "tc_ptx.cuh"

namespace mc {
namespace tcg {

using namespace ptx;

constexpr int kChunk = 128 * 128;       // 128 rows x 64 fp16 (128 bytes per row)
constexpr int kStage = 4 * kChunk;      // A hi, A lo, B hi, B lo
constexpr int kStages = 3;
constexpr int kOffBar = kStages * kStage;
constexpr int kEpiPitch = 36;                        // floats per staged row: 32 + 4 (conflict-free 16-byte accesses)
constexpr int kEpiStage = 32 * kEpiPitch * 4;        // one warp's 32 x 32 block
constexpr int kOffEpi = kOffBar + 256;
constexpr int kSmem = kOffEpi + 4 * kEpiStage + 1024;
constexpr int kThreads = 192;
enum Bar { kFull0 = 0, kEmpty0 = 3, kTFull0 = 6, kTEmpty0 = 8, kNumBars = 10 };

struct GemmParams {
  int M, N, K;
  int tiles_m, tiles_n, ksplit, chunks_per_split, chunks_total;
  const float* scale_a;  // {s, 1/s}
  const float* scale_b;
  float* C;              // direct output (ksplit == 1) or partials (ksplit x M x N)
  int64_t ldc;
  const float* bias;
  float* gelu_out;
  int vec_ok;            // 16-byte stores allowed
  int coalesce;          // epilogue stores go through a per-warp shared-memory transpose (full 128-byte lines)
};

template <int EPI>
__global__ void __launch_bounds__(kThreads, 1)
gemm_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
            const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
            const GemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* const sbase = smem_raw + (base - raw);
  const uint32_t bar0 = base + kOffBar;
  auto bar = [&](int i) -> uint32_t { return bar0 + 8u * i; };
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(sbase + kOffBar + 8 * kNumBars);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int njobs = p.tiles_m * p.tiles_n * p.ksplit;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) { mbar_init(bar(kFull0 + s), 1); mbar_init(bar(kEmpty0 + s), 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(bar(kTFull0 + i), 1); mbar_init(bar(kTEmpty0 + i), 128); }
    fence_mbar_init();
    prefetch_tmap(&map_a_hi); prefetch_tmap(&map_a_lo); prefetch_tmap(&map_b_hi); prefetch_tmap(&map_b_lo);
  }
  if (warp == 1) tmem_alloc_1cta(smem_u32(tmem_slot), 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto job_coords = [&](int job, int& tm, int& tn, int& c0, int& c1) {
    const int tile = job % (p.tiles_m * p.tiles_n), ks = job / (p.tiles_m * p.tiles_n);
    // the shorter tile dimension runs fastest: CTAs working side by side then share their long operand in L2
    // (x W^T has 256 row tiles x 2 column tiles: with rows fastest the 268 MB activation was streamed from HBM twice)
    if (p.tiles_n <= p.tiles_m) {
      tn = tile % p.tiles_n;
      tm = tile / p.tiles_n;
    } else {
      tm = tile % p.tiles_m;
      tn = tile / p.tiles_m;
    }
    c0 = ks * p.chunks_per_split;
    c1 = min(c0 + p.chunks_per_split, p.chunks_total);
  };

  if (warp == 0) {
    if (elect_one()) {
      uint32_t it = 0;
      for (int job = blockIdx.x; job < njobs; job += gridDim.x) {
        int tm, tn, c0, c1;
        job_coords(job, tm, tn, c0, c1);
        for (int c = c0; c < c1; ++c, ++it) {
          const uint32_t stage = it % kStages, par = (it / kStages) & 1;
          mbar_wait(bar(kEmpty0 + stage), par ^ 1);
          const uint32_t fb = bar(kFull0 + stage);
          mbar_arrive_expect_tx(fb, kStage);
          const uint32_t sb = base + stage * kStage;
          tma_load_2d(sb, &map_a_hi, fb, c * 64, tm * 128);
          tma_load_2d(sb + kChunk, &map_a_lo, fb, c * 64, tm * 128);
          tma_load_2d(sb + 2 * kChunk, &map_b_hi, fb, c * 64, tn * 128);
          tma_load_2d(sb + 3 * kChunk, &map_b_lo, fb, c * 64, tn * 128);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc = idesc_f16(128, 128);
      uint32_t it = 0, tt = 0;
      for (int job = blockIdx.x; job < njobs; job += gridDim.x, ++tt) {
        int tm, tn, c0, c1;
        job_coords(job, tm, tn, c0, c1);
        const uint32_t buf = tt & 1, use = tt >> 1;
        mbar_wait(bar(kTEmpty0 + buf), (use & 1) ^ 1);
        tc_fence_after();
        const uint32_t td = tmem_base + buf * 128;
        for (int c = c0; c < c1; ++c, ++it) {
          const uint32_t stage = it % kStages, par = (it / kStages) & 1;
          mbar_wait(bar(kFull0 + stage), par);
          tc_fence_after();
          const uint32_t sb = base + stage * kStage;
          const uint64_t ah = smem_desc_sw128(sb), al = smem_desc_sw128(sb + kChunk);
          const uint64_t bh = smem_desc_sw128(sb + 2 * kChunk), bl = smem_desc_sw128(sb + 3 * kChunk);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint32_t acc = (c > c0 || ks > 0) ? 1u : 0u;
            mma_f16_1cta(td, desc_advance_k(ah, ks), desc_advance_k(bh, ks), idesc, acc);
            mma_f16_1cta(td, desc_advance_k(ah, ks), desc_advance_k(bl, ks), idesc, 1u);
            mma_f16_1cta(td, desc_advance_k(al, ks), desc_advance_k(bh, ks), idesc, 1u);
          }
          mma_commit_1cta(bar(kEmpty0 + stage));
        }
        mma_commit_1cta(bar(kTFull0 + buf));
      }
    }
    __syncwarp();
  } else {
    const int quarter = warp & 3;
    const uint32_t lane_field = (uint32_t)(quarter * 32) << 16;
    const float scale = p.scale_a[1] * p.scale_b[1];
    uint32_t tt = 0;
    for (int job = blockIdx.x; job < njobs; job += gridDim.x, ++tt) {
      int tm, tn, c0, c1;
      job_coords(job, tm, tn, c0, c1);
      const int ks = job / (p.tiles_m * p.tiles_n);
      const uint32_t buf = tt & 1, use = tt >> 1;
      mbar_wait(bar(kTFull0 + buf), use & 1);
      tc_fence_after();
      const int row = tm * 128 + quarter * 32 + lane;
      const bool split = p.ksplit > 1;
      float* crow = split ? p.C + ((size_t)ks * p.M + row) * p.N : p.C + (size_t)row * p.ldc;
      float* grow = (EPI == kEpiGelu && p.gelu_out) ? p.gelu_out + (size_t)row * p.ldc : nullptr;
#pragma unroll 1
      for (int cc = 0; cc < 128; cc += 32) {
        float v[32];
        tmem_ld32(tmem_base + lane_field + buf * 128 + cc, v);
        tmem_ld_wait();
        if (cc == 96) {  // all four reads of this tile are done: release the buffer
          tc_fence_before();
          mbar_arrive_local(bar(kTEmpty0 + buf));
        }
        const int col0 = tn * 128 + cc;
        if (row >= p.M || col0 >= p.N) continue;
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          v[e] *= scale;
          if (!split && p.bias && col0 + e < p.N) v[e] += p.bias[col0 + e];
        }
        if (p.coalesce && p.vec_ok && col0 + 32 <= p.N && tm * 128 + quarter * 32 + 32 <= p.M) {
          // a lane owns a ROW of the warp's 32 x 32 block: stored as it is, one instruction touches 32 lines with
          // 16 bytes each.  Through shared memory eight lanes cover 128 contiguous bytes of one row instead.
          float* const stg = reinterpret_cast<float*>(sbase + kOffEpi + quarter * kEpiStage);
          float* const cblk = (split ? p.C + ((size_t)ks * p.M + tm * 128 + quarter * 32) * p.N
                                     : p.C + (size_t)(tm * 128 + quarter * 32) * p.ldc) + col0;
          const int64_t ldo = split ? p.N : p.ldc;
#pragma unroll
          for (int e = 0; e < 32; e += 4)
            *reinterpret_cast<float4*>(stg + lane * kEpiPitch + e) = make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]);
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = i * 4 + (lane >> 3), c4 = (lane & 7) * 4;
            *reinterpret_cast<float4*>(cblk + (size_t)r * ldo + c4) =
                *reinterpret_cast<const float4*>(stg + r * kEpiPitch + c4);
          }
          if (EPI == kEpiGelu && grow) {
            float* const gblk = p.gelu_out + (size_t)(tm * 128 + quarter * 32) * p.ldc + col0;
            __syncwarp();
#pragma unroll
            for (int e = 0; e < 32; e += 4)
              *reinterpret_cast<float4*>(stg + lane * kEpiPitch + e) =
                  make_float4(gelu_erf(v[e]), gelu_erf(v[e + 1]), gelu_erf(v[e + 2]), gelu_erf(v[e + 3]));
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int r = i * 4 + (lane >> 3), c4 = (lane & 7) * 4;
              *reinterpret_cast<float4*>(gblk + (size_t)r * p.ldc + c4) =
                  *reinterpret_cast<const float4*>(stg + r * kEpiPitch + c4);
            }
          }
          __syncwarp();
        } else if (p.vec_ok && col0 + 32 <= p.N) {
#pragma unroll
          for (int e = 0; e < 32; e += 4) {
            *reinterpret_cast<float4*>(crow + col0 + e) = make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]);
            if (EPI == kEpiGelu && grow)
              *reinterpret_cast<float4*>(grow + col0 + e) =
                  make_float4(gelu_erf(v[e]), gelu_erf(v[e + 1]), gelu_erf(v[e + 2]), gelu_erf(v[e + 3]));
          }
        } else {
          for (int e = 0; e < 32; ++e) {
            if (col0 + e < p.N) {
              crow[col0 + e] = v[e];
              if (EPI == kEpiGelu && grow) grow[col0 + e] = gelu_erf(v[e]);
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc_1cta(tmem_base, 256);
}

// C[m][n] = sum_ks part[ks][m][n] (+ bias[n])
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ part, int ksplit, int M, int N,
                                                            const float* __restrict__ bias, float* __restrict__ C,
                                                            int64_t ldc) {
  const size_t total = (size_t)M * N;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int m = (int)(i / N), n = (int)(i % N);
    float acc = 0.f;
    for (int k = 0; k < ksplit; ++k) acc += part[(size_t)k * total + i];
    if (bias) acc += bias[n];
    C[(size_t)m * ldc + n] = acc;
  }
}

// ---- staging ----------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) amax2d_kernel(const float* __restrict__ src, int R, int C, int64_t lds,
                                                     unsigned int* __restrict__ amax_bits) {
  float a = 0.f;
  const size_t total = (size_t)R * C;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
    a = fmaxf(a, fabsf(src[(i / C) * lds + (i % C)]));
  a = warp_max(a);
  if ((threadIdx.x & 31) == 0 && a > 0.f) atomicMax(amax_bits, __float_as_uint(a));
}

// dense case (lds == C): the matrix is one flat array; four 16-byte loads in flight per thread
__global__ void __launch_bounds__(256) amax_flat_kernel(const float4* __restrict__ src, size_t n4,
                                                        unsigned int* __restrict__ amax_bits) {
  float a = 0.f;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < n4; i += 4 * stride) {
    const float4 v0 = ld_stream(src + i), v1 = ld_stream(src + i + stride), v2 = ld_stream(src + i + 2 * stride),
                 v3 = ld_stream(src + i + 3 * stride);
    a = fmaxf(a, fmaxf(fmaxf(fabsf(v0.x), fabsf(v0.y)), fmaxf(fabsf(v0.z), fabsf(v0.w))));
    a = fmaxf(a, fmaxf(fmaxf(fabsf(v1.x), fabsf(v1.y)), fmaxf(fabsf(v1.z), fabsf(v1.w))));
    a = fmaxf(a, fmaxf(fmaxf(fabsf(v2.x), fabsf(v2.y)), fmaxf(fabsf(v2.z), fabsf(v2.w))));
    a = fmaxf(a, fmaxf(fmaxf(fabsf(v3.x), fabsf(v3.y)), fmaxf(fabsf(v3.z), fabsf(v3.w))));
  }
  for (; i < n4; i += stride) {
    const float4 v = ld_stream(src + i);
    a = fmaxf(a, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
  }
  a = warp_max(a);
  if ((threadIdx.x & 31) == 0 && a > 0.f) atomicMax(amax_bits, __float_as_uint(a));
}

__device__ __forceinline__ float scale_from_amax(float amax) {
  float s = 1.f;
  if (amax > 0.f && amax < INFINITY) {
    int e;
    frexpf(amax, &e);
    s = ldexpf(1.f, 1 - e);  // amax * s in [1, 2)
  }
  return s;
}

// scale slot layout: [0] = s, [1] = 1/s, [2] = amax bits (written by amax2d_kernel)
__global__ void __launch_bounds__(256) stage_kernel(const float* __restrict__ src, int R, int C, int64_t lds,
                                                    int pitch, __half* __restrict__ hi, __half* __restrict__ lo,
                                                    float* __restrict__ scale, const unsigned int* __restrict__ amax_bits) {
  const float s = scale_from_amax(__uint_as_float(amax_bits[0]));
  if (blockIdx.x == 0 && threadIdx.x == 0) { scale[0] = s; scale[1] = 1.f / s; }
  const size_t total = (size_t)R * pitch;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / pitch), c = (int)(i % pitch);
    const float x = c < C ? src[(size_t)r * lds + c] * s : 0.f;
    const __half h = __float2half_rn(x);
    hi[i] = h;
    lo[i] = __float2half_rn(x - __half2float(h));
  }
}

// dst (C rows x R cols, pitch) = src^T, 32 x 32 tiles through shared memory
__global__ void __launch_bounds__(256) stage_T_kernel(const float* __restrict__ src, int R, int C, int64_t lds,
                                                      int pitch, __half* __restrict__ hi, __half* __restrict__ lo,
                                                      float* __restrict__ scale, const unsigned int* __restrict__ amax_bits) {
  __shared__ float tile[32][33];
  const float s = scale_from_amax(__uint_as_float(amax_bits[0]));
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) { scale[0] = s; scale[1] = 1.f / s; }
  const int r0 = blockIdx.x * 32, c0 = blockIdx.y * 32;  // tile of src: rows r0.., cols c0..
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int k = ty; k < 32; k += 8) {
    const int r = r0 + k, c = c0 + tx;
    tile[k][tx] = (r < R && c < C) ? src[(size_t)r * lds + c] * s : 0.f;
  }
  __syncthreads();
  for (int k = ty; k < 32; k += 8) {
    const int orow = c0 + k, ocol = r0 + tx;  // dst[orow][ocol] = src[ocol][orow]
    if (orow < C && ocol < pitch) {
      const float x = tile[tx][k];
      const __half h = __float2half_rn(x);
      hi[(size_t)orow * pitch + ocol] = h;
      lo[(size_t)orow * pitch + ocol] = __float2half_rn(x - __half2float(h));
    }
  }
}

__device__ __forceinline__ void split4(const float4 v, float s, uint2& h, uint2& l) {
  const float x[4] = {v.x * s, v.y * s, v.z * s, v.w * s};
  __half hh[4], ll[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    hh[e] = __float2half_rn(x[e]);
    ll[e] = __float2half_rn(x[e] - __half2float(hh[e]));
  }
  __half2 h01 = __halves2half2(hh[0], hh[1]), h23 = __halves2half2(hh[2], hh[3]);
  __half2 l01 = __halves2half2(ll[0], ll[1]), l23 = __halves2half2(ll[2], ll[3]);
  h = make_uint2(*reinterpret_cast<uint32_t*>(&h01), *reinterpret_cast<uint32_t*>(&h23));
  l = make_uint2(*reinterpret_cast<uint32_t*>(&l01), *reinterpret_cast<uint32_t*>(&l23));
}

// dense, pitch == C == lds: flat 16-byte loads, 8-byte stores to each plane
__global__ void __launch_bounds__(256) stage_flat_kernel(const float4* __restrict__ src, size_t n4,
                                                         uint2* __restrict__ hi, uint2* __restrict__ lo,
                                                         float* __restrict__ scale, const unsigned int* __restrict__ amax_bits) {
  const float s = scale_from_amax(__uint_as_float(amax_bits[0]));
  if (blockIdx.x == 0 && threadIdx.x == 0) { scale[0] = s; scale[1] = 1.f / s; }
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < n4; i += 4 * stride) {
    float4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = ld_stream(src + i + u * stride);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      uint2 h, l;
      split4(v[u], s, h, l);
      hi[i + u * stride] = h;
      lo[i + u * stride] = l;
    }
  }
  for (; i < n4; i += stride) {
    uint2 h, l;
    split4(ld_stream(src + i), s, h, l);
    hi[i] = h;
    lo[i] = l;
  }
}

// transposing stage, 64 x 64 tiles: 16-byte loads along the source rows, 32-byte runs per thread along the
// destination rows (a warp writes eight full 128-byte lines per plane).  Needs R % 64 == 0 handled by guards,
// C % 4 == 0, lds % 4 == 0, pitch % 8 == 0.
__global__ void __launch_bounds__(256) stage_T64_kernel(const float* __restrict__ src, int R, int C, int64_t lds,
                                                        int pitch, __half* __restrict__ hi, __half* __restrict__ lo,
                                                        float* __restrict__ scale, const unsigned int* __restrict__ amax_bits) {
  __shared__ float tile[64][65];
  const float s = scale_from_amax(__uint_as_float(amax_bits[0]));
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) { scale[0] = s; scale[1] = 1.f / s; }
  const int r0 = blockIdx.x * 64, c0 = blockIdx.y * 64;
  const int lc4 = threadIdx.x & 15, lr = threadIdx.x >> 4;  // 16 float4 columns x 16 rows per pass
  float4 v[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = r0 + lr + 16 * i, c = c0 + 4 * lc4;
    v[i] = (r < R && c < C) ? ld_stream(reinterpret_cast<const float4*>(src + (size_t)r * lds + c))
                            : make_float4(0.f, 0.f, 0.f, 0.f);  // C % 4 == 0: a float4 is inside or outside
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float* t = &tile[lr + 16 * i][4 * lc4];
    t[0] = v[i].x * s; t[1] = v[i].y * s; t[2] = v[i].z * s; t[3] = v[i].w * s;
  }
  __syncthreads();
  // destination row = source column c0 + orow; this thread writes 16 consecutive destination columns
  const int orow = threadIdx.x >> 2, seg = threadIdx.x & 3;
  const int drow = c0 + orow, dcol0 = r0 + 16 * seg;
  if (drow >= C || dcol0 >= pitch) return;
  uint32_t hw[8], lw[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float x0 = tile[16 * seg + 2 * j][orow], x1 = tile[16 * seg + 2 * j + 1][orow];
    const __half h0 = __float2half_rn(x0), h1 = __float2half_rn(x1);
    __half2 hh = __halves2half2(h0, h1);
    __half2 ll = __halves2half2(__float2half_rn(x0 - __half2float(h0)), __float2half_rn(x1 - __half2float(h1)));
    hw[j] = *reinterpret_cast<uint32_t*>(&hh);
    lw[j] = *reinterpret_cast<uint32_t*>(&ll);
  }
  uint4* ph = reinterpret_cast<uint4*>(hi + (size_t)drow * pitch + dcol0);
  uint4* pl = reinterpret_cast<uint4*>(lo + (size_t)drow * pitch + dcol0);
  if (dcol0 + 16 <= pitch) {
    ph[0] = make_uint4(hw[0], hw[1], hw[2], hw[3]); ph[1] = make_uint4(hw[4], hw[5], hw[6], hw[7]);
    pl[0] = make_uint4(lw[0], lw[1], lw[2], lw[3]); pl[1] = make_uint4(lw[4], lw[5], lw[6], lw[7]);
  } else {  // pitch % 8 == 0: the row ends after the first half
    ph[0] = make_uint4(hw[0], hw[1], hw[2], hw[3]);
    pl[0] = make_uint4(lw[0], lw[1], lw[2], lw[3]);
  }
}

static size_t plane_elems(int rows, int cols) { return (size_t)rows * round_up((size_t)cols, 8); }

size_t planes_bytes(int rows, int cols) {
  return 2 * round_up(plane_elems(rows, cols) * sizeof(__half), 256) + 256;
}

Planes carve_planes(void* mem, int rows, int cols) {
  Planes pl;
  char* p = static_cast<char*>(mem);
  const size_t one = round_up(plane_elems(rows, cols) * sizeof(__half), 256);
  pl.scale = reinterpret_cast<float*>(p);
  pl.hi = reinterpret_cast<__half*>(p + 256);
  pl.lo = reinterpret_cast<__half*>(p + 256 + one);
  pl.rows = rows;
  pl.cols = cols;
  pl.pitch = (int)round_up((size_t)cols, 8);
  return pl;
}

int amax(const float* src, int R, int C, int64_t lds, unsigned int* slot, cudaStream_t st) {
  MC_REQUIRE(src && slot && R > 0 && C > 0, MC_ERR_BAD_ARG, "amax: bad argument");
  MC_CUDA(cudaMemsetAsync(slot, 0, 4, st));
  const size_t total = (size_t)R * C;
  const int cap = num_sms() * 8;
  if (lds == C && total % 4 == 0 && aligned(src, 16)) {
    int fb = (int)((total / 4 + 1023) / 1024);
    if (fb > cap) fb = cap;
    if (fb < 1) fb = 1;
    amax_flat_kernel<<<fb, 256, 0, st>>>(reinterpret_cast<const float4*>(src), total / 4, slot);
  } else {
    int ab = (int)((total + 255) / 256);
    if (ab > cap) ab = cap;
    amax2d_kernel<<<ab, 256, 0, st>>>(src, R, C, lds, slot);
  }
  MC_LAUNCH_CHECK();
  return MC_OK;
}

int stage(const float* src, int R, int C, int64_t lds, int transpose, const Planes& dst, cudaStream_t st,
          const unsigned int* known_amax) {
  MC_REQUIRE(src && dst.hi && dst.lo && dst.scale, MC_ERR_BAD_ARG, "stage: null pointer");
  MC_REQUIRE(dst.rows == (transpose ? C : R) && dst.cols == (transpose ? R : C), MC_ERR_BAD_ARG,
             "stage: destination planes are %d x %d, expected %d x %d", dst.rows, dst.cols, transpose ? C : R,
             transpose ? R : C);
  const size_t total = (size_t)R * C;
  const int cap = num_sms() * 8;
  const bool flat = lds == C && total % 4 == 0 && aligned(src, 16);
  // max |src|: taken from `known_amax` when a producer kernel (or an earlier staging of the same tensor in the
  // other orientation) already reduced it, else reduced here into the planes' own slot
  const unsigned int* amax_bits = known_amax;
  if (!amax_bits) {
    MC_CUDA(cudaMemsetAsync(dst.scale, 0, 16, st));
    unsigned int* slot = reinterpret_cast<unsigned int*>(dst.scale) + 2;
    if (flat) {
      int fb = (int)((total / 4 + 1023) / 1024);
      if (fb > cap) fb = cap;
      if (fb < 1) fb = 1;
      amax_flat_kernel<<<fb, 256, 0, st>>>(reinterpret_cast<const float4*>(src), total / 4, slot);
    } else {
      int ab = (int)((total + 255) / 256);
      if (ab > cap) ab = cap;
      amax2d_kernel<<<ab, 256, 0, st>>>(src, R, C, lds, slot);
    }
    MC_LAUNCH_CHECK();
    amax_bits = slot;
  }
  if (!transpose) {
    if (flat && dst.pitch == C) {
      int fb = (int)((total / 4 + 1023) / 1024);
      if (fb > cap) fb = cap;
      if (fb < 1) fb = 1;
      stage_flat_kernel<<<fb, 256, 0, st>>>(reinterpret_cast<const float4*>(src), total / 4,
                                            reinterpret_cast<uint2*>(dst.hi), reinterpret_cast<uint2*>(dst.lo), dst.scale,
                                            amax_bits);
    } else {
      const size_t tot = (size_t)R * dst.pitch;
      int nb = (int)((tot + 255) / 256);
      if (nb > cap) nb = cap;
      stage_kernel<<<nb, 256, 0, st>>>(src, R, C, lds, dst.pitch, dst.hi, dst.lo, dst.scale, amax_bits);
    }
  } else if (C % 4 == 0 && lds % 4 == 0 && aligned(src, 16)) {
    dim3 grid((dst.pitch + 63) / 64, (C + 63) / 64);  // covers the padding columns [R, pitch) too
    stage_T64_kernel<<<grid, 256, 0, st>>>(src, R, C, lds, dst.pitch, dst.hi, dst.lo, dst.scale, amax_bits);
  } else {
    // cover the padding columns [R, pitch) too
    dim3 grid((dst.pitch + 31) / 32, (C + 31) / 32);
    stage_T_kernel<<<grid, 256, 0, st>>>(src, R, C, lds, dst.pitch, dst.hi, dst.lo, dst.scale, amax_bits);
  }
  MC_LAUNCH_CHECK();
  return MC_OK;
}

// ---- two weight matrices in one launch -------------------------------------------------------------
struct StageJobDev {
  const float* src;
  int R, C, transpose, pitch;
  __half* hi;
  __half* lo;
  float* scale;
};
__device__ __forceinline__ void stage_job_amax(const StageJobDev& j, unsigned int* slot) {
  float a = 0.f;
  const size_t total = (size_t)j.R * j.C;
  const size_t stride = (size_t)gridDim.x * blockDim.x, t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (total % 4 == 0 && (reinterpret_cast<uintptr_t>(j.src) & 15) == 0) {
    const float4* s4 = reinterpret_cast<const float4*>(j.src);
    for (size_t i = t0; i < total / 4; i += stride) {
      const float4 v = s4[i];
      a = fmaxf(a, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
    }
  } else {
    for (size_t i = t0; i < total; i += stride) a = fmaxf(a, fabsf(j.src[i]));
  }
  a = warp_max(a);
  if ((threadIdx.x & 31) == 0 && a > 0.f) atomicMax(slot, __float_as_uint(a));
}
__device__ __forceinline__ void stage_job_split(const StageJobDev& j, unsigned int amax_bits, float (*tile)[33]) {
  const float s = scale_from_amax(__uint_as_float(amax_bits));
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    j.scale[0] = s; j.scale[1] = 1.f / s;
    reinterpret_cast<unsigned int*>(j.scale)[2] = amax_bits;
  }
  if (!j.transpose) {
    const size_t total = (size_t)j.R * j.pitch;
    const size_t stride = (size_t)gridDim.x * blockDim.x, t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j.pitch == j.C && total % 4 == 0 && (reinterpret_cast<uintptr_t>(j.src) & 15) == 0) {
      const float4* s4 = reinterpret_cast<const float4*>(j.src);
      uint2* h2 = reinterpret_cast<uint2*>(j.hi);
      uint2* l2 = reinterpret_cast<uint2*>(j.lo);
      for (size_t i = t0; i < total / 4; i += stride) {
        uint2 h, l;
        split4(s4[i], s, h, l);
        h2[i] = h;
        l2[i] = l;
      }
    } else {
      for (size_t i = t0; i < total; i += stride) {
        const int r = (int)(i / j.pitch), c = (int)(i % j.pitch);
        const float x = c < j.C ? j.src[(size_t)r * j.C + c] * s : 0.f;
        const __half h = __float2half_rn(x);
        j.hi[i] = h;
        j.lo[i] = __float2half_rn(x - __half2float(h));
      }
    }
    return;
  }
  // transposed: dst (C rows x R cols, pitch) = src^T.  A WARP owns a 32 x 32 tile: lane = source column; it reads its
  // column of 32 source rows (32 independent coalesced loads per warp) and writes the 32 values as 64 contiguous bytes
  // of one destination row per plane - no shared memory, no block barrier, all tiles in flight at once.
  (void)tile;
  const int tr = (j.pitch + 31) / 32, tc = (j.C + 31) / 32;   // tiles along the source rows (incl. padding) / columns
  const int lane = threadIdx.x & 31;
  const int nwarps = gridDim.x * (blockDim.x >> 5), w0 = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  for (int t = w0; t < tr * tc; t += nwarps) {
    const int r0 = (t % tr) * 32, c = (t / tr) * 32 + lane;
    float v[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) v[k] = (r0 + k < j.R && c < j.C) ? j.src[(size_t)(r0 + k) * j.C + c] * s : 0.f;
    if (c >= j.C) continue;
    uint32_t hw[16], lw[16];
#pragma unroll
    for (int k = 0; k < 32; k += 2) {
      const __half h0 = __float2half_rn(v[k]), h1 = __float2half_rn(v[k + 1]);
      const __half2 hh = __halves2half2(h0, h1);
      const __half2 ll = __halves2half2(__float2half_rn(v[k] - __half2float(h0)), __float2half_rn(v[k + 1] - __half2float(h1)));
      hw[k >> 1] = *reinterpret_cast<const uint32_t*>(&hh);
      lw[k >> 1] = *reinterpret_cast<const uint32_t*>(&ll);
    }
    __half* ph = j.hi + (size_t)c * j.pitch + r0;
    __half* pl = j.lo + (size_t)c * j.pitch + r0;
    if (r0 + 32 <= j.pitch && (reinterpret_cast<uintptr_t>(ph) & 15) == 0 && (reinterpret_cast<uintptr_t>(pl) & 15) == 0) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        reinterpret_cast<uint4*>(ph)[u] = make_uint4(hw[4 * u], hw[4 * u + 1], hw[4 * u + 2], hw[4 * u + 3]);
        reinterpret_cast<uint4*>(pl)[u] = make_uint4(lw[4 * u], lw[4 * u + 1], lw[4 * u + 2], lw[4 * u + 3]);
      }
    } else {
      for (int k = 0; k < 32 && r0 + k < j.pitch; ++k) {
        const uint32_t hv = hw[k >> 1], lv = lw[k >> 1];
        const unsigned short hb = (k & 1) ? (unsigned short)(hv >> 16) : (unsigned short)(hv & 0xffffu);
        const unsigned short lb = (k & 1) ? (unsigned short)(lv >> 16) : (unsigned short)(lv & 0xffffu);
        reinterpret_cast<unsigned short*>(ph)[k] = hb;
        reinterpret_cast<unsigned short*>(pl)[k] = lb;
      }
    }
  }
}
// every block is resident (grid <= number of SMs), so a counter barrier between the two phases is safe
__global__ void __launch_bounds__(256) stage_pair_kernel(StageJobDev a, StageJobDev b, unsigned int* sync,
                                                         const unsigned int* known, unsigned int* amax_out) {
  __shared__ float tile[32][33];
  unsigned int ba, bb;
  if (known) {   // both maxima were reduced by an earlier call on the same (unchanged) matrices: no barrier needed
    ba = known[0];
    bb = known[1];
  } else {
    stage_job_amax(a, sync + 1);
    stage_job_amax(b, sync + 2);
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      atomicAdd(sync, 1u);
      while (*reinterpret_cast<volatile unsigned int*>(sync) < gridDim.x) __nanosleep(20);
      __threadfence();
    }
    __syncthreads();
    ba = *reinterpret_cast<volatile unsigned int*>(sync + 1);
    bb = *reinterpret_cast<volatile unsigned int*>(sync + 2);
    if (amax_out && blockIdx.x == 0 && threadIdx.x == 0) { amax_out[0] = ba; amax_out[1] = bb; }
  }
  stage_job_split(a, ba, tile);
  stage_job_split(b, bb, tile);
}

int stage_pair(const StageJob& a, const StageJob& b, unsigned int* sync, cudaStream_t st, const unsigned int* known,
               unsigned int* amax_out) {
  const StageJob* jobs[2] = {&a, &b};
  StageJobDev d[2];
  for (int k = 0; k < 2; ++k) {
    const StageJob& j = *jobs[k];
    MC_REQUIRE(j.src && j.dst.hi && j.dst.lo && j.dst.scale && sync, MC_ERR_BAD_ARG, "stage_pair: null pointer");
    MC_REQUIRE(j.dst.rows == (j.transpose ? j.C : j.R) && j.dst.cols == (j.transpose ? j.R : j.C), MC_ERR_BAD_ARG,
               "stage_pair: destination planes are %d x %d", j.dst.rows, j.dst.cols);
    d[k] = StageJobDev{j.src, j.R, j.C, j.transpose, j.dst.pitch, j.dst.hi, j.dst.lo, j.dst.scale};
  }
  if (!known) MC_CUDA(cudaMemsetAsync(sync, 0, 16, st));
  stage_pair_kernel<<<num_sms(), 256, 0, st>>>(d[0], d[1], sync, known, amax_out);
  MC_LAUNCH_CHECK();
  return MC_OK;
}

// ---- host side of the GEMM ---------------------------------------------------------------------
// Split K when there are fewer tiles than SMs (the weight-gradient GEMMs: K is the batch).  jobs = tiles x ksplit
// should fill whole waves of the persistent grid: pick the wave count (1..3) with the best fill, fewer waves on ties
// (less partial traffic).  4 tiles -> 37 splits (148 jobs, one full wave); 32 tiles -> 9 splits (288 of 296).
static int choose_ksplit(int M, int N, int K) {
  const int tiles = ((M + 127) / 128) * ((N + 127) / 128);
  const int chunks = (K + 63) / 64;
  const int sms = num_sms();
  if (tiles >= sms) return 1;
  int best = 1;
  double best_fill = (double)tiles / sms;
  for (int w = 1; w <= 3; ++w) {
    int ks = (w * sms) / tiles;
    if (ks > chunks) ks = chunks;
    if (ks > 64) ks = 64;
    if (ks < 1) ks = 1;
    const int jobs = tiles * ks;
    const int waves = (jobs + sms - 1) / sms;
    const double fill = (double)jobs / ((double)waves * sms);
    if (fill > best_fill + 0.02) { best_fill = fill; best = ks; }
  }
  return best;
}

size_t gemm_workspace_bytes(int M, int N, int K) {
  const int ks = choose_ksplit(M, N, K);
  return ks > 1 ? round_up((size_t)ks * M * N * sizeof(float), 256) : 256;
}

int gemm(const Planes& A, const Planes& B, int M, int N, int K, const GemmOut& out, int epilogue, void* ws,
         size_t ws_bytes, cudaStream_t st) {
  MC_REQUIRE(A.rows == M && A.cols == K && B.rows == N && B.cols == K, MC_ERR_BAD_ARG,
             "tc gemm: operand shapes (%d x %d) . (%d x %d)^T do not match M=%d N=%d K=%d", A.rows, A.cols, B.rows,
             B.cols, M, N, K);
  MC_REQUIRE(out.C != nullptr, MC_ERR_BAD_ARG, "tc gemm: null output");
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
  int rc;
  const CUtensorMapDataType f16 = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  const CUtensorMapSwizzle sw = CU_TENSOR_MAP_SWIZZLE_128B;
  if ((rc = make_map(&ma_hi, f16, A.hi, A.rows, A.cols, A.pitch * sizeof(__half), 64, 128, sw))) return rc;
  if ((rc = make_map(&ma_lo, f16, A.lo, A.rows, A.cols, A.pitch * sizeof(__half), 64, 128, sw))) return rc;
  if ((rc = make_map(&mb_hi, f16, B.hi, B.rows, B.cols, B.pitch * sizeof(__half), 64, 128, sw))) return rc;
  if ((rc = make_map(&mb_lo, f16, B.lo, B.rows, B.cols, B.pitch * sizeof(__half), 64, 128, sw))) return rc;
  GemmParams p;
  p.M = M; p.N = N; p.K = K;
  p.tiles_m = (M + 127) / 128;
  p.tiles_n = (N + 127) / 128;
  p.chunks_total = (K + 63) / 64;
  p.ksplit = choose_ksplit(M, N, K);
  if (epilogue == kEpiGelu) p.ksplit = 1;
  p.chunks_per_split = (p.chunks_total + p.ksplit - 1) / p.ksplit;
  p.ksplit = (p.chunks_total + p.chunks_per_split - 1) / p.chunks_per_split;  // no empty splits
  p.scale_a = A.scale;
  p.scale_b = B.scale;
  p.bias = out.bias;
  p.gelu_out = out.gelu_out;
  if (p.ksplit > 1) {
    MC_REQUIRE(ws && ws_bytes >= (size_t)p.ksplit * M * N * sizeof(float), MC_ERR_WORKSPACE,
               "tc gemm: split-K workspace too small");
    p.C = static_cast<float*>(ws);
    p.ldc = N;
    p.vec_ok = (N % 4 == 0) && aligned(ws, 16);
  } else {
    p.C = out.C;
    p.ldc = out.ldc;
    p.vec_ok = (out.ldc % 4 == 0) && aligned(out.C, 16) && (!out.gelu_out || aligned(out.gelu_out, 16));
  }
  // epilogue stores through the per-warp transpose (image head fwd+bwd 0.955 -> 0.893 ms, profiles/r01j_head_coalesce_ab.log);
  // MAE_CLIP_GEMM_COALESCE=0 restores the per-lane row stores (A/B switch)
  static const bool coalesce_off = getenv("MAE_CLIP_GEMM_COALESCE") != nullptr && getenv("MAE_CLIP_GEMM_COALESCE")[0] == '0';
  p.coalesce = coalesce_off ? 0 : 1;
  const int njobs = p.tiles_m * p.tiles_n * p.ksplit;
  const int grid = njobs < num_sms() ? njobs : num_sms();
  if (epilogue == kEpiGelu) {
    MC_CUDA(ensure_dynamic_smem<gemm_kernel<kEpiGelu>>(kSmem));
    gemm_kernel<kEpiGelu><<<grid, kThreads, kSmem, st>>>(ma_hi, ma_lo, mb_hi, mb_lo, p);
  } else {
    MC_CUDA(ensure_dynamic_smem<gemm_kernel<kEpiPlain>>(kSmem));
    gemm_kernel<kEpiPlain><<<grid, kThreads, kSmem, st>>>(ma_hi, ma_lo, mb_hi, mb_lo, p);
  }
  MC_LAUNCH_CHECK();
  if (p.ksplit > 1) {
    const size_t total = (size_t)M * N;
    int nb = (int)((total + 255) / 256);
    const int cap = num_sms() * 8;
    if (nb > cap) nb = cap;
    splitk_reduce_kernel<<<nb, 256, 0, st>>>(static_cast<const float*>(ws), p.ksplit, M, N, out.bias, out.C, out.ldc);
    MC_LAUNCH_CHECK();
  }
  return MC_OK;
}

}  // namespace tcg
}  // namespace mc

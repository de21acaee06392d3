// ProjectionHead GEMMs on the 5th-gen tensor cores, second generation (reference: /root/reference modules.py:63-75
// and their autograd).  What round 1 measured (profiles/r01_ncu_summary.md section 8): 36% of a head went into staging
// fp16 hi/lo planes of ACTIVATIONS in HBM, and the 128 x 128 single-CTA tiles were bound by shared-memory bandwidth
// (every MMA read 8 KB of operands from shared memory; three passes per K step).  Here:
//
//   * a CTA PAIR (cluster of 2, tcgen05 cta_group::2, M = 256: 128 rows per CTA) owns a tile; the B operand is split
//     between the two CTAs, so each feeds only HALF of it from its shared memory;
//   * the activation operand A arrives as fp32 tiles by TMA; a CONVERTER warpgroup (thread = row) splits it into fp16
//     hi / lo and writes it straight into TENSOR MEMORY (tcgen05.st); the MMAs take A from TMEM (the .ts form), so the
//     converted activation never touches shared memory again and is never staged in HBM;
//   * the epilogue owns whole rows (TMEM lane = row), so bias + GELU, dropout + residual + LayerNorm (N = 256 is one
//     tile row) and the GELU backward are fused into the GEMM that produces their input;
//   * the weight-gradient GEMMs (K = batch) read BOTH operands as fp32 row-major tiles and transpose them in the
//     converter (registers), so no transposed plane is staged either.
//
// Three kernels share the helpers below:
//   row_kernel   out(M, 256)  = A(M, K) W(256, K)^T     x Wp^T (+bias, GELU) ; h Wf^T (+bias, dropout, residual, LN) ;
//                                                       dy Wf (GELU backward)
//   ares_kernel  C(M, N)      = A(M, K<=256) W(N, K)^T  dx = dp Wp: the converted row block stays RESIDENT in TMEM
//   tt_kernel    C(256, N)    = A(K, 256)^T B(K, N)     dWf = dy^T h, dWp = dp^T x (split-K, deterministic reduce)
// Precision as in gemm_tc.cu: x = (hi + lo) / s with a power-of-two s per matrix; hi*hi + hi*lo + lo*hi into fp32.
#include <assert.h>
#include <stdlib.h>

#include "head_tc.cuh"
#include "tc_launch.cuh"
#include "tc_ptx.cuh"

namespace mc {
namespace hg {

using namespace ptx;

bool supported(int P) { return P == 256; }

// ------------------------------------------------------------------------------------------------ extra PTX
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st32f(uint32_t taddr, const float* v) {
  const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
  tmem_st16(taddr, r);
  tmem_st16(taddr + 16, r + 16);
}
// 32 lanes x 16 columns of 32-bit
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// D[tmem] (+)= A[tmem] * B[smem]^T over the CTA pair (A: lane = row, 32-bit columns hold two consecutive K elements)
__device__ __forceinline__ void mma_f16_pair_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                                uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float lds32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

__device__ __forceinline__ float scale_from_amax_bits(unsigned int bits) {
  const float amax = __uint_as_float(bits);
  float s = 1.f;
  if (amax > 0.f && amax < INFINITY) {
    int e;
    frexpf(amax, &e);
    s = ldexpf(1.f, 1 - e);  // amax * s in [1, 2)
  }
  return s;
}

// Was a power-of-two scale taken from `stale` (max |A| of an EARLIER call) safe for data whose true maximum is `live`?
// stale * s lies in [1, 2), so live * s estimates live / stale within a factor of two.  Safe = no fp16 overflow
// (live * s < 2^14) and enough of the fp16 range left for the lo plane (live * s >= 2^-5; an all-zero A is always safe).
// A subnormal `stale` is never trusted: its scale 2^(1 - e) can pass 2^127 (+inf), and 0 * inf turns an all-zero A to NaN.
__device__ __forceinline__ bool scale_window_ok(unsigned int stale_bits, unsigned int live_bits) {
  const float st = __uint_as_float(stale_bits), lv = __uint_as_float(live_bits);
  if (!(st >= 1.17549435e-38f) || !(st < INFINITY) || !(lv < INFINITY)) return false;   // FLT_MIN
  if (lv == 0.f) return true;
  const float r = lv * scale_from_amax_bits(stale_bits);
  return r < 16384.f && r >= 0.03125f;
}

// two scaled fp32 values -> packed fp16 hi pair and packed fp16 lo pair (lo = fp16(x - hi), exact difference)
__device__ __forceinline__ void split2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(x0, x1);
  const float2 b = __half22float2(h);
  const __half2 l = __floats2half2_rn(x0 - b.x, x1 - b.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

// exact-erf GELU (modules.py:64, nn.GELU()) and its derivative through ONE exponential: Abramowitz-Stegun 7.1.26,
//   erf(u) = 1 - (a1 t + ... + a5 t^5) e^{-u^2}, t = 1 / (1 + 0.3275911 u), u >= 0,  |error| <= 1.5e-7,
// with u = |x| / sqrt(2), so that e^{-u^2} = e^{-x^2/2} is also the Gaussian of the derivative.  erff() costs ~70
// instructions with a divergent branch; this is ~18 and keeps the epilogues inside the instruction cache.
__device__ __forceinline__ void gelu_core(float x, float& cdf, float& gauss) {
  const float ax = fabsf(x);
  const float t = __frcp_rn(fmaf(0.3275911f * 0.70710678118654752f, ax, 1.f));
  gauss = exp2f(-0.72134752044448170f * x * x);   // e^{-x^2/2}
  float pl = fmaf(1.061405429f, t, -1.453152027f);
  pl = fmaf(pl, t, 1.421413741f);
  pl = fmaf(pl, t, -0.284496736f);
  pl = fmaf(pl, t, 0.254829592f);
  const float half_tail = 0.5f * pl * t * gauss;    // (1 - erf(u)) / 2
  cdf = x >= 0.f ? 1.f - half_tail : half_tail;
}
__device__ __forceinline__ float gelu_as(float x) {
  float cdf, g;
  gelu_core(x, cdf, g);
  return x * cdf;
}
__device__ __forceinline__ float gelu_grad_as(float x) {
  float cdf, g;
  gelu_core(x, cdf, g);
  return fmaf(x * 0.3989422804014327f, g, cdf);
}

// ------------------------------------------------------------------------------------------------ epilogue I/O
// A warp owns a 32 x 32 block (lane = row).  Global traffic goes through a per-warp shared-memory transpose so that
// eight lanes cover 128 contiguous bytes of one row (a lane-per-row access touches 32 lines with 16 bytes each).
constexpr int kStgPitch = 36;                   // floats: 32 + 4 keeps the 16-byte accesses conflict-free
constexpr int kStgBytes = 32 * kStgPitch * 4;   // 4608

__device__ __forceinline__ void block_store(float* stg, int lane, const float* v, float* g, int64_t ld, int rows_valid,
                                            int cols_valid) {
#pragma unroll
  for (int e = 0; e < 32; e += 4)
    *reinterpret_cast<float4*>(stg + lane * kStgPitch + e) = make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]);
  __syncwarp();
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = i * 4 + (lane >> 3), c4 = (lane & 7) * 4;
    if (r < rows_valid && c4 + 4 <= cols_valid)
      *reinterpret_cast<float4*>(g + (size_t)r * ld + c4) = *reinterpret_cast<const float4*>(stg + r * kStgPitch + c4);
  }
  __syncwarp();
}
// same, and returns the sum over the block's rows of column `lane` (rows beyond rows_valid must hold zeros)
__device__ __forceinline__ float block_store_colsum(float* stg, int lane, const float* v, float* g, int64_t ld,
                                                    int rows_valid) {
#pragma unroll
  for (int e = 0; e < 32; e += 4)
    *reinterpret_cast<float4*>(stg + lane * kStgPitch + e) = make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]);
  __syncwarp();
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = i * 4 + (lane >> 3), c4 = (lane & 7) * 4;
    if (r < rows_valid)
      *reinterpret_cast<float4*>(g + (size_t)r * ld + c4) = *reinterpret_cast<const float4*>(stg + r * kStgPitch + c4);
  }
  float cs = 0.f;
#pragma unroll
  for (int r = 0; r < 32; ++r) cs += stg[r * kStgPitch + lane];
  __syncwarp();
  return cs;
}
__device__ __forceinline__ void block_load(float* stg, int lane, const float* g, int64_t ld, int rows_valid, float* v) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = i * 4 + (lane >> 3), c4 = (lane & 7) * 4;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < rows_valid) x = ld_stream(reinterpret_cast<const float4*>(g + (size_t)r * ld + c4));
    *reinterpret_cast<float4*>(stg + r * kStgPitch + c4) = x;
  }
  __syncwarp();
#pragma unroll
  for (int e = 0; e < 32; e += 4) {
    const float4 x = *reinterpret_cast<const float4*>(stg + lane * kStgPitch + e);
    v[e] = x.x; v[e + 1] = x.y; v[e + 2] = x.z; v[e + 3] = x.w;
  }
  __syncwarp();
}

// ------------------------------------------------------------------------------------------------ converters
// fp32 tile [128 rows][32 k] as TMA wrote it with SWIZZLE_128B (row = 128 bytes, 16-byte chunk j of row r at
// j ^ (r & 7)) -> 16 packed hi words + 16 packed lo words of row `row` (two consecutive k per word), scaled by s
template <bool LO>
__device__ __forceinline__ void convert_row32(uint32_t box, int row, float s, uint32_t* hw, uint32_t* lw, float& amax) {
  const uint32_t rbase = box + (uint32_t)row * 128u;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 f = lds128(rbase + (uint32_t)((j ^ (row & 7)) << 4));
    amax = fmaxf(amax, fmaxf(fmaxf(fabsf(f.x), fabsf(f.y)), fmaxf(fabsf(f.z), fabsf(f.w))));
    uint32_t l0, l1;
    split2(f.x * s, f.y * s, hw[2 * j], l0);
    split2(f.z * s, f.w * s, hw[2 * j + 1], l1);
    if (LO) { lw[2 * j] = l0; lw[2 * j + 1] = l1; }
  }
}
// fp32 tile [32 k][128 cols] (no swizzle, 512-byte rows) -> the 32 k values of column `col` as 16 hi + 16 lo words
template <bool LO>
__device__ __forceinline__ void convert_col32(uint32_t box, int col, float s, uint32_t* hw, uint32_t* lw) {
  const uint32_t cbase = box + (uint32_t)col * 4u;
#pragma unroll
  for (int kk = 0; kk < 32; kk += 2) {
    const float x0 = lds32(cbase + (uint32_t)kk * 512u) * s, x1 = lds32(cbase + (uint32_t)(kk + 1) * 512u) * s;
    uint32_t l;
    split2(x0, x1, hw[kk >> 1], l);
    if (LO) lw[kk >> 1] = l;
  }
}

// ================================================================================================ row kernel
namespace rowk {
constexpr int kThreads = 480;   // warp 0 W producer, warp 1 MMA, warps 2-5 converter, warps 6-13 epilogue, warp 14 A producer
// Two shared-memory / tensor-memory plans (template flag ASMEM):
//   long K (x Wp^T)       A in TMEM (the MMAs then read only W from shared memory: with A there too the three passes
//                         would need more shared-memory bandwidth than an SM has), ONE accumulator: [0, 256) + A stages
//                         at 256 + 64 s; rings: 5 source boxes, 3 W slots
//   K <= 256 (h Wf^T, dy Wf)  these are bound by their epilogues (HBM traffic of the fused LayerNorm / GELU backward),
//                         so the accumulator is DOUBLE-buffered ([0, 256), [256, 512)): the epilogue of a tile runs
//                         under the loads, conversion and MMAs of the next; A goes to shared memory instead
//                         (2 stages of hi + lo), rings: 3 source boxes, 2 W slots
constexpr int kSrcSlot = 16384;                        // fp32 A: one swizzled box [128 rows][32 k]; a 64-k chunk = 2 slots
constexpr int kBSlot = 32768;                          // W half of this CTA: hi [128 rows][64 k] + lo
constexpr int kASlot = 32768;                          // ASMEM: converted A of this CTA: hi [128 rows][64 k] + lo
constexpr int kOffSrc = 0;
constexpr int kOffStg = 180224;                        // both plans fill [0, 180224) with their rings
constexpr int kOffLnx = kOffStg + 8 * kStgBytes;       // 217088: [2 exchanges][2 halves][128 rows] floats
constexpr int kOffBar = kOffLnx + 8 * 128 * 4;         // 221184 (the LayerNorm exchange uses the first 2 KB; the
                                                       // GELU-backward column sums 8 warps x 128 floats)
constexpr int kSmem = kOffBar + 256 + 1024;
enum Bar { kSrcFull = 0, kSrcEmpty = 5, kAFull = 10, kAEmpty = 12, kBFull = 14, kBEmpty = 17, kAccFull = 20, kAccEmpty = 22,
           kNumBars = 24 };
constexpr uint32_t kACol = 256;       // !ASMEM: A stage s at TMEM columns 256 + 64 s (hi: 32 columns, lo: 32)
}  // namespace rowk

struct RowParams {
  int M, K, n_tiles, chunks;
  const unsigned int* a_amax;
  const float* w_scale;   // {s, 1/s}
  const float* bias;
  float* out0;
  float* out1;
  const float* in0;
  const float* in1;
  const uint8_t* keep;
  float drop_scale, eps;
  const float* gamma;
  const float* beta;
  float* mean;
  float* rstd;
  unsigned int* out_amax;
  float* colpart;
  // scale source of A (see head_tc.cuh "scale protocol"): vmode 0 = *a_amax; 1 = first attempt with the PREVIOUS call's
  // max |A| (*v_stale) while the true one is reduced into *a_live; 2 = redo: return at once when the stale scale was
  // inside the safe window, else run again with *v_live; 3 = consumer of an operand produced under that protocol:
  // *a_amax when the first attempt was valid, else *a_alt (and *amax_publish := the one chosen)
  int vmode;
  const unsigned int* a_alt;
  const unsigned int* v_stale;
  const unsigned int* v_live;
  unsigned int* a_live;
  unsigned int* amax_publish;
  unsigned long long* dbg;   // optional timeline of pair 0's leader CTA (globaltimer ns), tools/head_timeline.py
};
__device__ __forceinline__ unsigned long long gtime_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
#define HG_MARK(idx)                                                              \
  do {                                                                            \
    if (p.dbg && blockIdx.x == 0 && lane == 0) p.dbg[(idx)] = gtime_ns();         \
  } while (0)

// The epilogue works on a warp's 32 x 32 block in two thread mappings: ROW (lane = row: what tcgen05.ld delivers, and
// what row reductions want) and PIECE (iteration i of 8: row 4 i + (lane >> 3), columns 4 (lane & 7) .. +3: eight lanes
// cover 128 contiguous bytes of one row, so global loads / stores are coalesced and can all be issued before first use).
// The accumulator block crosses from one mapping to the other through the warp's staging buffer.
__device__ __forceinline__ void stg_put_rows(float* stg, int lane, const float* v) {
#pragma unroll
  for (int e = 0; e < 32; e += 4)
    *reinterpret_cast<float4*>(stg + lane * kStgPitch + e) = make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]);
}
__device__ __forceinline__ void stg_get_rows(const float* stg, int lane, float* v) {
#pragma unroll
  for (int e = 0; e < 32; e += 4) {
    const float4 x = *reinterpret_cast<const float4*>(stg + lane * kStgPitch + e);
    v[e] = x.x; v[e + 1] = x.y; v[e + 2] = x.z; v[e + 3] = x.w;
  }
}
// accumulator block (32 columns of this lane's row) -> staging buffer, 16 columns at a time (register pressure)
__device__ __forceinline__ void tmem_to_stg_rows(uint32_t taddr, float* stg, int lane) {
#pragma unroll
  for (int hcol = 0; hcol < 32; hcol += 16) {
    float v[16];
    tmem_ld16(taddr + hcol, v);
    tmem_ld_wait();
#pragma unroll
    for (int e = 0; e < 16; e += 4)
      *reinterpret_cast<float4*>(stg + lane * kStgPitch + hcol + e) = make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]);
  }
}
__device__ __forceinline__ float amax4(float a, const float4 v) {
  return fmaxf(a, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
}

template <int EPI, int PASSES, bool ASMEM>
__global__ void __launch_bounds__(rowk::kThreads, 1)
row_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_wh,
           const __grid_constant__ CUtensorMap map_wl, const RowParams p) {
  using namespace rowk;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* const sbase = smem_raw + (base - raw);
  const uint32_t bar0 = base + kOffBar;
  auto bar = [&](int i) -> uint32_t { return bar0 + 8u * i; };
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(sbase + kOffBar + 8 * kNumBars);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair_id = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  constexpr bool kLo = PASSES == 3;
  constexpr int kSrcSlots = ASMEM ? 3 : 5, kBSlots = ASMEM ? 2 : 3, kNAcc = ASMEM ? 2 : 1;
  constexpr int kOffA = kSrcSlots * kSrcSlot;                          // ASMEM only: 2 x kASlot
  constexpr int kOffB = ASMEM ? kOffA + 2 * kASlot : kSrcSlots * kSrcSlot;
  static_assert(kOffB + kBSlots * kBSlot == kOffStg, "ring plan does not fill the ring region");

  // scale source of A (uniform over the whole grid; decided before any barrier so that a redo launch can leave at once)
  unsigned int a_bits;
  if (p.vmode == 0) {
    a_bits = *p.a_amax;
  } else if (p.vmode == 1) {
    a_bits = *p.v_stale;
  } else {
    const bool ok = scale_window_ok(*p.v_stale, *p.v_live);
    if (p.vmode == 2) {
      if (ok) return;
      a_bits = *p.v_live;
    } else {
      a_bits = ok ? *p.a_amax : *p.a_alt;
      if (p.amax_publish && blockIdx.x == 0 && threadIdx.x == 0) *p.amax_publish = a_bits;
    }
  }

  if (threadIdx.x == 0) {
    for (int s = 0; s < kSrcSlots; ++s) { mbar_init(bar(kSrcFull + s), 1); mbar_init(bar(kSrcEmpty + s), 4); }
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar(kAFull + s), 8);     // one lane of each converter warp, both CTAs (leader's copy is the one used)
      mbar_init(bar(kAEmpty + s), 1);
    }
    for (int s = 0; s < kBSlots; ++s) { mbar_init(bar(kBFull + s), 1); mbar_init(bar(kBEmpty + s), 1); }
    for (int b = 0; b < kNAcc; ++b) {
      mbar_init(bar(kAccFull + b), 1);
      mbar_init(bar(kAccEmpty + b), 16);   // one lane of each epilogue warp, both CTAs
    }
    fence_mbar_init();
    prefetch_tmap(&map_a); prefetch_tmap(&map_wh); prefetch_tmap(&map_wl);
  }
  if (warp == 1) {
    tmem_alloc_pair(smem_u32(tmem_slot), 512);
    tmem_relinquish_pair();
  }
  if (warp == 0) HG_MARK(0);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (warp == 0) HG_MARK(1);

  if (warp == 0) {
    // ============================================================ W producer (both CTAs: own half of the W rows)
    if (elect_one()) {
      uint32_t it = 0;
      for (int tile = pair_id; tile < p.n_tiles; tile += npairs) {
        for (int c = 0; c < p.chunks; ++c, ++it) {
          const uint32_t slot = it % kBSlots, par = (it / kBSlots) & 1;
          mbar_wait(bar(kBEmpty + slot), par ^ 1);
          const uint32_t fb = bar(kBFull + slot);
          if (leader) mbar_arrive_expect_tx(fb, (kLo ? 2u : 1u) * 2u * 16384u);
          const uint32_t sb = base + kOffB + slot * kBSlot;
          tma_load_2d_pair(sb, &map_wh, fb, c * 64, (int)rank * 128);
          if (kLo) tma_load_2d_pair(sb + 16384, &map_wl, fb, c * 64, (int)rank * 128);
        }
      }
    }
    __syncwarp();
  } else if (warp == 14) {
    // ============================================================ A producer: fp32 rows of this CTA, 32-k boxes
    if (elect_one()) {
      uint32_t h = 0;
      for (int tile = pair_id; tile < p.n_tiles; tile += npairs) {
        const int row0 = tile * 256 + (int)rank * 128;
        for (int c = 0; c < 2 * p.chunks; ++c, ++h) {
          const uint32_t slot = h % kSrcSlots, par = (h / kSrcSlots) & 1;
          mbar_wait(bar(kSrcEmpty + slot), par ^ 1);
          const uint32_t fb = bar(kSrcFull + slot);
          mbar_arrive_expect_tx(fb, (uint32_t)kSrcSlot);
          tma_load_2d(base + kOffSrc + slot * kSrcSlot, &map_a, fb, c * 32, row0);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ============================================================ MMA issuer (leader CTA, one elected lane)
    if (leader && elect_one()) {
      constexpr uint32_t idesc = idesc_f16(256, 256);
      uint32_t it = 0, tt = 0;
      for (int tile = pair_id; tile < p.n_tiles; tile += npairs, ++tt) {
        const uint32_t buf = ASMEM ? (tt & 1) : 0u, use = ASMEM ? (tt >> 1) : tt;
        mbar_wait(bar(kAccEmpty + buf), (use & 1) ^ 1);   // the epilogue drained this accumulator buffer
        tc_fence_after();
        const uint32_t td = tmem_base + buf * 256;
        if (tt < 2 && p.dbg && blockIdx.x == 0) p.dbg[2 + 4 * tt] = gtime_ns();
        for (int c = 0; c < p.chunks; ++c, ++it) {
          const uint32_t s = it & 1, par = (it >> 1) & 1;
          const uint32_t bs = it % kBSlots, bp = (it / kBSlots) & 1;
          mbar_wait(bar(kAFull + s), par);
          if (c == 0 && tt < 2 && p.dbg && blockIdx.x == 0) p.dbg[3 + 4 * tt] = gtime_ns();
          mbar_wait(bar(kBFull + bs), bp);
          if (c == 0 && tt < 2 && p.dbg && blockIdx.x == 0) p.dbg[4 + 4 * tt] = gtime_ns();
          tc_fence_after();
          const uint32_t sb = base + kOffB + bs * kBSlot;
          const uint64_t bh = smem_desc_sw128(sb), bl = smem_desc_sw128(sb + 16384);
          if (ASMEM) {
            const uint32_t sa = base + kOffA + s * kASlot;
            const uint64_t ah = smem_desc_sw128(sa), al = smem_desc_sw128(sa + 16384);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              const uint32_t acc = (c > 0 || ks > 0) ? 1u : 0u;
              mma_f16_pair(td, desc_advance_k(ah, ks), desc_advance_k(bh, ks), idesc, acc);
              if (kLo) {
                mma_f16_pair(td, desc_advance_k(ah, ks), desc_advance_k(bl, ks), idesc, 1u);
                mma_f16_pair(td, desc_advance_k(al, ks), desc_advance_k(bh, ks), idesc, 1u);
              }
            }
          } else {
            const uint32_t ah = tmem_base + kACol + s * 64, al = ah + 32;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              const uint32_t acc = (c > 0 || ks > 0) ? 1u : 0u;
              mma_f16_pair_ts(td, ah + ks * 8, desc_advance_k(bh, ks), idesc, acc);
              if (kLo) {
                mma_f16_pair_ts(td, ah + ks * 8, desc_advance_k(bl, ks), idesc, 1u);
                mma_f16_pair_ts(td, al + ks * 8, desc_advance_k(bh, ks), idesc, 1u);
              }
            }
          }
          mma_commit_pair(bar(kAEmpty + s), 3);
          mma_commit_pair(bar(kBEmpty + bs), 3);
        }
        mma_commit_pair(bar(kAccFull + buf), 3);
        if (tt < 2 && p.dbg && blockIdx.x == 0) p.dbg[5 + 4 * tt] = gtime_ns();
      }
    }
    __syncwarp();
  } else if (warp < 6) {
    // ============================================================ converter: fp32 rows -> fp16 hi / lo in tensor memory
    const int q = warp & 3, row = q * 32 + lane;
    const uint32_t lane_field = (uint32_t)(q * 32) << 16;
    const float s = scale_from_amax_bits(a_bits);
    float amax = 0.f;
    uint32_t it = 0;
    for (int tile = pair_id; tile < p.n_tiles; tile += npairs) {
      for (int c = 0; c < p.chunks; ++c, ++it) {
        const uint32_t as = it & 1, ap = (it >> 1) & 1;
        mbar_wait(bar(kAEmpty + as), ap ^ 1);   // the MMAs that read this TMEM stage have completed
        tc_fence_after();
        const uint32_t ta = tmem_base + lane_field + kACol + as * 64;
        const uint32_t arow = base + kOffA + as * kASlot + (uint32_t)row * 128u;
#pragma unroll
        for (int bx = 0; bx < 2; ++bx) {
          const uint32_t h = 2 * it + bx, ss = h % kSrcSlots, sp = (h / kSrcSlots) & 1;
          mbar_wait(bar(kSrcFull + ss), sp);
          uint32_t hw[16], lw[16];
          convert_row32<kLo>(base + kOffSrc + ss * kSrcSlot, row, s, hw, lw, amax);
          __syncwarp();
          if (lane == 0) mbar_arrive_local(bar(kSrcEmpty + ss));   // the box is in registers
          if (ASMEM) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const uint32_t off = (uint32_t)(((4 * bx + i) ^ (row & 7)) << 4);
              sts128(arow + off, hw[4 * i], hw[4 * i + 1], hw[4 * i + 2], hw[4 * i + 3]);
              if (kLo) sts128(arow + 16384 + off, lw[4 * i], lw[4 * i + 1], lw[4 * i + 2], lw[4 * i + 3]);
            }
          } else {
            tmem_st16(ta + bx * 16, hw);
            if (kLo) tmem_st16(ta + 32 + bx * 16, lw);
          }
        }
        if (ASMEM) {
          fence_proxy_async_smem();
        } else {
          tmem_st_wait();
          tc_fence_before();
        }
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(bar(kAFull + as), 0);
      }
    }
    if (p.vmode == 1 && p.a_live) {   // the true max |A| (rows beyond M and columns beyond K were zero-filled by TMA)
      amax = warp_max(amax);
      if (lane == 0 && amax > 0.f) atomicMax(p.a_live, __float_as_uint(amax));
    }
  } else {
    // ============================================================ epilogue: 8 warps = 4 TMEM lane quarters x 2 column halves
    const int we = warp - 6, q = warp & 3, hf = we >> 2;
    const int lrow = q * 32 + lane;
    const uint32_t tacc0 = tmem_base + ((uint32_t)(q * 32) << 16);
    float* const stg = reinterpret_cast<float*>(sbase + kOffStg + we * kStgBytes);
    float* const lnx = reinterpret_cast<float*>(sbase + kOffLnx);
    const float inv = (1.f / scale_from_amax_bits(a_bits)) * p.w_scale[1];
    const int pr = lane >> 3, pc = (lane & 7) * 4;   // piece mapping: row 4 i + pr, columns pc .. pc + 3
    float amax = 0.f;
    float* const colsm = lnx + we * 128;   // kEpiGeluBwd: this warp's running column sums (its 128 columns)
    if (EPI == kEpiGeluBwd) {
      for (int i = lane; i < 128; i += 32) colsm[i] = 0.f;
      __syncwarp();
    }
    uint32_t tt = 0;
    for (int tile = pair_id; tile < p.n_tiles; tile += npairs, ++tt) {
      const int blk_row0 = tile * 256 + (int)rank * 128 + q * 32;
      const int grow = blk_row0 + lane;
      const int rows_valid = p.M - blk_row0;   // may be <= 0 or > 32
      const bool row_ok = grow < p.M;
      const uint32_t buf = ASMEM ? (tt & 1) : 0u, full_par = (ASMEM ? (tt >> 1) : tt) & 1;
      const uint32_t tacc = tacc0 + buf * 256;
      // global address of this lane's piece 0 of slab 0 (column half hf) in a (M, 256) tensor
      const size_t poff = (size_t)(blk_row0 + pr) * 256 + hf * 128 + pc;

      if (EPI == kEpiPlain || EPI == kEpiBiasGelu) {
        mbar_wait(bar(kAccFull + buf), full_par);
        tc_fence_after();
        if (we == 0 && tt < 2) HG_MARK(10 + 2 * tt);
#pragma unroll 1
        for (int sl = 0; sl < 4; ++sl) {
          const int col0 = hf * 128 + sl * 32;
          float v[32];
          tmem_ld32(tacc + col0, v);
          float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
          if (p.bias) b4 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + pc));
          tmem_ld_wait();
          stg_put_rows(stg, lane, v);
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = 4 * i + pr;
            float4 a = *reinterpret_cast<const float4*>(stg + r * kStgPitch + pc);
            a.x = fmaf(a.x, inv, b4.x); a.y = fmaf(a.y, inv, b4.y); a.z = fmaf(a.z, inv, b4.z); a.w = fmaf(a.w, inv, b4.w);
            const size_t o = poff + (size_t)(4 * i) * 256 + sl * 32;
            if (r < rows_valid) {
              *reinterpret_cast<float4*>(p.out0 + o) = a;
              if (EPI == kEpiBiasGelu) {
                const float4 g = make_float4(gelu_as(a.x), gelu_as(a.y), gelu_as(a.z), gelu_as(a.w));
                amax = amax4(amax, g);
                if (p.out1) *reinterpret_cast<float4*>(p.out1 + o) = g;
              }
            }
          }
          __syncwarp();
        }
      } else if (EPI == kEpiLN) {
        // ---- pass 1 (piece mapping): z = keep * (acc + bias) / (1-p) + projected; loads issued before the accumulator is
        // waited for and refilled for the next slab as soon as a piece has been consumed
        float4 P[8];
        uint32_t Kp[8];
        auto fetch = [&](int i, int sl) {
          const int r = 4 * i + pr;
          const size_t o = poff + (size_t)(4 * i) * 256 + sl * 32;
          P[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          Kp[i] = 0x01010101u;
          if (r < rows_valid) {
            P[i] = ld_stream(reinterpret_cast<const float4*>(p.in0 + o));
            if (p.keep) Kp[i] = __ldg(reinterpret_cast<const unsigned int*>(p.keep + o));
          }
        };
#pragma unroll
        for (int i = 0; i < 8; ++i) fetch(i, 0);
        mbar_wait(bar(kAccFull + buf), full_par);
        tc_fence_after();
        if (we == 0 && tt < 2) HG_MARK(10 + 2 * tt);
        float sum = 0.f;
#pragma unroll 1
        for (int sl = 0; sl < 4; ++sl) {
          const int col0 = hf * 128 + sl * 32;
          float v[32];
          tmem_ld32(tacc + col0, v);
          const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + pc));
          tmem_ld_wait();
          stg_put_rows(stg, lane, v);
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = 4 * i + pr;
            float4 a = *reinterpret_cast<const float4*>(stg + r * kStgPitch + pc);
            a.x = fmaf(a.x, inv, b4.x); a.y = fmaf(a.y, inv, b4.y); a.z = fmaf(a.z, inv, b4.z); a.w = fmaf(a.w, inv, b4.w);
            if (p.keep) {
              const uint32_t k = Kp[i];
              a.x = (k & 0xffu) ? a.x * p.drop_scale : 0.f;
              a.y = (k & 0xff00u) ? a.y * p.drop_scale : 0.f;
              a.z = (k & 0xff0000u) ? a.z * p.drop_scale : 0.f;
              a.w = (k & 0xff000000u) ? a.w * p.drop_scale : 0.f;
            }
            a.x += P[i].x; a.y += P[i].y; a.z += P[i].z; a.w += P[i].w;
            *reinterpret_cast<float4*>(stg + r * kStgPitch + pc) = a;
            if (p.out1 && r < rows_valid) *reinterpret_cast<float4*>(p.out1 + poff + (size_t)(4 * i) * 256 + sl * 32) = a;
            if (sl < 3) fetch(i, sl + 1);
          }
          __syncwarp();
          stg_get_rows(stg, lane, v);      // back to the row mapping: z of this lane's row
#pragma unroll
          for (int e = 0; e < 32; ++e) sum += v[e];
          tmem_st32f(tacc + col0, v);      // z stays in tensor memory (over the accumulator) for the next two passes
          __syncwarp();
        }
        tmem_st_wait();
        lnx[(0 * 2 + hf) * 128 + lrow] = sum;
        named_bar_sync(1 + q, 64);
        const float mean = (lnx[(0 * 2 + 0) * 128 + lrow] + lnx[(0 * 2 + 1) * 128 + lrow]) * (1.f / 256.f);
        float var = 0.f;
#pragma unroll 1
        for (int sl = 0; sl < 4; ++sl) {
          float v[32];
          tmem_ld32(tacc + hf * 128 + sl * 32, v);
          tmem_ld_wait();
#pragma unroll
          for (int e = 0; e < 32; ++e) { const float d = v[e] - mean; var = fmaf(d, d, var); }
        }
        lnx[(1 * 2 + hf) * 128 + lrow] = var;
        named_bar_sync(1 + q, 64);
        const float rstd = rsqrtf((lnx[(1 * 2 + 0) * 128 + lrow] + lnx[(1 * 2 + 1) * 128 + lrow]) * (1.f / 256.f) + p.eps);
#pragma unroll 1
        for (int sl = 0; sl < 4; ++sl) {
          const int col0 = hf * 128 + sl * 32;
          float v[32];
          tmem_ld32(tacc + col0, v);
          const float4 g4 = __ldg(reinterpret_cast<const float4*>(p.gamma + col0 + pc));
          const float4 t4 = __ldg(reinterpret_cast<const float4*>(p.beta + col0 + pc));
          tmem_ld_wait();
#pragma unroll
          for (int e = 0; e < 32; ++e) v[e] = (v[e] - mean) * rstd;
          stg_put_rows(stg, lane, v);
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = 4 * i + pr;
            float4 a = *reinterpret_cast<const float4*>(stg + r * kStgPitch + pc);
            a.x = fmaf(a.x, g4.x, t4.x); a.y = fmaf(a.y, g4.y, t4.y); a.z = fmaf(a.z, g4.z, t4.z); a.w = fmaf(a.w, g4.w, t4.w);
            if (r < rows_valid) *reinterpret_cast<float4*>(p.out0 + poff + (size_t)(4 * i) * 256 + sl * 32) = a;
          }
          __syncwarp();
        }
        if (hf == 0 && row_ok) {
          if (p.mean) p.mean[grow] = mean;
          if (p.rstd) p.rstd[grow] = rstd;
        }
      } else {
        // ---- kEpiGeluBwd (piece mapping): dp = dh * gelu'(projected) + dz, column sums of dp, max |dp|
        float4 P[8], Dz[8];
        auto fetch = [&](int i, int sl) {
          const int r = 4 * i + pr;
          const size_t o = poff + (size_t)(4 * i) * 256 + sl * 32;
          P[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          Dz[i] = P[i];
          if (r < rows_valid) {
            P[i] = ld_stream(reinterpret_cast<const float4*>(p.in0 + o));
            Dz[i] = ld_stream(reinterpret_cast<const float4*>(p.in1 + o));
          }
        };
#pragma unroll
        for (int i = 0; i < 8; ++i) fetch(i, 0);
        mbar_wait(bar(kAccFull + buf), full_par);
        tc_fence_after();
        if (we == 0 && tt < 2) HG_MARK(10 + 2 * tt);
#pragma unroll 1
        for (int sl = 0; sl < 4; ++sl) {
          const int col0 = hf * 128 + sl * 32;
          tmem_to_stg_rows(tacc + col0, stg, lane);
          __syncwarp();
          float4 cs = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = 4 * i + pr;
            float4 a = *reinterpret_cast<const float4*>(stg + r * kStgPitch + pc);
            a.x = fmaf(a.x * inv, gelu_grad_as(P[i].x), Dz[i].x);   // rows beyond M: acc = 0 and dz = 0 -> 0
            a.y = fmaf(a.y * inv, gelu_grad_as(P[i].y), Dz[i].y);
            a.z = fmaf(a.z * inv, gelu_grad_as(P[i].z), Dz[i].z);
            a.w = fmaf(a.w * inv, gelu_grad_as(P[i].w), Dz[i].w);
            if (r < rows_valid) *reinterpret_cast<float4*>(p.out0 + poff + (size_t)(4 * i) * 256 + sl * 32) = a;
            amax = amax4(amax, a);
            cs.x += a.x; cs.y += a.y; cs.z += a.z; cs.w += a.w;
            if (sl < 3) fetch(i, sl + 1);
          }
          // lanes with the same (lane & 7) hold partial sums of the same four columns: fold the four row groups
#pragma unroll
          for (int o = 8; o <= 16; o <<= 1) {
            cs.x += __shfl_xor_sync(0xffffffffu, cs.x, o); cs.y += __shfl_xor_sync(0xffffffffu, cs.y, o);
            cs.z += __shfl_xor_sync(0xffffffffu, cs.z, o); cs.w += __shfl_xor_sync(0xffffffffu, cs.w, o);
          }
          if (lane < 8) {
            float4* acc4 = reinterpret_cast<float4*>(colsm + sl * 32 + pc);
            float4 t4 = *acc4;
            t4.x += cs.x; t4.y += cs.y; t4.z += cs.z; t4.w += cs.w;
            *acc4 = t4;
          }
          __syncwarp();
        }
      }
      if (we == 0 && tt < 2) HG_MARK(11 + 2 * tt);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(bar(kAccEmpty + buf), 0);
    }
    if ((EPI == kEpiBiasGelu || EPI == kEpiGeluBwd) && p.out_amax) {
      amax = warp_max(amax);
      if (lane == 0 && amax > 0.f) atomicMax(p.out_amax, __float_as_uint(amax));
    }
    if (EPI == kEpiGeluBwd && p.colpart) {
      __syncwarp();
      for (int i = lane; i < 128; i += 32)
        p.colpart[((size_t)blockIdx.x * 4 + q) * 256 + hf * 128 + i] = colsm[i];
    }
  }

  if (warp == 0) HG_MARK(15);
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc_pair(tmem_base, 512);
}

// ================================================================================================ A-resident kernel
namespace aresk {
constexpr int kThreads = 448;
constexpr int kSrcSlot = 32768, kSrcSlots = 2;
constexpr int kBSlot = 16384, kBSlots = 6;             // W rows of this CTA for one (column tile, chunk): hi [64][64 k] + lo
constexpr int kOffSrc = 0;
constexpr int kOffB = kOffSrc + kSrcSlots * kSrcSlot;  // 65536
constexpr int kOffStg = kOffB + kBSlots * kBSlot;      // 163840
constexpr int kOffBar = kOffStg + 8 * kStgBytes;       // 200704
constexpr int kSmem = kOffBar + 256 + 1024;
enum Bar { kSrcFull = 0, kSrcEmpty = 2, kAFull = 4, kAFree = 8, kBFull = 9, kBEmpty = 15, kAccFull = 21, kAccEmpty = 23,
           kNumBars = 25 };
constexpr uint32_t kACol = 256;       // TMEM: accumulators [0, 128) and [128, 256); A chunk c at 256 + 64 c
}  // namespace aresk

struct AresParams {
  int M, N, K, n_row_blocks, n_col_tiles, chunks;
  const unsigned int* a_amax;
  const float* w_scale;
  // The epilogues' fields share their storage, so that the store and rank instantiations keep the parameter block
  // (and the code) they had before the top-k epilogue existed.
  union {
    struct {
      float* C;
      int64_t ldc;
      // kAresRanks only (retrieval ranks, see AresRankArgs in head_tc.cuh)
      const unsigned int* thr_row;
      const unsigned int* thr_col;
      const int64_t* key_row;
      const int64_t* key_col;
      int* cnt_row;
      int* cnt_col;
    };
    struct {
      // kAresTopk only (retrieval top-k, see AresTopkArgs in head_tc.cuh).  This launch's chunk of the bank starts at
      // row block rb0 (bank rows) or column tile ct0 (bank columns); n_row_blocks / n_col_tiles count the chunk.
      int query_rows, rb0, ct0, cap;
      const unsigned int* theta;
      unsigned long long* surv;
      unsigned int* cnt;
    };
  };
};

// Epilogues of the resident kernel: kAresStore writes C (the heads' dx = dp Wp); kAresRanks writes nothing per element
// and counts, per row and per column, the scores above that row's / column's threshold (retrieval evaluation);
// kAresTopk appends the scores at or above each query's running threshold to that query's survivor slots.
enum AresEpilogue { kAresStore = 0, kAresRanks = 1, kAresTopk = 2 };

// Order-preserving bits of the engine's score acc * inv (inv a power of two, as the store epilogue forms it); -0 and
// +0 are one score.  The top-k key is (these bits << 32 | ~bank index): unique, larger = better, ties -> lower index.
__device__ __forceinline__ unsigned int score_ord(float acc, float inv) {
  const float s = acc * inv;
  return float_to_ord(s == 0.f ? 0.f : s);
}
__device__ __forceinline__ unsigned long long survivor_key(unsigned int ord, int n) {
  return ((unsigned long long)ord << 32) | (unsigned long long)(~(uint32_t)n);
}

// Rank epilogue of one warp's 32 rows x 32 columns: v[e] = raw accumulator of (lane's row, column e).  ct / ck: the
// columns' scaled thresholds and keys in shared memory (uniform addresses: broadcasts).  A pair (row, column) is a
// positive when the keys match; positives are never counted.  rc += columns of this row above trow; cc (lane e) =
// rows of this warp above column e's threshold.
__device__ __forceinline__ void rank_count32(const float* v, const float* ct, const int* ck, float trow, int krow,
                                             int lane, int& rc, int& cc) {
#pragma unroll
  for (int e4 = 0; e4 < 32; e4 += 4) {
    const float4 t4 = *reinterpret_cast<const float4*>(ct + e4);
    const int4 k4 = *reinterpret_cast<const int4*>(ck + e4);
    const float tt[4] = {t4.x, t4.y, t4.z, t4.w};
    const int kk[4] = {k4.x, k4.y, k4.z, k4.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float s = v[e4 + i];
      const bool neg = kk[i] != krow;
      rc += (neg && s > trow) ? 1 : 0;
      const int n = __popc(__ballot_sync(0xffffffffu, neg && s > tt[i]));
      if (lane == e4 + i) cc = n;
    }
  }
}

// Work split of the resident kernel.  A job = (row block, range of column tiles).  Every pair first takes ONE whole row
// block; the column tiles of the remaining row blocks are dealt out evenly in tile units (a pair then converts part
// of a row block it shares with a neighbour), so that 128 row blocks on 74 pairs cost 1.73 blocks of time, not 2.
struct AresJobs {
  int n_row_blocks, n_col_tiles, npairs, pair_id;
  int stage;     // 0: the whole row block `pair_id`; >= 1: segments of the remainder
  long cur, end;
  __device__ AresJobs(int nrb, int nct, int np, int pid) : n_row_blocks(nrb), n_col_tiles(nct), npairs(np), pair_id(pid), stage(0) {
    const long rem = (long)max(nrb - np, 0) * nct;
    cur = rem * pid / np;
    end = rem * (pid + 1) / np;
  }
  __device__ bool next(int& rb, int& nt0, int& nt1) {
    if (stage == 0) {
      stage = 1;
      if (pair_id < n_row_blocks) { rb = pair_id; nt0 = 0; nt1 = n_col_tiles; return true; }
    }
    if (cur >= end) return false;
    rb = npairs + (int)(cur / n_col_tiles);
    nt0 = (int)(cur % n_col_tiles);
    const long take = min((long)(n_col_tiles - nt0), end - cur);
    nt1 = nt0 + (int)take;
    cur += take;
    return true;
  }
};

template <int PASSES, int EPI>
__global__ void __launch_bounds__(aresk::kThreads, 1)
ares_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_wh,
            const __grid_constant__ CUtensorMap map_wl, const AresParams p) {
  using namespace aresk;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* const sbase = smem_raw + (base - raw);
  const uint32_t bar0 = base + kOffBar;
  auto bar = [&](int i) -> uint32_t { return bar0 + 8u * i; };
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(sbase + kOffBar + 8 * kNumBars);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair_id = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  constexpr bool kLo = PASSES == 3;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kSrcSlots; ++s) { mbar_init(bar(kSrcFull + s), 1); mbar_init(bar(kSrcEmpty + s), 4); }
    for (int c = 0; c < 4; ++c) mbar_init(bar(kAFull + c), 8);
    mbar_init(bar(kAFree), 1);
    for (int s = 0; s < kBSlots; ++s) { mbar_init(bar(kBFull + s), 1); mbar_init(bar(kBEmpty + s), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(bar(kAccFull + b), 1); mbar_init(bar(kAccEmpty + b), 16); }
    fence_mbar_init();
    prefetch_tmap(&map_a); prefetch_tmap(&map_wh); prefetch_tmap(&map_wl);
  }
  if (warp == 1) {
    tmem_alloc_pair(smem_u32(tmem_slot), 512);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      uint32_t is = 0, ib = 0;
      AresJobs jobs(p.n_row_blocks, p.n_col_tiles, npairs, pair_id);
      int rb, nt0, nt1;
      while (jobs.next(rb, nt0, nt1)) {
        if constexpr (EPI == kAresTopk) { rb += p.rb0; nt0 += p.ct0; nt1 += p.ct0; }
        const int row0 = rb * 256 + (int)rank * 128;
        for (int c = 0; c < p.chunks; ++c, ++is) {
          const uint32_t slot = is % kSrcSlots, par = (is / kSrcSlots) & 1;
          mbar_wait(bar(kSrcEmpty + slot), par ^ 1);
          const uint32_t fb = bar(kSrcFull + slot);
          mbar_arrive_expect_tx(fb, (uint32_t)kSrcSlot);
          const uint32_t sa = base + kOffSrc + slot * kSrcSlot;
          tma_load_2d(sa, &map_a, fb, c * 64, row0);
          tma_load_2d(sa + 16384, &map_a, fb, c * 64 + 32, row0);
        }
        for (int nt = nt0; nt < nt1; ++nt) {
          const int wrow = nt * 128 + (int)rank * 64;
          for (int c = 0; c < p.chunks; ++c, ++ib) {
            const uint32_t slot = ib % kBSlots, par = (ib / kBSlots) & 1;
            mbar_wait(bar(kBEmpty + slot), par ^ 1);
            const uint32_t fb = bar(kBFull + slot);
            if (leader) mbar_arrive_expect_tx(fb, (kLo ? 2u : 1u) * 2u * 8192u);
            const uint32_t sb = base + kOffB + slot * kBSlot;
            tma_load_2d_pair(sb, &map_wh, fb, c * 64, wrow);
            if (kLo) tma_load_2d_pair(sb + 8192, &map_wl, fb, c * 64, wrow);
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (leader && elect_one()) {
      constexpr uint32_t idesc = idesc_f16(256, 128);
      uint32_t ib = 0, tn = 0, nb = 0;
      AresJobs jobs(p.n_row_blocks, p.n_col_tiles, npairs, pair_id);
      int rb, nt0, nt1;
      for (; jobs.next(rb, nt0, nt1); ++nb) {
        for (int nt = nt0; nt < nt1; ++nt, ++tn) {
          const uint32_t buf = tn & 1, use = tn >> 1;
          mbar_wait(bar(kAccEmpty + buf), (use & 1) ^ 1);
          tc_fence_after();
          const uint32_t td = tmem_base + buf * 128;
          for (int c = 0; c < p.chunks; ++c, ++ib) {
            if (nt == nt0) mbar_wait(bar(kAFull + c), nb & 1);   // this job's chunk c is in tensor memory
            const uint32_t slot = ib % kBSlots, par = (ib / kBSlots) & 1;
            mbar_wait(bar(kBFull + slot), par);
            tc_fence_after();
            const uint32_t sb = base + kOffB + slot * kBSlot;
            const uint64_t bh = smem_desc_sw128(sb), bl = smem_desc_sw128(sb + 8192);
            const uint32_t ah = tmem_base + kACol + c * 64, al = ah + 32;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              const uint32_t acc = (c > 0 || ks > 0) ? 1u : 0u;
              mma_f16_pair_ts(td, ah + ks * 8, desc_advance_k(bh, ks), idesc, acc);
              if (kLo) {
                mma_f16_pair_ts(td, ah + ks * 8, desc_advance_k(bl, ks), idesc, 1u);
                mma_f16_pair_ts(td, al + ks * 8, desc_advance_k(bh, ks), idesc, 1u);
              }
            }
            mma_commit_pair(bar(kBEmpty + slot), 3);
          }
          mma_commit_pair(bar(kAccFull + buf), 3);
        }
        mma_commit_pair(bar(kAFree), 3);   // every MMA that reads this row block's A has completed
      }
    }
    __syncwarp();
  } else if (warp < 6) {
    const int q = warp & 3, row = q * 32 + lane;
    const uint32_t lane_field = (uint32_t)(q * 32) << 16;
    const float s = scale_from_amax_bits(*p.a_amax);
    float amax = 0.f;
    uint32_t is = 0, nb = 0;
    AresJobs jobs(p.n_row_blocks, p.n_col_tiles, npairs, pair_id);
    int rb, nt0, nt1;
    for (; jobs.next(rb, nt0, nt1); ++nb) {
      mbar_wait(bar(kAFree), (nb & 1) ^ 1);
      tc_fence_after();
      for (int c = 0; c < p.chunks; ++c, ++is) {
        const uint32_t ss = is % kSrcSlots, sp = (is / kSrcSlots) & 1;
        mbar_wait(bar(kSrcFull + ss), sp);
        const uint32_t sa = base + kOffSrc + ss * kSrcSlot;
        const uint32_t ta = tmem_base + lane_field + kACol + c * 64;
#pragma unroll
        for (int bx = 0; bx < 2; ++bx) {
          uint32_t hw[16], lw[16];
          convert_row32<kLo>(sa + bx * 16384, row, s, hw, lw, amax);
          tmem_st16(ta + bx * 16, hw);
          if (kLo) tmem_st16(ta + 32 + bx * 16, lw);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive_local(bar(kSrcEmpty + ss));
          mbar_arrive_cluster(bar(kAFull + c), 0);
        }
      }
    }
    (void)amax;
  } else if constexpr (EPI == kAresRanks) {
    // Rank counts.  Warp (q, hf) sees rows q*32 + lane of this CTA's 128 and columns hf*64 .. +64 of each tile.  The
    // thresholds are compared with the RAW accumulator: score = acc * inv with inv a power of two, so
    // acc > thr / inv <=> score > thr exactly.
    const int we = warp - 6, q = warp & 3, hf = we >> 2;
    const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16);
    const float to_acc = scale_from_amax_bits(*p.a_amax) * p.w_scale[0];   // 1 / inv
    int* const xch = reinterpret_cast<int*>(sbase + kOffStg);               // [2 buffers][2 halves][4 warps][64]
    float* const ct = reinterpret_cast<float*>(sbase + kOffStg + 4096 + we * 512);   // this warp's 64 thresholds
    int* const ck = reinterpret_cast<int*>(sbase + kOffStg + 4096 + we * 512 + 256); // and 64 keys
    uint32_t tn = 0;
    AresJobs jobs(p.n_row_blocks, p.n_col_tiles, npairs, pair_id);
    int rb, nt0, nt1;
    while (jobs.next(rb, nt0, nt1)) {
      const int row = rb * 256 + (int)rank * 128 + q * 32 + lane;
      const bool row_ok = row < p.M;
      float trow = INFINITY;
      int krow = -1;
      if (row_ok) {
        trow = ord_to_float(p.thr_row[row]) * to_acc;
        krow = p.key_row ? (int)p.key_row[row] : row;
      }
      int rc = 0;
      for (int nt = nt0; nt < nt1; ++nt, ++tn) {
        const uint32_t buf = tn & 1, use = tn >> 1;
        const int col0 = nt * 128 + hf * 64, cols_valid = p.N - col0;
        __syncwarp();
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int c = col0 + h * 32 + lane;
          float t = INFINITY;
          int k = -2;
          if (h * 32 + lane < cols_valid) {
            t = ord_to_float(p.thr_col[c]) * to_acc;
            k = p.key_col ? (int)p.key_col[c] : c;
          }
          ct[h * 32 + lane] = t;
          ck[h * 32 + lane] = k;
        }
        mbar_wait(bar(kAccFull + buf), use & 1);
        tc_fence_after();
        float v0[32], v1[32];
        tmem_ld32(tacc + buf * 128 + hf * 64, v0);
        tmem_ld32(tacc + buf * 128 + hf * 64 + 32, v1);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(bar(kAccEmpty + buf), 0);
        if (!row_ok || cols_valid < 64) {   // padding rows / columns hold zeros, which can beat a negative threshold
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            if (!row_ok || e >= cols_valid) v0[e] = -INFINITY;
            if (!row_ok || e + 32 >= cols_valid) v1[e] = -INFINITY;
          }
        }
        int cc0 = 0, cc1 = 0;
        rank_count32(v0, ct, ck, trow, krow, lane, rc, cc0);
        rank_count32(v1, ct + 32, ck + 32, trow, krow, lane, rc, cc1);
        // the four row-quarter warps of this column half meet in shared memory; one of them (rotating) adds the
        // CTA's count of each column to global memory.  Double-buffered: the barrier of tile tn + 1 orders the reads
        // of tile tn before the writes of tile tn + 2.
        int* const xb = xch + (buf * 2 + hf) * 256;
        xb[q * 64 + lane] = cc0;
        xb[q * 64 + 32 + lane] = cc1;
        named_bar_sync(1 + hf, 128);
        if (q == (int)(tn & 3)) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int i = h * 32 + lane;
            const int s = xb[i] + xb[64 + i] + xb[128 + i] + xb[192 + i];
            if (s > 0 && i < cols_valid) atomicAdd(p.cnt_col + col0 + i, s);
          }
        }
      }
      if (row_ok && rc > 0) atomicAdd(p.cnt_row + row, rc);   // remainder jobs share a row block: atomic
    }
  } else if constexpr (EPI == kAresTopk) {
    // Top-k survivors.  A score survives when its order-preserving bits are >= its query's running threshold theta
    // (0 before the query has k candidates: everything survives); it is appended as survivor_key to the query's slots
    // [query * cap, (query + 1) * cap).  One launch covers one chunk of at most `cap` bank entries and every (query,
    // bank entry) pair is visited once, so a query's counter ends at most at cap.  Padding rows and columns (TMA zero
    // fill) score 0 and must never survive: they are masked by index, not by value.
    const int we = warp - 6, q = warp & 3, hf = we >> 2;
    const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16);
    const float inv = (1.f / scale_from_amax_bits(*p.a_amax)) * p.w_scale[1];
    unsigned int* const cth = reinterpret_cast<unsigned int*>(sbase + kOffStg + we * 256);   // this warp's 64 columns
    const bool qrows = p.query_rows != 0;
    const size_t cap = (size_t)p.cap;
    uint32_t tn = 0;
    AresJobs jobs(p.n_row_blocks, p.n_col_tiles, npairs, pair_id);
    int rb, nt0, nt1;
    while (jobs.next(rb, nt0, nt1)) {
      rb += p.rb0; nt0 += p.ct0; nt1 += p.ct0;
      const int row = rb * 256 + (int)rank * 128 + q * 32 + lane;
      const bool row_ok = row < p.M;
      const unsigned int trow = (qrows && row_ok) ? p.theta[row] : 0u;
      for (int nt = nt0; nt < nt1; ++nt, ++tn) {
        const uint32_t buf = tn & 1, use = tn >> 1;
        const int col0 = nt * 128 + hf * 64, cols_valid = p.N - col0;
        if (!qrows) {   // queries are columns: their thresholds through shared memory (uniform reads: broadcasts)
          __syncwarp();
#pragma unroll
          for (int h = 0; h < 2; ++h) cth[h * 32 + lane] = h * 32 + lane < cols_valid ? p.theta[col0 + h * 32 + lane] : 0u;
          __syncwarp();
        }
        mbar_wait(bar(kAccFull + buf), use & 1);
        tc_fence_after();
        float v0[32], v1[32];
        tmem_ld32(tacc + buf * 128 + hf * 64, v0);
        tmem_ld32(tacc + buf * 128 + hf * 64 + 32, v1);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(bar(kAccEmpty + buf), 0);
        if (qrows) {
          // lane = query row: count its survivors among the 64 columns, one atomic claims that many slots
          if (row_ok) {
            unsigned long long m = 0ull;
#pragma unroll
            for (int e = 0; e < 64; ++e) {
              const unsigned int o = score_ord(e < 32 ? v0[e] : v1[e - 32], inv);
              if (e < cols_valid && o >= trow) m |= 1ull << e;
            }
            const int n = __popcll(m);
            if (n > 0) {
              const unsigned int slot = atomicAdd(p.cnt + row, (unsigned int)n);
#ifdef MC_DEBUG_ASSERTS
              assert(slot + (unsigned int)n <= (unsigned int)p.cap);
#endif
              unsigned long long* dst = p.surv + (size_t)row * cap + slot;
#pragma unroll
              for (int e = 0; e < 64; ++e)
                if ((m >> e) & 1ull) *dst++ = survivor_key(score_ord(e < 32 ? v0[e] : v1[e - 32], inv), col0 + e);
            }
          }
        } else {
          // lane = bank row, column e = query col0 + e: a ballot per column, one atomic per column with survivors
          const unsigned int lt = (1u << lane) - 1u;
#pragma unroll
          for (int e = 0; e < 64; ++e) {
            const unsigned int o = score_ord(e < 32 ? v0[e] : v1[e - 32], inv);
            const bool sv = row_ok && e < cols_valid && o >= cth[e];
            const unsigned int bal = __ballot_sync(0xffffffffu, sv);
            if (bal) {
              unsigned int slot = 0;
              if (lane == 0) slot = atomicAdd(p.cnt + col0 + e, (unsigned int)__popc(bal));
              slot = __shfl_sync(0xffffffffu, slot, 0);
#ifdef MC_DEBUG_ASSERTS
              assert(slot + (unsigned int)__popc(bal) <= (unsigned int)p.cap);
#endif
              if (sv) p.surv[(size_t)(col0 + e) * cap + slot + __popc(bal & lt)] = survivor_key(o, row);
            }
          }
        }
      }
    }
  } else {
    const int we = warp - 6, q = warp & 3, hf = we >> 2;
    const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16);
    float* const stg = reinterpret_cast<float*>(sbase + kOffStg + we * kStgBytes);
    const float inv = (1.f / scale_from_amax_bits(*p.a_amax)) * p.w_scale[1];
    uint32_t tn = 0;
    AresJobs jobs(p.n_row_blocks, p.n_col_tiles, npairs, pair_id);
    int rb, nt0, nt1;
    while (jobs.next(rb, nt0, nt1)) {
      const int blk_row0 = rb * 256 + (int)rank * 128 + q * 32;
      const int rows_valid = p.M - blk_row0;
      for (int nt = nt0; nt < nt1; ++nt, ++tn) {
        const uint32_t buf = tn & 1, use = tn >> 1;
        mbar_wait(bar(kAccFull + buf), use & 1);
        tc_fence_after();
        float v0[32], v1[32];
        tmem_ld32(tacc + buf * 128 + hf * 64, v0);
        tmem_ld32(tacc + buf * 128 + hf * 64 + 32, v1);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(bar(kAccEmpty + buf), 0);   // the tile is in registers: hand the buffer back
        const int col0 = nt * 128 + hf * 64;
#pragma unroll
        for (int e = 0; e < 32; ++e) { v0[e] *= inv; v1[e] *= inv; }
        block_store(stg, lane, v0, p.C + (size_t)blk_row0 * p.ldc + col0, p.ldc, rows_valid, p.N - col0);
        block_store(stg, lane, v1, p.C + (size_t)blk_row0 * p.ldc + col0 + 32, p.ldc, rows_valid, p.N - col0 - 32);
      }
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc_pair(tmem_base, 512);
}

// ================================================================================================ transposed-operands kernel
namespace ttk {
constexpr int kThreads = 320;   // warp 0 TMA, warp 1 MMA, warps 2-5 convert A -> TMEM, warps 6-9 convert B -> smem; 2-9 epilogue
constexpr int kSrcSlot = 32768, kSrcSlots = 5;         // 32 k rows: A box [32][128 cols] fp32 + B box [32][128 cols]
constexpr int kOpSlot = 32768;                         // B operand of one 64-k chunk: hi [128 rows][64 k] + lo
constexpr int kOffSrc = 0;
constexpr int kOffOp = kOffSrc + kSrcSlots * kSrcSlot; // 163840
constexpr int kOffStg = kOffSrc;                       // the epilogue runs once, after the last load was consumed: it
                                                       // stages through the (idle) source ring
constexpr int kOffBar = kOffOp + 2 * kOpSlot;          // 229376
constexpr int kSmem = kOffBar + 256 + 1024;
enum Bar { kSrcFull = 0, kSrcEmpty = 5, kOpFull = 10, kOpEmpty = 12, kAccFull = 14, kNumBars = 15 };
constexpr uint32_t kACol = 256;
}  // namespace ttk

struct TtParams {
  int K, No, n_tiles, ksplit, chunks_per_split, chunks_total;
  const unsigned int* a_amax;
  const unsigned int* b_amax;
  float* part;   // [ksplit][256][No]
};

template <int PASSES>
__global__ void __launch_bounds__(ttk::kThreads, 1)
tt_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const TtParams p) {
  using namespace ttk;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* const sbase = smem_raw + (base - raw);
  const uint32_t bar0 = base + kOffBar;
  auto bar = [&](int i) -> uint32_t { return bar0 + 8u * i; };
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(sbase + kOffBar + 8 * kNumBars);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int job = blockIdx.x >> 1;            // one (column tile, K split) per pair
  const int nt = job % p.n_tiles, ks = job / p.n_tiles;
  const int c0 = ks * p.chunks_per_split, c1 = min(c0 + p.chunks_per_split, p.chunks_total);
  const int nchunks = c1 - c0;
  constexpr bool kLo = PASSES == 3;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kSrcSlots; ++s) { mbar_init(bar(kSrcFull + s), 1); mbar_init(bar(kSrcEmpty + s), 8); }
    for (int s = 0; s < 2; ++s) { mbar_init(bar(kOpFull + s), 16); mbar_init(bar(kOpEmpty + s), 1); }
    mbar_init(bar(kAccFull), 1);
    fence_mbar_init();
    prefetch_tmap(&map_a); prefetch_tmap(&map_b);
  }
  if (warp == 1) {
    tmem_alloc_pair(smem_u32(tmem_slot), 512);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      for (int h = 0; h < 2 * nchunks; ++h) {   // 32-k half chunks
        const uint32_t slot = h % kSrcSlots, par = (h / kSrcSlots) & 1;
        mbar_wait(bar(kSrcEmpty + slot), par ^ 1);
        const uint32_t fb = bar(kSrcFull + slot);
        mbar_arrive_expect_tx(fb, (uint32_t)kSrcSlot);
        const uint32_t sa = base + kOffSrc + slot * kSrcSlot;
        const int k0 = c0 * 64 + h * 32;
        tma_load_2d(sa, &map_a, fb, (int)rank * 128, k0);
        tma_load_2d(sa + 16384, &map_b, fb, nt * 256 + (int)rank * 128, k0);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (leader && elect_one()) {
      constexpr uint32_t idesc = idesc_f16(256, 256);
      for (int c = 0; c < nchunks; ++c) {
        const uint32_t s = c & 1, par = (c >> 1) & 1;
        mbar_wait(bar(kOpFull + s), par);
        tc_fence_after();
        const uint32_t sb = base + kOffOp + s * kOpSlot;
        const uint64_t bh = smem_desc_sw128(sb), bl = smem_desc_sw128(sb + 16384);
        const uint32_t ah = tmem_base + kACol + s * 64, al = ah + 32;
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4) {
          const uint32_t acc = (c > 0 || k4 > 0) ? 1u : 0u;
          mma_f16_pair_ts(tmem_base, ah + k4 * 8, desc_advance_k(bh, k4), idesc, acc);
          if (kLo) {
            mma_f16_pair_ts(tmem_base, ah + k4 * 8, desc_advance_k(bl, k4), idesc, 1u);
            mma_f16_pair_ts(tmem_base, al + k4 * 8, desc_advance_k(bh, k4), idesc, 1u);
          }
        }
        mma_commit_pair(bar(kOpEmpty + s), 3);
      }
      mma_commit_pair(bar(kAccFull), 3);
    }
    __syncwarp();
  } else {
    const bool conv_a = warp < 6;
    const int q = warp & 3;
    const int col = conv_a ? q * 32 + lane : (warp - 6) * 32 + lane;   // A: TMEM lane = output row; B: operand row
    const uint32_t lane_field = (uint32_t)(q * 32) << 16;
    const float s = scale_from_amax_bits(conv_a ? *p.a_amax : *p.b_amax);
    for (int c = 0; c < nchunks; ++c) {
      const uint32_t os = c & 1, op = (c >> 1) & 1;
      mbar_wait(bar(kOpEmpty + os), op ^ 1);   // the MMAs of chunk c - 2 are done with this stage
      tc_fence_after();
#pragma unroll 1
      for (int hh = 0; hh < 2; ++hh) {
        const uint32_t h = 2 * c + hh, ss = h % kSrcSlots, sp = (h / kSrcSlots) & 1;
        mbar_wait(bar(kSrcFull + ss), sp);
        const uint32_t src = base + kOffSrc + ss * kSrcSlot + (conv_a ? 0u : 16384u);
        uint32_t hw[16], lw[16];
        convert_col32<kLo>(src, col, s, hw, lw);
        if (conv_a) {
          const uint32_t ta = tmem_base + lane_field + kACol + os * 64 + hh * 16;
          tmem_st16(ta, hw);
          if (kLo) tmem_st16(ta + 32, lw);
        } else {
          const uint32_t rowb = base + kOffOp + os * kOpSlot + (uint32_t)col * 128u;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint32_t off = (uint32_t)(((4 * hh + i) ^ (col & 7)) << 4);
            sts128(rowb + off, hw[4 * i], hw[4 * i + 1], hw[4 * i + 2], hw[4 * i + 3]);
            if (kLo) sts128(rowb + 16384 + off, lw[4 * i], lw[4 * i + 1], lw[4 * i + 2], lw[4 * i + 3]);
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive_local(bar(kSrcEmpty + ss));
      }
      if (conv_a) {
        tmem_st_wait();
        tc_fence_before();
      } else {
        fence_proxy_async_smem();
      }
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(bar(kOpFull + os), 0);
    }
    // ---- epilogue: this CTA's 128 output rows x 256 columns of the pair's tile -> split-K partial
    const int we = warp - 2, hf = we >> 2;
    float* const stg = reinterpret_cast<float*>(sbase + kOffStg + we * kStgBytes);
    const float inv = (1.f / scale_from_amax_bits(*p.a_amax)) * (1.f / scale_from_amax_bits(*p.b_amax));
    mbar_wait(bar(kAccFull), 0);
    tc_fence_after();
    const int orow0 = (int)rank * 128 + q * 32;
    float* const pbase = p.part + ((size_t)ks * 256 + orow0) * p.No;
#pragma unroll 1
    for (int sl = 0; sl < 4; ++sl) {
      const int col0 = nt * 256 + hf * 128 + sl * 32;
      float v[32];
      tmem_ld32(tmem_base + lane_field + hf * 128 + sl * 32, v);
      tmem_ld_wait();
#pragma unroll
      for (int e = 0; e < 32; ++e) v[e] *= inv;
      if (col0 < p.No) block_store(stg, lane, v, pbase + col0, p.No, 32, p.No - col0);
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc_pair(tmem_base, 512);
}

// C[m][n] = sum_ks part[ks][m][n]: a block of (64 float4 columns) x (4 split groups); every thread keeps eight loads in
// flight, the four groups meet in shared memory in a fixed order (deterministic)
__global__ void __launch_bounds__(256) tt_reduce_kernel(const float4* __restrict__ part, int ksplit, size_t n4, int No4,
                                                        float* __restrict__ C, int64_t ldc) {
  __shared__ float4 sm[4][64];
  const int tx = threadIdx.x & 63, g = threadIdx.x >> 6;
  const size_t i = (size_t)blockIdx.x * 64 + tx;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  if (i < n4) {
    int k = g;
    for (; k + 28 < ksplit; k += 32) {
      float4 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = ld_stream(part + (size_t)(k + 4 * u) * n4 + i);
#pragma unroll
      for (int u = 0; u < 8; ++u) { a.x += v[u].x; a.y += v[u].y; a.z += v[u].z; a.w += v[u].w; }
    }
    for (; k < ksplit; k += 4) {
      const float4 v = ld_stream(part + (size_t)k * n4 + i);
      a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
  }
  sm[g][tx] = a;
  __syncthreads();
  if (g == 0 && i < n4) {
#pragma unroll
    for (int u = 1; u < 4; ++u) { const float4 v = sm[u][tx]; a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w; }
    const size_t m = i / No4, n = (i % No4) * 4;
    *reinterpret_cast<float4*>(C + m * ldc + n) = a;
  }
}

// ================================================================================================ host side
static int row_pairs(int M) { return pairs_for((M + 255) / 256); }
int colpart_rows(int M) { return 2 * row_pairs(M) * 4; }

template <int EPI>
static int launch_row(int passes, int npairs, const CUtensorMap& ma, const CUtensorMap& wh, const CUtensorMap& wl,
                      const RowParams& p, cudaStream_t st) {
  return with_passes(passes == 3, [&](auto P) {
    // K <= 256: the epilogue-bound plan (A in shared memory, two accumulators); longer K: A in tensor memory
    if (p.K <= 256) return launch_pairs<row_kernel<EPI, P, true>>(npairs, rowk::kThreads, rowk::kSmem, st, ma, wh, wl, p);
    return launch_pairs<row_kernel<EPI, P, false>>(npairs, rowk::kThreads, rowk::kSmem, st, ma, wh, wl, p);
  });
}

int rows_gemm(const RowArgs& a, cudaStream_t st) {
  MC_REQUIRE(a.A && (a.a_amax || a.vmode == 1 || a.vmode == 2) && a.W.hi && a.W.lo && a.W.scale && a.out0, MC_ERR_BAD_ARG,
             "head rows gemm: null pointer");
  MC_REQUIRE(a.M > 0 && a.K > 0 && a.K % 4 == 0 && a.lda % 4 == 0, MC_ERR_UNSUPPORTED,
             "head rows gemm: K (%d) and the row stride must be multiples of 4", a.K);
  MC_REQUIRE(a.W.rows == 256 && a.W.cols == a.K, MC_ERR_BAD_ARG, "head rows gemm: weight planes are %d x %d, expected 256 x %d",
             a.W.rows, a.W.cols, a.K);
  MC_REQUIRE(a.passes == 1 || a.passes == 3, MC_ERR_BAD_ARG, "head rows gemm: passes %d", a.passes);
  MC_REQUIRE(aligned(a.out0, 16) && (!a.out1 || aligned(a.out1, 16)) && (!a.in0 || aligned(a.in0, 16)) &&
                 (!a.in1 || aligned(a.in1, 16)) && (!a.keep || aligned(a.keep, 16)),
             MC_ERR_ALIGN, "head rows gemm: epilogue tensors must be 16-byte aligned");
  CUtensorMap ma, wh, wl;
  int rc;
  if ((rc = make_map(&ma, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, a.A, a.M, a.K, (uint64_t)a.lda * 4, 32, 128,
                     CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = make_map(&wh, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, a.W.hi, 256, a.K, (uint64_t)a.W.pitch * 2, 64, 128,
                     CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = make_map(&wl, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, a.W.lo, 256, a.K, (uint64_t)a.W.pitch * 2, 64, 128,
                     CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  RowParams p;
  p.M = a.M; p.K = a.K;
  p.n_tiles = (a.M + 255) / 256;
  p.chunks = (a.K + 63) / 64;
  p.a_amax = a.a_amax;
  p.w_scale = a.W.scale;
  p.bias = a.bias; p.out0 = a.out0; p.out1 = a.out1; p.in0 = a.in0; p.in1 = a.in1; p.keep = a.keep;
  p.drop_scale = a.drop_scale; p.eps = a.eps; p.gamma = a.gamma; p.beta = a.beta; p.mean = a.mean; p.rstd = a.rstd;
  p.out_amax = a.out_amax; p.colpart = a.colpart;
  p.vmode = a.vmode; p.a_alt = a.a_alt; p.v_stale = a.v_stale; p.v_live = a.v_live; p.a_live = a.a_live;
  p.amax_publish = a.amax_publish;
  MC_REQUIRE(a.vmode >= 0 && a.vmode <= 3 && (a.vmode == 0 || (a.v_stale && a.v_live)) && (a.vmode != 3 || a.a_alt) &&
                 (a.vmode != 1 || a.a_live),
             MC_ERR_BAD_ARG, "head rows gemm: scale protocol pointers missing for vmode %d", a.vmode);
  p.dbg = nullptr;
  if (const char* e = getenv("MAE_CLIP_HG_DBG"))   // tools/head_timeline.py: device address of a 16-word timeline buffer
    p.dbg = reinterpret_cast<unsigned long long*>(strtoull(e, nullptr, 0));
  const int npairs = row_pairs(a.M);
  switch (a.epilogue) {
    case kEpiPlain: return launch_row<kEpiPlain>(a.passes, npairs, ma, wh, wl, p, st);
    case kEpiBiasGelu:
      MC_REQUIRE(a.bias, MC_ERR_BAD_ARG, "head rows gemm: the GELU epilogue needs a bias");
      return launch_row<kEpiBiasGelu>(a.passes, npairs, ma, wh, wl, p, st);
    case kEpiLN:
      MC_REQUIRE(a.bias && a.in0 && a.gamma && a.beta, MC_ERR_BAD_ARG, "head rows gemm: LayerNorm epilogue inputs missing");
      return launch_row<kEpiLN>(a.passes, npairs, ma, wh, wl, p, st);
    case kEpiGeluBwd:
      MC_REQUIRE(a.in0 && a.in1, MC_ERR_BAD_ARG, "head rows gemm: GELU-backward epilogue inputs missing");
      return launch_row<kEpiGeluBwd>(a.passes, npairs, ma, wh, wl, p, st);
  }
  MC_REQUIRE(false, MC_ERR_BAD_ARG, "head rows gemm: unknown epilogue %d", a.epilogue);
  return MC_ERR_BAD_ARG;
}

// tensor maps and the geometry fields of the resident kernel's parameters (both epilogues)
static int ares_setup(const float* A, int64_t lda, const tcg::Planes& W, int M, int N, int K, const unsigned int* a_amax,
                      CUtensorMap* ma, CUtensorMap* wh, CUtensorMap* wl, AresParams* p) {
  int rc;
  if ((rc = make_map(ma, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, A, M, K, (uint64_t)lda * 4, 32, 128,
                     CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = make_map(wh, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, W.hi, N, K, (uint64_t)W.pitch * 2, 64, 64,
                     CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = make_map(wl, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, W.lo, N, K, (uint64_t)W.pitch * 2, 64, 64,
                     CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  *p = AresParams{};
  p->M = M; p->N = N; p->K = K;
  p->n_row_blocks = (M + 255) / 256;
  p->n_col_tiles = (N + 127) / 128;
  p->chunks = (K + 63) / 64;
  p->a_amax = a_amax; p->w_scale = W.scale;
  return MC_OK;
}
template <int EPI>
static int launch_ares(int passes, int npairs, const CUtensorMap& ma, const CUtensorMap& wh, const CUtensorMap& wl,
                       const AresParams& p, cudaStream_t st) {
  return with_passes(passes == 3, [&](auto P) {
    return launch_pairs<ares_kernel<P, EPI>>(npairs, aresk::kThreads, aresk::kSmem, st, ma, wh, wl, p);
  });
}

int ares_gemm(const AresArgs& a, cudaStream_t st) {
  MC_REQUIRE(a.A && a.a_amax && a.W.hi && a.W.lo && a.W.scale && a.C, MC_ERR_BAD_ARG, "head resident gemm: null pointer");
  MC_REQUIRE(a.M > 0 && a.N > 0 && a.K > 0 && a.K <= 256 && a.K % 4 == 0 && a.N % 4 == 0 && a.lda % 4 == 0 && a.ldc % 4 == 0,
             MC_ERR_UNSUPPORTED, "head resident gemm: needs K <= 256 and K, N, strides multiples of 4 (K=%d N=%d)", a.K, a.N);
  MC_REQUIRE(a.W.rows == a.N && a.W.cols == a.K, MC_ERR_BAD_ARG, "head resident gemm: weight planes %d x %d, expected %d x %d",
             a.W.rows, a.W.cols, a.N, a.K);
  MC_REQUIRE(aligned(a.C, 16), MC_ERR_ALIGN, "head resident gemm: output must be 16-byte aligned");
  CUtensorMap ma, wh, wl;
  AresParams p;
  int rc;
  if ((rc = ares_setup(a.A, a.lda, a.W, a.M, a.N, a.K, a.a_amax, &ma, &wh, &wl, &p))) return rc;
  p.C = a.C; p.ldc = a.ldc;
  return launch_ares<kAresStore>(a.passes, row_pairs(a.M), ma, wh, wl, p, st);
}

int ares_ranks(const AresRankArgs& a, cudaStream_t st) {
  MC_REQUIRE(a.A && a.a_amax && a.W.hi && a.W.lo && a.W.scale && a.thr_row && a.thr_col && a.cnt_row && a.cnt_col,
             MC_ERR_BAD_ARG, "resident rank counts: null pointer");
  MC_REQUIRE(a.M > 0 && a.N > 0 && a.K > 0 && a.K <= 256 && a.K % 4 == 0, MC_ERR_UNSUPPORTED,
             "resident rank counts: needs K <= 256 and K %% 4 == 0 (K=%d)", a.K);
  MC_REQUIRE(a.W.rows == a.N && a.W.cols == a.K, MC_ERR_BAD_ARG, "resident rank counts: planes %d x %d, expected %d x %d",
             a.W.rows, a.W.cols, a.N, a.K);
  MC_REQUIRE(a.passes == 1 || a.passes == 3, MC_ERR_BAD_ARG, "resident rank counts: passes %d", a.passes);
  CUtensorMap ma, wh, wl;
  AresParams p;
  int rc;
  if ((rc = ares_setup(a.A, a.K, a.W, a.M, a.N, a.K, a.a_amax, &ma, &wh, &wl, &p))) return rc;
  p.thr_row = a.thr_row; p.thr_col = a.thr_col; p.key_row = a.key_row; p.key_col = a.key_col;
  p.cnt_row = a.cnt_row; p.cnt_col = a.cnt_col;
  return launch_ares<kAresRanks>(a.passes, row_pairs(a.M), ma, wh, wl, p, st);
}

int ares_topk(const AresTopkArgs& a, cudaStream_t st) {
  MC_REQUIRE(a.A && a.a_amax && a.W.hi && a.W.lo && a.W.scale && a.theta && a.surv && a.cnt && a.after_chunk,
             MC_ERR_BAD_ARG, "resident top-k: null pointer");
  MC_REQUIRE(a.M > 0 && a.N > 0 && a.K > 0 && a.K <= 256 && a.K % 4 == 0, MC_ERR_UNSUPPORTED,
             "resident top-k: needs K <= 256 and K %% 4 == 0 (K=%d)", a.K);
  MC_REQUIRE(a.W.rows == a.N && a.W.cols == a.K, MC_ERR_BAD_ARG, "resident top-k: planes %d x %d, expected %d x %d",
             a.W.rows, a.W.cols, a.N, a.K);
  MC_REQUIRE(a.passes == 1 || a.passes == 3, MC_ERR_BAD_ARG, "resident top-k: passes %d", a.passes);
  const int unit = a.query_rows ? 128 : 256;   // a chunk is whole column tiles / whole row blocks of the bank
  MC_REQUIRE(a.cap > 0 && a.cap % unit == 0, MC_ERR_BAD_ARG, "resident top-k: chunk %d is not a multiple of %d", a.cap,
             unit);
  CUtensorMap ma, wh, wl;
  AresParams p;
  int rc;
  if ((rc = ares_setup(a.A, a.K, a.W, a.M, a.N, a.K, a.a_amax, &ma, &wh, &wl, &p))) return rc;   // once per call
  p.query_rows = a.query_rows ? 1 : 0;
  p.cap = a.cap;
  p.theta = a.theta; p.surv = a.surv; p.cnt = a.cnt;
  const int bank_units = a.query_rows ? p.n_col_tiles : p.n_row_blocks, per_chunk = a.cap / unit;
  for (int u0 = 0; u0 < bank_units; u0 += per_chunk) {
    const int nu = bank_units - u0 < per_chunk ? bank_units - u0 : per_chunk;
    if (a.query_rows) { p.ct0 = u0; p.n_col_tiles = nu; }
    else { p.rb0 = u0; p.n_row_blocks = nu; }
    if ((rc = launch_ares<kAresTopk>(a.passes, row_pairs(p.n_row_blocks * 256), ma, wh, wl, p, st)) ||
        (rc = a.after_chunk(a.ctx, st)))
      return rc;
  }
  return MC_OK;
}

struct TtPlan {
  int n_tiles, ksplit, cps, chunks;
};
static TtPlan tt_plan(int No, int K) {
  TtPlan t;
  t.n_tiles = (No + 255) / 256;
  t.chunks = (K + 63) / 64;
  const int np = num_sms() / 2;
  int ks = np / t.n_tiles;
  if (ks < 1) ks = 1;
  if (ks > t.chunks) ks = t.chunks;
  t.cps = (t.chunks + ks - 1) / ks;
  t.ksplit = (t.chunks + t.cps - 1) / t.cps;
  return t;
}
size_t tt_workspace_bytes(int No, int K) {
  if (No <= 0 || K <= 0) return 0;
  return round_up((size_t)tt_plan(No, K).ksplit * 256 * No * sizeof(float), 256);
}

int tt_gemm(const TtArgs& a, void* ws, size_t ws_bytes, cudaStream_t st) {
  MC_REQUIRE(a.A && a.B && a.a_amax && a.b_amax && a.C && ws, MC_ERR_BAD_ARG, "head weight-gradient gemm: null pointer");
  MC_REQUIRE(a.K > 0 && a.No > 0 && a.No % 4 == 0 && a.lda % 4 == 0 && a.ldb % 4 == 0 && a.ldc % 4 == 0, MC_ERR_UNSUPPORTED,
             "head weight-gradient gemm: N (%d) and the strides must be multiples of 4", a.No);
  MC_REQUIRE(aligned(a.C, 16) && aligned(ws, 16), MC_ERR_ALIGN, "head weight-gradient gemm: output / workspace alignment");
  const TtPlan t = tt_plan(a.No, a.K);
  MC_REQUIRE(t.n_tiles * t.ksplit <= num_sms() / 2, MC_ERR_UNSUPPORTED, "head weight-gradient gemm: %d column tiles exceed the grid",
             t.n_tiles);
  MC_REQUIRE(ws_bytes >= tt_workspace_bytes(a.No, a.K), MC_ERR_WORKSPACE, "head weight-gradient gemm: workspace too small");
  CUtensorMap ma, mb;
  int rc;
  if ((rc = make_map(&ma, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, a.A, a.K, 256, (uint64_t)a.lda * 4, 128, 32,
                     CU_TENSOR_MAP_SWIZZLE_NONE))) return rc;
  if ((rc = make_map(&mb, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, a.B, a.K, a.No, (uint64_t)a.ldb * 4, 128, 32,
                     CU_TENSOR_MAP_SWIZZLE_NONE))) return rc;
  TtParams p;
  p.K = a.K; p.No = a.No; p.n_tiles = t.n_tiles; p.ksplit = t.ksplit; p.chunks_per_split = t.cps; p.chunks_total = t.chunks;
  p.a_amax = a.a_amax; p.b_amax = a.b_amax;
  p.part = static_cast<float*>(ws);
  rc = with_passes(a.passes == 3, [&](auto P) {
    return launch_pairs<tt_kernel<P>>(t.n_tiles * t.ksplit, ttk::kThreads, ttk::kSmem, st, ma, mb, p);
  });
  if (rc) return rc;
  const size_t n4 = (size_t)256 * a.No / 4;
  const int nb = (int)((n4 + 63) / 64);
  tt_reduce_kernel<<<nb, 256, 0, st>>>(static_cast<const float4*>(ws), t.ksplit, n4, a.No / 4, a.C, a.ldc);
  MC_LAUNCH_CHECK();
  return MC_OK;
}

}  // namespace hg
}  // namespace mc

using namespace mc;

extern "C" {

size_t mc_head_gemm_workspace_bytes(int kind, int M, int N, int K) {
  if (M <= 0 || N <= 0 || K <= 0 || kind < 0 || kind > 2) return 0;
  if (kind == 2) return 256 + hg::tt_workspace_bytes(N, K);
  return 256 + round_up(tcg::planes_bytes(N, K), 256);
}

int mc_head_gemm(int kind, const float* A, const float* B, int M, int N, int K, const float* bias, float* C,
                 float* gelu_out, int passes, void* ws, size_t ws_bytes, void* stream) {
  MC_ARCH_GUARD();
  MC_REQUIRE(A && B && C && ws, MC_ERR_BAD_ARG, "head_gemm: null pointer");
  MC_REQUIRE(kind >= 0 && kind <= 2 && M > 0 && N > 0 && K > 0, MC_ERR_BAD_ARG, "head_gemm: bad kind / sizes");
  MC_REQUIRE(aligned(ws, 256) && ws_bytes >= mc_head_gemm_workspace_bytes(kind, M, N, K), MC_ERR_WORKSPACE,
             "head_gemm: workspace missing, misaligned or too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* base = static_cast<char*>(ws);
  unsigned int* amax_a = reinterpret_cast<unsigned int*>(base);
  unsigned int* amax_b = amax_a + 1;
  int rc;
  if (kind == 2) {  // C(256, N) = A(K, 256)^T B(K, N)
    MC_REQUIRE(M == 256, MC_ERR_UNSUPPORTED, "head_gemm kind 2: M must be 256 (got %d)", M);
    if ((rc = tcg::amax(A, K, 256, 256, amax_a, st))) return rc;
    if ((rc = tcg::amax(B, K, N, N, amax_b, st))) return rc;
    hg::TtArgs t{A, 256, amax_a, B, N, amax_b, K, N, passes, C, N};
    return hg::tt_gemm(t, base + 256, ws_bytes - 256, st);
  }
  tcg::Planes w = tcg::carve_planes(base + 256, N, K);
  if ((rc = tcg::amax(A, M, K, K, amax_a, st))) return rc;
  if ((rc = tcg::stage(B, N, K, K, 0, w, st))) return rc;
  if (kind == 0) {
    MC_REQUIRE(N == 256, MC_ERR_UNSUPPORTED, "head_gemm kind 0: N must be 256 (got %d)", N);
    hg::RowArgs r = {};
    r.A = A; r.lda = K; r.a_amax = amax_a; r.W = w; r.M = M; r.K = K; r.passes = passes;
    r.epilogue = gelu_out ? hg::kEpiBiasGelu : hg::kEpiPlain;
    r.bias = bias; r.out0 = C; r.out1 = gelu_out;
    return hg::rows_gemm(r, st);
  }
  hg::AresArgs r{A, K, amax_a, w, M, N, K, passes, C, N};
  return hg::ares_gemm(r, st);
}

}  // extern "C"


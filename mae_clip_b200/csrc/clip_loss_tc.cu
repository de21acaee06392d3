// L3-L6, engines MC_GEMM_TC_F16X3 / MC_GEMM_TC_F16: the contrastive soft-target loss on the 5th-gen
// tensor cores.  Reference arithmetic: /root/reference CLIP.py:34-43 and its autograd (main.py:58),
// closed form in SURVEY.md section 8 row L6.  No B x B tensor of logits or targets ever reaches HBM (the stored-weights
// gradient keeps ONE b x B fp16 strip of gradient weights between its two halves, see kBwdW / rowgrad_kernel): every sweep
// recomputes the 128 x 128 tiles of
//     S  = T_i I_j^T / tau      St = I_i T_j^T / tau  (= S_ji)      Z = (I_i I_j^T + T_i T_j^T) tau/2
// in tensor memory and reduces them in the epilogue.
//
// Kernels in this file (DESIGN.md 4.1 has the dispatch table and the measurements behind it):
//   pair_kernel<PHASE, PASSES>      128 x 128 tiles over a CTA pair of 128 rows: every phase for small problems, the flagged-
//                                   tile sweeps (exact-Z statistics, row loss, soft-target part of the gradient) and the
//                                   own-rows gradient always
//   rowsweep_kernel<KIND, PASSES>   256 x 128 tiles over a CTA pair of 256 rows: S statistics / tile-flag probe of Z (the
//                                   probe multiplies out probe_chunks() of K and bounds the rest; probe_gate_kernel sends
//                                   a batch the bound cannot serve back through the full probe)
//   rowgrad_kernel<PASSES>          same skeleton: S -> softmax part of the gradient weights -> dT, stores the weights
//   colgrad_kernel                  dI from the stored weights (MN-major tcgen05 operand)
// and the staging, fold and gate kernels around them.
//
// pair_kernel's execution model (one kernel template; phases: statistics [probe form when tile flags are on], exact-Z
// statistics on the flagged tiles, row loss, gradient in its own-rows / stored-weights / flagged-tile forms):
//   * a CTA PAIR (cluster of 2, tcgen05 cta_group::2, M = 128) owns 128 samples i, 64 per CTA; the
//     64 x N accumulator tile of a CTA lives in TMEM as 128 lanes x N/2 columns (lanes 0-63: first
//     half of the tile's columns, lanes 64-127: second half);
//   * operands are fp16 planes of X = [I || T] (scaled by one power of two): `hi` = fp16(x),
//     `lo` = fp16(x - hi).  F16X3 issues hi*hi + hi*lo + lo*hi (relative operand error ~2^-22, i.e.
//     fp32-class logits); F16 issues hi*hi only;
//   * warp 0 = TMA producer, warp 1 = MMA issuer (leader CTA, one elected lane) + TMEM allocator, warp 2 = X^T tile
//     producer (gradient sweeps), warp 3 = per-column constants of the gradient sweeps (one tile ahead of the epilogue),
//     warps 4-11 = epilogue (two threads per TMEM lane, 32 columns each).  The hi plane of
//     the pair's own rows stays resident in shared memory for the whole job (the lo plane too in the forward sweeps);
//     the column tiles stream through an mbarrier ring;
//   * the gradient sweep converts each tile into fp16 weight tiles (dS, dS^T, dZ + dZ^T) in shared
//     memory and feeds them straight back to the tensor cores against X^T tiles, accumulating
//     dT_i and dI_i (64 x D each per CTA) in TMEM for the whole job;
//   * tile flags (PairParams::flags / flags_out): tiles that cannot hold soft-target mass (P_ij < 2^-44 throughout)
//     skip their Z work in every sweep - see DESIGN.md section 4.1.
#include <stdlib.h>
#include <string.h>

#include "clip_loss.cuh"
#include "tc_ptx.cuh"

#include <type_traits>

namespace mc {
namespace tc {

using namespace ptx;


constexpr int kTileN = 128;             // columns j per pair tile
constexpr int kRowsCta = 64;            // samples per CTA
constexpr int kChunkBytes = 64 * 128;   // 64 rows x 64 fp16
constexpr int kThreads = 384;      // warps 0-3: TMA / MMA / X^T producer / spare; warps 4-11: epilogue
constexpr int kEpiThreads = 256;
constexpr int kMaxSplit = 16;
constexpr int kIssuers = 1;         // MMA-issuing warps per leader CTA (see the issuer role)

enum Phase { kStats = 0, kRowLoss = 1, kBwd = 2, kStatsZ = 3, kBwdW = 4, kBwdP = 5 };
// kBwdP is the soft-target part of the gradient in the own-rows form, on the FLAGGED tiles only: dS_ij = -2 P_ij,
// dS_ji = -2 P_ji and the dZ weights (everything that vanishes where P does).  It complements rowgrad_kernel, which
// computes the softmax part of dS on every tile.
// kBwdW is the row half of the "stored weights" gradient: like kBwd it recomputes S (and, on flagged tiles only, S^T and
// Z) and accumulates dT_i, but instead of recomputing the transposed strip everywhere to form dS^T for dI_i, it writes
// the fp16 weight tile dS_ij to global memory (PairParams::wout); colgrad_kernel then forms dI_j = sum_i dS_ij T_i from
// the stored tiles (5 GEMM units per tile pair instead of 8).  dI_i of this sweep holds the soft-target (dZ) part only.
// kStats with tile flags requested is the PROBE form: S, S^T at full precision, Z from the hi planes only - enough to
// tell which tiles can hold soft-target mass; kStatsZ then computes S and the exact Z on those tiles (rz, sum P S).

// shared-memory map (offsets from a 1024-byte aligned base)
constexpr int kOffA = 0;                      // resident hi plane of the CTA's 64 rows: 2D/64 chunks
constexpr int kOffStage = 65536;              // TMA ring, 96 KB
constexpr int kStageRegion = 98304;
constexpr int kOffW = kOffStage + kStageRegion;   // three 64 x 64 fp16 weight half-tiles (24 KB)
constexpr int kOffXT = kOffW + 3 * kChunkBytes;   // X^T half tiles: 2 x (D/2 rows x 64 j) (<= 32 KB)
constexpr int kOffConst = kOffXT + 32768;         // per-column constants, 2 x 128 x 8 floats
constexpr int kOffBar = kOffConst + 8192;
constexpr int kSmemBytes = kOffBar + 512 + 1024;  // + alignment slack

enum Bar {
  kFull0 = 0,        // +slot (<= 9)
  kEmpty0 = 9,       // +slot
  kAFull = 18,
  kJobDone = 19,
  kTmemFull0 = 20,   // +buf
  kTmemEmpty0 = 22,  // +buf
  kWFull = 24,
  kGradDone = 25,    // column half 0
  kXTFull = 26,
  kAccFull = 27,
  kAccEmpty = 28,
  kGradDone1 = 29,   // column half 1
  kWFull1 = 30,      // kBwdW: the column halves have their own weight and X^T buffers
  kXTFull1 = 31,
  kCstFull0 = 32,    // +buf: per-column constants of a tile (gradient sweep: produced by warp 3)
  kCstEmpty0 = 34,   // +buf
  kNumBars = 36
};

struct PairParams {
  int b, B, Bp, D, row_offset;
  int n_row_blocks, n_tiles, nsplit, tiles_per_split, bpad;
  float inv_tau, half_tau, inv_2B;
  const float* scale;                  // {s, 1/s, 1/s^2}: global power-of-two scale of the fp16 planes
  const float *r, *c, *rz, *g, *q;     // length-B statistics (phase dependent, may be null)
  const float* ps;                     // row-loss sweep: sum_j P_ij S_ij of the owned rows (length b)
  float* part;                         // partial results of this phase
  const float* wscale;                 // gradient sweep: power-of-two scale of the fp16 weight tiles
  // Tile relevance of the soft targets (see "tile flags" below): the statistics sweep WRITES flags_out
  // [n_row_blocks][n_tiles] (1 = some P_ij of the tile may exceed 2^-44); the row-loss sweep skips tiles whose
  // (symmetrised) flag is 0 and the gradient sweep skips their Z recompute and dZ GEMMs.  Null = dense.
  uint8_t* flags_out;
  const uint8_t* flags;
  const float *norm_i, *norm_t;        // ||I_i||, ||T_i|| of ALL rows (statistics sweep: Z_ii lower-bounds rz_i)
  // Statistics sweep, column partials (see "column LSE" below): when set, the transposed strip S^T is NOT computed; each
  // epilogue warp writes the log-sum-exp of its 32 rows for each of its 32 columns, log2 units, to
  // colpart[(strip row / 32) * Bp + column]; mc::tc::colpart_merge folds them into c.
  float* colpart;
  const int* gate;                     // gradient form switch (ClipProblem::gate): the kernel returns unless *gate == gate_want
  int gate_want;
  __half* wout;                        // kBwdW: (bpad x Bp) fp16 weights 2B dS_ij / tau * wscale / s, row = strip row
  // Arrival-ordered launches of the statistics sweep (host-buffer entry: the batch arrives over PCIe in `chunks` row
  // chunks of chunk_blocks row blocks; nsplit = chunks * chunk_m, so a column split lies inside one chunk).  Launch k
  // takes the jobs (row block, column split) whose LATER chunk is k: everything that became computable when chunk k
  // landed.  chunk_k < 0: every job.
  int chunk_k, chunk_blocks, chunk_m;
};
// job index -> (row block, column split); the filtered launches enumerate their jobs densely so that the pairs stay evenly
// loaded: first the row blocks of chunk k against the splits of chunks 0..k, then the earlier row blocks against chunk k's
__device__ __forceinline__ int pair_njobs(const PairParams& p) {
  if (p.chunk_k < 0) return p.n_row_blocks * p.nsplit;
  const int rows_k = min(p.chunk_blocks, p.n_row_blocks - p.chunk_k * p.chunk_blocks);
  return rows_k * (p.chunk_k + 1) * p.chunk_m + p.chunk_k * p.chunk_blocks * p.chunk_m;
}
__device__ __forceinline__ void pair_job(const PairParams& p, int job, int& rb, int& sp) {
  if (p.chunk_k < 0) { rb = job / p.nsplit; sp = job % p.nsplit; return; }
  const int rows_k = min(p.chunk_blocks, p.n_row_blocks - p.chunk_k * p.chunk_blocks);
  const int w = (p.chunk_k + 1) * p.chunk_m, first = rows_k * w;
  if (job < first) { rb = p.chunk_k * p.chunk_blocks + job / w; sp = job % w; return; }
  job -= first;
  rb = job / p.chunk_m;
  sp = p.chunk_k * p.chunk_m + job % p.chunk_m;
}
// -DMC_WAIT_PROFILE: where do the roles of pair_kernel wait?  Cycles spent in each class of mbarrier wait, summed over the
// pairs (issuer / producers: the elected thread; epilogue: threads 128 and 256 of the leader CTA), read back through
// mc_debug_wait_profile (tools/wait_profile.py).  Not part of the product build.
#ifdef MC_WAIT_PROFILE
__device__ unsigned long long g_wait_prof[64];
__device__ __forceinline__ void mbar_wait_t(uint32_t bar, uint32_t parity, int tag, bool rec) {
  const long long t0 = clock64();
  mbar_wait(bar, parity);
  if (rec) atomicAdd(&g_wait_prof[tag], (unsigned long long)(clock64() - t0));
}
#define MC_PROF_TOTAL(tag, t0, rec) do { if (rec) atomicAdd(&g_wait_prof[tag], (unsigned long long)(clock64() - (t0))); } while (0)
#define MC_PROF_NOW() clock64()
#else
#define MC_PROF_NOW() 0LL
#define mbar_wait_t(bar, parity, tag, rec) mbar_wait(bar, parity)
#define MC_PROF_TOTAL(tag, t0, rec) do { } while (0)
#endif
// Timing ablations (never in the product build; results are garbage, only the clock matters):
//   -DMC_ABLATE_TMA  the ring producer signals its slots full without loading anything
//   -DMC_ABLATE_EPI  the epilogue hands the tile buffer back and skips its arithmetic
#ifdef MC_ABLATE_TMA
#define MC_RING_LOAD(...) do { } while (0)
#define MC_RING_ARM(fb, bytes) mbar_arrive_local(fb)
#else
#define MC_RING_LOAD(...) tma_load_2d_pair(__VA_ARGS__)
#define MC_RING_ARM(fb, bytes) mbar_arrive_expect_tx(fb, bytes)
#endif
constexpr float kFlagTheta2 = 44.f;
constexpr float kProbeMargin2 = 2.f;  // slack on top of the probe's worst-case rounding bound (see zmargin2)    // log2 units: dropped terms are below 2^-44 of their row's soft-target mass

struct PlanesLayout {
  size_t off_hdr, off_norm_i, off_norm_t, off_rho, off_hi, off_lo, off_hiT, total;
  int Bp;
};
static PlanesLayout planes_layout(int B, int D) {
  PlanesLayout l;
  l.Bp = (int)round_up((size_t)B, 128);
  size_t plane = (size_t)l.Bp * 2 * D * sizeof(__half);
  size_t vec = round_up((size_t)l.Bp * 4, 1024);
  l.off_hdr = 0;              // {amax bits, s, 1/s, 1/s^2}
  l.off_norm_i = 1024;        // ||I_i||_2
  l.off_norm_t = 1024 + vec;  // ||T_i||_2
  l.off_rho = 1024 + 2 * vec; // norm of the dimensions the tile-flag probe does NOT multiply out (probe_chunks)
  l.off_hi = 1024 + 3 * vec;
  l.off_lo = l.off_hi + plane;
  l.off_hiT = l.off_lo + plane;
  l.total = l.off_hiT + plane;
  return l;
}

// D/4 accumulator columns per epilogue thread must be a multiple of the 32-column TMEM load
bool supported(int D) { return D == 128 || D == 256; }

// The tile-flag probe of rowsweep_kernel<kRsZ> multiplies out only the first probe_chunks(D) 64-wide K chunks of each
// half of X = [I || T] and bounds the rest of Z_ij by Cauchy-Schwarz with the per-row norm rho of the left-out
// dimensions (written by the staging kernel): Z_ij <= E_ij + tau/2 rho_i rho_j.  Still a rigorous superset of the
// relevant tiles, at half (D = 256) of the probe's MMA work; a batch whose bound is too loose to be useful is
// detected on the device and probed in full (probe_gate_kernel).  Default: two chunks (128 dimensions) of each tower -
// for LayerNorm rows that leaves the bound ~38 nats below the threshold at B = 8192, while ONE chunk does not work at all
// (the left-out energy of a row fluctuates by +-10%, which eats the threshold: measured, half of all tiles flagged);
// D = 128 is therefore probed in full.  MAE_CLIP_PROBE_CHUNKS = D / 64 restores the full probe everywhere.
static int probe_chunks(int D) {
  static const int env = getenv("MAE_CLIP_PROBE_CHUNKS") ? atoi(getenv("MAE_CLIP_PROBE_CHUNKS")) : 2;
  const int nkc = D / 64;
  return env < 1 ? 1 : (env > nkc ? nkc : env);
}

// ------------------------------------------------------------------------------------------
// staging: fp32 embeddings -> scaled fp16 hi / lo planes of X = [I || T], the per-row scale, and
// the transposed hi plane (K-major B operand of the gradient GEMMs).
// ------------------------------------------------------------------------------------------
// largest magnitude over both embedding matrices (non-negative floats order like their bit patterns)
__global__ void __launch_bounds__(256) amax_kernel(const float* __restrict__ I, const float* __restrict__ T,
                                                   size_t n, unsigned int* __restrict__ amax_bits) {
  float a = 0.f;
  size_t i0 = 0;
  if (((reinterpret_cast<uintptr_t>(I) | reinterpret_cast<uintptr_t>(T)) & 15) == 0) {   // 16-byte loads, two streams in flight
    const size_t n4 = n >> 2;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
      const float4 x = reinterpret_cast<const float4*>(I)[i], y = reinterpret_cast<const float4*>(T)[i];
      a = fmaxf(a, fmaxf(fmaxf(fabsf(x.x), fabsf(x.y)), fmaxf(fabsf(x.z), fabsf(x.w))));
      a = fmaxf(a, fmaxf(fmaxf(fabsf(y.x), fabsf(y.y)), fmaxf(fabsf(y.z), fabsf(y.w))));
    }
    i0 = n4 << 2;
  }
  for (size_t i = i0 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    a = fmaxf(a, fmaxf(fabsf(I[i]), fabsf(T[i])));
  a = warp_max(a);
  if ((threadIdx.x & 31) == 0 && a > 0.f) atomicMax(amax_bits, __float_as_uint(a));
}

// ------------------------------------------------------------------------------------------
// the pair kernel
// ------------------------------------------------------------------------------------------
// The TMA ring is made of 16 KB slots (two 64 x 64 fp16 chunks).  Per 64-wide K chunk c:
//   F16X3: slot A  = [I_i lo | T_i lo]   (this CTA's rows; the hi plane is resident)
//          slot BI = [I_j hi | I_j lo],  slot BT = [T_j hi | T_j lo]
//   F16  : slot B  = [I_j hi | T_j hi]
// Small slots keep 4-5 loads in flight ahead of the tensor cores, which hides the L2 latency.
constexpr int kSlotBytes = 2 * kChunkBytes;
constexpr int kSlotsBwd = kStageRegion / kSlotBytes;                                // 6
// the statistics / row-loss sweeps have no weight and X^T tiles: their ring extends over that space
constexpr int kSlotsFwd = (kStageRegion + 3 * kChunkBytes + 32768) / kSlotBytes;    // 9

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2f(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Gradient weights of the padding columns j >= B of a ragged last tile must be exactly zero.  Their logits are 0 (the
// staged planes are zero there), so the softmax terms come out as 2^(-r2_i) and friends: far above the bound the weight
// scale is chosen from (wscale_kernel) when a row statistic is far negative, and an fp16 inf meets the zero rows of the
// other tower in the MMA as NaN.  Clears the K positions [k0, k1) of one 128-byte row (64 fp16 weights, SWIZZLE_128B,
// row m of its tile) in shared memory.  Callers branch on the tile being ragged (tile-uniform) and keep the loop rolled,
// so the hot loop of an aligned batch is left as it was.
__device__ __forceinline__ void zero_padding_cols(uint8_t* row, int m, int k0, int k1) {
#pragma unroll 1
  for (int k = k0; k < k1; ++k) *reinterpret_cast<uint16_t*>(row + ((((k >> 3) ^ (m & 7)) << 4) | ((k & 7) << 1))) = 0;
}

struct OnlineLse2 {  // running log2-domain log-sum-exp
  float m, s;
  __device__ __forceinline__ void init() { m = -INFINITY; s = 0.f; }
  __device__ __forceinline__ void add32(const float* x) {
    float cm = x[0];
#pragma unroll
    for (int e = 1; e < 32; ++e) cm = fmaxf(cm, x[e]);
    const float mn = fmaxf(m, cm);
    if (mn == -INFINITY) return;
    float acc = 0.f;
#pragma unroll
    for (int e = 0; e < 32; ++e) acc += ex2f(x[e] - mn);
    s = s * ex2f(m - mn) + acc;
    m = mn;
  }
  __device__ __forceinline__ void merge(float m2, float s2) {
    const float mn = fmaxf(m, m2);
    if (mn == -INFINITY) return;
    s = s * ex2f(m - mn) + s2 * ex2f(m2 - mn);
    m = mn;
  }
};

// Sparse sweeps (row loss, exact-Z statistics): does the job (row block, column split) contain a flagged tile at all?
// Every role evaluates this on its own and skips the job consistently (no resident loads, no barrier traffic).
__device__ __forceinline__ bool job_has_tiles(const uint8_t* __restrict__ frow, int t0, int t1) {
  unsigned any = 0;
  int t = t0;
  if ((reinterpret_cast<uintptr_t>(frow + t0) & 15) == 0) {
    for (; t + 16 <= t1; t += 16) {
      const uint4 v = *reinterpret_cast<const uint4*>(frow + t);
      any |= v.x | v.y | v.z | v.w;
    }
  }
  for (; t < t1; ++t) any |= frow[t];
  return any != 0;
}

// First flagged tile at or after t (t1 when there is none).  The sparse sweeps visit a handful of tiles per row block: a
// byte-by-byte scan costs one dependent global load per tile (256 of them per job at B = 32768 - 70k cycles, three
// quarters of the flagged-tile sweeps' time); 16 flags per load bring that down to 16.
__device__ __forceinline__ int next_flagged(const uint8_t* __restrict__ f, int t, int t1) {
  while (t < t1) {
    if ((reinterpret_cast<uintptr_t>(f + t) & 15) == 0 && t + 16 <= t1) {
      const uint4 v = *reinterpret_cast<const uint4*>(f + t);
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
      int hit = -1;
#pragma unroll
      for (int k = 3; k >= 0; --k)
        if (w[k]) hit = 4 * k + ((__ffs(w[k]) - 1) >> 3);   // little endian: byte 0 sits in the low bits
      if (hit < 0) { t += 16; continue; }
      return t + hit;
    }
    if (f[t]) return t;
    ++t;
  }
  return t1;
}

template <int PHASE, int PASSES>
__global__ void __launch_bounds__(kThreads, 1)
pair_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
            const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
            const __grid_constant__ CUtensorMap map_t, const PairParams p) {
  if (p.gate != nullptr && *p.gate != p.gate_want) return;   // the other gradient form runs (uniform over the grid)
  // TMEM: tile buffers of 3 x 64 columns (S, St, Z) from column 0; the gradient sweep keeps one tile
  // buffer (the epilogue empties it into registers at once) and its accumulators at 256 (dT), 256 + D/2 (dI)
  constexpr bool kIsBwd = PHASE == kBwd || PHASE == kBwdW || PHASE == kBwdP;
  constexpr bool kSparse = PHASE == kRowLoss || PHASE == kStatsZ || PHASE == kBwdP;   // flagged tiles / jobs only
  constexpr bool kP = PHASE == kBwdP;
  constexpr bool kW = PHASE == kBwdW;
  constexpr int kNBuf = kIsBwd ? 1 : 2;
  constexpr uint32_t kAccCol = 256;
  // Forward sweeps of the 3-pass engine keep the LO plane of the CTA's rows resident too (the gradient sweep has no
  // room: weights + X^T tiles): a third less L2 -> shared-memory traffic per tile, five ring slots left.
  constexpr bool kResLo = !kIsBwd && PASSES == 3;
  constexpr int kOffAlo = kOffStage;                                   // resident lo plane (64 KB) when kResLo
  constexpr int kOffRing = kResLo ? kOffStage + 65536 : kOffStage;
  constexpr int kSlots = kIsBwd ? kSlotsBwd : (kResLo ? kSlotsFwd - 65536 / kSlotBytes : kSlotsFwd);
  static_assert(kOffRing + kSlots * kSlotBytes <= kOffConst, "ring overlaps the column constants");

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* const sbase = smem_raw + (base - raw);
  const uint32_t bar0 = base + kOffBar;
  auto bar = [&](int i) -> uint32_t { return bar0 + 8u * i; };
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(sbase + kOffBar + 8 * kNumBars);

  // warp index through a shuffle: provably warp-uniform, so the role branches (and setmaxnreg) are uniform
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair_id = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int D = p.D, nkc = D >> 6;
  const int njobs = pair_njobs(p);

  if (threadIdx.x == 0) {
    for (int s = 0; s < kSlots; ++s) { mbar_init(bar(kFull0 + s), 1); mbar_init(bar(kEmpty0 + s), kIssuers); }
    mbar_init(bar(kAFull), 1);
    mbar_init(bar(kJobDone), kIssuers);
    for (int i = 0; i < 2; ++i) { mbar_init(bar(kTmemFull0 + i), kIssuers); mbar_init(bar(kTmemEmpty0 + i), 2 * kEpiThreads); }
    mbar_init(bar(kWFull), kEpiThreads);  // one column half at a time: 2 CTAs x 128 threads
    mbar_init(bar(kGradDone), kIssuers);
    mbar_init(bar(kGradDone1), kIssuers);
    mbar_init(bar(kXTFull), 1);
    mbar_init(bar(kWFull1), kEpiThreads);
    mbar_init(bar(kXTFull1), 1);
    for (int i = 0; i < 2; ++i) { mbar_init(bar(kCstFull0 + i), 32); mbar_init(bar(kCstEmpty0 + i), kEpiThreads); }
    mbar_init(bar(kAccFull), kIssuers);
    mbar_init(bar(kAccEmpty), 2 * kEpiThreads);
    fence_mbar_init();
    prefetch_tmap(&map_a_hi); prefetch_tmap(&map_a_lo); prefetch_tmap(&map_b_hi); prefetch_tmap(&map_b_lo);
    prefetch_tmap(&map_t);
  }
  if (warp == 1) {
    tmem_alloc_pair(smem_u32(tmem_slot), 512);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    // warpgroup 0: data movement and MMA issue.  No setmaxnreg here: ptxas (12.9) takes the SMALLEST setmaxnreg
    // immediate in a kernel as the register budget of the WHOLE kernel, so "dec 120 / inc 192" compiled the epilogue
    // for 120 registers (444 bytes of spills in its inner loop) while 192 sat allocated at run time.  With the plain
    // launch bound (384 threads -> 168 registers) the epilogue fits without spills: -3% (tc_f16x3), -12% (tc_f16).
    if (warp == 0) {
      // ========================================================= TMA producer: resident rows + ring
      if (elect_one()) {
        uint32_t it = 0, jj = 0;
        [[maybe_unused]] const long long prof_t0 = MC_PROF_NOW();
        for (int job = pair_id; job < njobs; job += npairs) {
          int rb, sp;
          pair_job(p, job, rb, sp);
          const int row_a = p.row_offset + rb * 128 + (int)rank * kRowsCta;
          const int t0 = sp * p.tiles_per_split, t1 = min(t0 + p.tiles_per_split, p.n_tiles);
          if (kSparse && p.flags &&
              !job_has_tiles(p.flags + (size_t)rb * p.n_tiles, t0, t1)) continue;   // jj counts processed jobs only
          const uint32_t jpar = jj++ & 1;
          mbar_wait_t(bar(kJobDone), jpar ^ 1, 8, leader);
          if (leader) mbar_arrive_expect_tx(bar(kAFull), (kResLo ? 2u : 1u) * 2u * 2u * nkc * kChunkBytes);
          for (int c = 0; c < 2 * nkc; ++c)
            tma_load_2d_pair(base + kOffA + c * kChunkBytes, &map_a_hi, bar(kAFull), c * 64, row_a);
          if (kResLo)
            for (int c = 0; c < 2 * nkc; ++c)
              tma_load_2d_pair(base + kOffAlo + c * kChunkBytes, &map_a_lo, bar(kAFull), c * 64, row_a);
          for (int t = t0; t < t1; ++t) {
            if (kSparse && p.flags) { t = next_flagged(p.flags + (size_t)rb * p.n_tiles, t, t1); if (t >= t1) break; }
            // kBwdW: a tile without soft-target mass needs S only - no T_j planes, no I_i lo
            const bool zt = !kW || !p.flags || p.flags[(size_t)rb * p.n_tiles + t] != 0;
            const int j0 = t * kTileN + 32 * (int)rank, j1 = j0 + 64;
            for (int c = 0; c < nkc; ++c) {
              const int ci = c * 64, ct = D + c * 64;
              uint32_t fb;
              auto acquire = [&](uint32_t bytes) -> uint32_t {  // next ring slot: wait until the MMAs released it, arm its barrier
                const uint32_t slot = it % kSlots, par = (it / kSlots) & 1;
                ++it;
                mbar_wait_t(bar(kEmpty0 + slot), par ^ 1, 9, leader);
                fb = bar(kFull0 + slot);
                if (leader) MC_RING_ARM(fb, bytes);
                return base + kOffRing + slot * kSlotBytes;
              };
              if (PASSES == 3) {
                uint32_t sb;
                if (!kResLo) {
                  sb = acquire(zt ? 2u * kSlotBytes : 2u * kChunkBytes);
                  if (zt) MC_RING_LOAD(sb, &map_a_lo, fb, ci, row_a);               // I_i lo
                  MC_RING_LOAD(sb + kChunkBytes, &map_a_lo, fb, ct, row_a);         // T_i lo
                }
                sb = acquire(2u * kSlotBytes);
                MC_RING_LOAD(sb, &map_b_hi, fb, ci, j0);                            // I_j hi
                MC_RING_LOAD(sb + 4096, &map_b_hi, fb, ci, j1);
                MC_RING_LOAD(sb + kChunkBytes, &map_b_lo, fb, ci, j0);              // I_j lo
                MC_RING_LOAD(sb + kChunkBytes + 4096, &map_b_lo, fb, ci, j1);
                if (zt) {
                  sb = acquire(2u * kSlotBytes);
                  MC_RING_LOAD(sb, &map_b_hi, fb, ct, j0);                          // T_j hi
                  MC_RING_LOAD(sb + 4096, &map_b_hi, fb, ct, j1);
                  MC_RING_LOAD(sb + kChunkBytes, &map_b_lo, fb, ct, j0);            // T_j lo
                  MC_RING_LOAD(sb + kChunkBytes + 4096, &map_b_lo, fb, ct, j1);
                }
              } else {
                const uint32_t sb = acquire(2u * kSlotBytes);
                MC_RING_LOAD(sb, &map_b_hi, fb, ci, j0);                            // I_j hi
                MC_RING_LOAD(sb + 4096, &map_b_hi, fb, ci, j1);
                MC_RING_LOAD(sb + kChunkBytes, &map_b_hi, fb, ct, j0);              // T_j hi
                MC_RING_LOAD(sb + kChunkBytes + 4096, &map_b_hi, fb, ct, j1);
              }
            }
          }
        }
        MC_PROF_TOTAL(10, prof_t0, leader);
      }
    } else if (warp == 2) {
      // ========================================================= TMA producer: X^T half tiles (gradient GEMMs)
      if (kIsBwd && elect_one()) {
        const uint32_t xt_bytes = (uint32_t)(D / 2) * 128u;  // D/2 rows x 64 j fp16
        uint32_t tt = 0;
        for (int job = pair_id; job < njobs; job += npairs) {
          int rb, sp;
          pair_job(p, job, rb, sp);
          const int t0 = sp * p.tiles_per_split, t1 = min(t0 + p.tiles_per_split, p.n_tiles);
          for (int t = t0; t < t1; ++t) {
            if (kSparse && p.flags) { t = next_flagged(p.flags + (size_t)rb * p.n_tiles, t, t1); if (t >= t1) break; }   // tt counts processed tiles
            const uint32_t tt_cur = tt++;
            (void)tt_cur;
            // kBwdW: T_j^T feeds the dZ GEMM only (dI's S part comes from the stored weights)
            const bool zt = !kW || !p.flags || p.flags[(size_t)rb * p.n_tiles + t] != 0;
            if (kW && !zt) {
              // no T_j^T tile: its buffer takes I_j^T of column half 1, so both halves load at once as soon as the
              // previous tile's gradient MMAs are done
              mbar_wait(bar(kGradDone1), (tt_cur & 1) ^ 1);
              for (int h = 0; h < 2; ++h) {
                const uint32_t fb = bar(h == 0 ? kXTFull : kXTFull1);
                if (leader) mbar_arrive_expect_tx(fb, 2u * xt_bytes);
                tma_load_2d_pair(base + kOffXT + h * xt_bytes, &map_t, fb, t * kTileN + 64 * h, (int)rank * (D / 2));
              }
              continue;
            }
            for (int h = 0; h < 2; ++h) {
              // the previous half's MMAs are done with the buffer: (tt-1, 1) before (tt, 0); (tt, 0) before (tt, 1)
              if (h == 0) mbar_wait(bar(kGradDone1), (tt_cur & 1) ^ 1); else mbar_wait(bar(kGradDone), tt_cur & 1);
              const uint32_t fb = bar((kW && h == 1) ? kXTFull1 : kXTFull);
              if (leader) mbar_arrive_expect_tx(fb, 2u * 2u * xt_bytes);
              const int jx = t * kTileN + 64 * h;
              tma_load_2d_pair(base + kOffXT, &map_t, fb, jx, (int)rank * (D / 2));
              tma_load_2d_pair(base + kOffXT + xt_bytes, &map_t, fb, jx, D + (int)rank * (D / 2));
            }
          }
        }
      }
    } else if (warp == 3 && kIsBwd && kIssuers == 1) {
      // ========================================================= per-column constants of the gradient sweep, one tile
      // ahead of the epilogue: -r2_j, -c2_j, B_j | -rz2_j, gh_j, D_j q_j | q_j, E_j (see weights32); lane l owns the
      // columns l, l + 32, l + 64, l + 96 of the tile
      float* const consts = reinterpret_cast<float*>(sbase + kOffConst);
      const float kL2e = 1.4426950408889634f;
      const bool fast = p.wscale[1] != 0.f;
      const float m_rc = p.wscale[2], m_z = p.wscale[3], twoB = 2.f * (float)p.B;
      uint32_t tt = 0;
      for (int job = pair_id; job < njobs; job += npairs) {
        int rb, sp;
        pair_job(p, job, rb, sp);
        const int t0 = sp * p.tiles_per_split, t1 = min(t0 + p.tiles_per_split, p.n_tiles);
        for (int t = t0; t < t1; ++t) {
          if (kSparse && p.flags) { t = next_flagged(p.flags + (size_t)rb * p.n_tiles, t, t1); if (t >= t1) break; }
          float vr[4], vc[4], vz[4], vg[4], vq[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int jcol = t * kTileN + lane + 32 * u;
            const bool ok = jcol < p.B;
            vr[u] = ok ? p.r[jcol] : 0.f; vc[u] = ok ? p.c[jcol] : 0.f; vz[u] = ok ? p.rz[jcol] : 0.f;
            vg[u] = ok ? p.g[jcol] : 0.f; vq[u] = ok ? p.q[jcol] : 0.f;
          }
          mbar_wait(bar(kCstEmpty0 + (tt & 1)), ((tt >> 1) & 1) ^ 1);
          float* dst = consts + (tt & 1) * (8 * 128);
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int col = lane + 32 * u;
            const bool ok = t * kTileN + col < p.B;
            const float r2 = vr[u] * kL2e, c2 = vc[u] * kL2e, rz2 = vz[u] * kL2e;
            dst[0 * 128 + col] = -r2;
            dst[1 * 128 + col] = -c2;
            dst[3 * 128 + col] = vg[u] * twoB * kL2e;
            if (fast) {
              dst[2 * 128 + col] = ok ? ex2f(m_z - rz2) : 0.f;
              dst[4 * 128 + col] = ok ? ex2f(m_rc - c2) * vq[u] : 0.f;
              dst[5 * 128 + col] = ok ? ex2f(r2 - m_rc) : 0.f;
            } else {
              dst[2 * 128 + col] = -rz2;
              dst[4 * 128 + col] = vq[u];
            }
          }
          mbar_arrive_local(bar(kCstFull0 + (tt & 1)));
          ++tt;
        }
      }
    } else if (warp == 1 || (kIssuers == 2 && warp == 3)) {
      // ========================================================= MMA issuer (leader CTA, one elected lane:
      // inside elect.sync the compiler knows a single thread is active and feeds the uniform-register
      // operands of UTCHMMA from vector registers without a per-lane waterfall loop).
      // kIssuers == 2 splits the stream over warps 1 (S, St, dT) and 3 (Z, dI); measured SLOWER on
      // B200 (the 128 x 128 x 16 pair MMA itself sustains ~45 cycles, not the issuing thread), kept off.
      const bool do_s = kIssuers == 1 || warp == 1, do_z = kIssuers == 1 || warp == 3;
      if (leader && elect_one()) {
        constexpr uint32_t idesc_tile = idesc_f16(128, kTileN);
        const uint32_t idesc_grad = idesc_f16(128, D);
        const uint32_t tDT = tmem_base + kAccCol, tDI = tDT + (uint32_t)(D / 2);
        const uint32_t xt_bytes = (uint32_t)(D / 2) * 128u;
        const uint64_t wS = smem_desc_sw128(base + kOffW), wSt = smem_desc_sw128(base + kOffW + kChunkBytes);
        const uint64_t wZ = smem_desc_sw128(base + kOffW + 2 * kChunkBytes);
        const uint64_t xI = smem_desc_sw128(base + kOffXT), xT = smem_desc_sw128(base + kOffXT + xt_bytes);
        uint32_t it = 0, tt = 0, hh = 0, jj = 0;
        [[maybe_unused]] const long long prof_t0 = MC_PROF_NOW();
        // one column half of a tile's gradient GEMMs: dT += W_S I_j + W_Z T_j, dI += W_St T_j + W_Z I_j
        bool zg = true;  // does the tile whose gradient GEMMs are being issued carry soft-target mass (tile flag)?
        bool di_live = false;  // kBwdW: has this job's dI accumulator been written yet (only flagged tiles touch it)?
        auto grad_half = [&](int h, bool first_of_job) {
          if (kW) {   // per-half buffers and barriers: one phase per tile
            mbar_wait_t(bar(h == 0 ? kWFull : kWFull1), (hh >> 1) & 1, 3, true);
            mbar_wait_t(bar(h == 0 ? kXTFull : kXTFull1), (hh >> 1) & 1, 4, true);
          } else {
            mbar_wait_t(bar(kWFull), hh & 1, 3, true);
            mbar_wait_t(bar(kXTFull), hh & 1, 4, true);
          }
          ++hh;
          tc_fence_after();
          const uint32_t first = (first_of_job && h == 0) ? 0u : 1u;
          // kBwdW: half 1 has its own weight buffer (the unused dS^T slot) and, on tiles without soft-target mass, its
          // own I_j^T buffer (the unused T_j^T slot)
          const uint64_t wS_h = (kW && h == 1) ? wSt : wS;
          const uint64_t xI_h = (kW && h == 1 && !zg) ? xT : xI;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint32_t acc = (first | (ks > 0)) ? 1u : 0u;
            const uint64_t kxI = desc_advance_k(xI_h, ks), kxT = desc_advance_k(xT, ks);
            const uint64_t kwZ = desc_advance_k(wZ, ks);
            if (do_s) {
              mma_f16_pair(tDT, desc_advance_k(wS_h, ks), kxI, idesc_grad, acc);   // dT += (dS/tau) I_j
              if (zg) mma_f16_pair(tDT, kwZ, kxT, idesc_grad, 1u);               // dT += (tau/2 dZs) T_j
            }
            if (do_z) {
              if (kW) {
                if (zg) mma_f16_pair(tDI, kwZ, kxI, idesc_grad, (di_live || ks > 0) ? 1u : 0u);  // dI += (tau/2 dZs) I_j
              } else {
                mma_f16_pair(tDI, desc_advance_k(wSt, ks), kxT, idesc_grad, acc);  // dI += (dS^T/tau) T_j
                if (zg) mma_f16_pair(tDI, kwZ, kxI, idesc_grad, 1u);               // dI += (tau/2 dZs) I_j
              }
            }
          }
          if (zg) di_live = true;
          mma_commit_pair(bar(h == 0 ? kGradDone : kGradDone1), 3);
        };
        for (int job = pair_id; job < njobs; job += npairs) {
          int rb, sp;
          pair_job(p, job, rb, sp);
          const int t0 = sp * p.tiles_per_split, t1 = min(t0 + p.tiles_per_split, p.n_tiles);
          const uint8_t* frow = p.flags ? p.flags + (size_t)rb * p.n_tiles : nullptr;
          if (kSparse && frow && !job_has_tiles(frow, t0, t1)) continue;
          const uint32_t jpar = jj++ & 1;
          mbar_wait_t(bar(kAFull), jpar, 0, true);
          tc_fence_after();
          bool zf = true, zf_prev = true;
          di_live = false;
          int nproc = 0;   // tiles of this job issued so far (sparse phases skip tiles)
          const bool zprobe = PHASE == kStats && p.flags_out != nullptr;  // Z from the hi planes only
          for (int t = t0; t < t1; ++t) {
            if (kSparse && frow) { t = next_flagged(frow, t, t1); if (t >= t1) break; }   // every role skips the same tiles
            zf_prev = zf;
            zf = !kIsBwd || !frow || frow[t] != 0;                 // gradient sweep: recompute Z only where P lives
            zg = zf_prev;                                          // the woven gradient GEMMs belong to tile t - 1
            const uint32_t buf = tt % kNBuf, use = tt / kNBuf;
            mbar_wait_t(bar(kTmemEmpty0 + buf), (use & 1) ^ 1, 1, true);
            tc_fence_after();
            const uint32_t tS = tmem_base + buf * 192, tSt = tS + 64, tZ = tS + 128;
            // The gradient GEMMs of tile t-1 are woven into the recompute of tile t: half 0 after the
            // first chunks (its weights are ready by then), half 1 after the last chunk, so the
            // single weight / X^T buffers are refilled while the tensor cores stay busy.
            const bool lagged = kIsBwd && nproc > 0;
            for (int c = 0; c < nkc; ++c) {
              if (!kW && lagged && c == nkc - 1) grad_half(0, nproc == 1);
              uint32_t slot_bar = 0;
              auto next_full = [&]() -> uint32_t {  // wait for the next ring slot to land
                const uint32_t slot = it % kSlots, par = (it / kSlots) & 1;
                ++it;
                mbar_wait_t(bar(kFull0 + slot), par, 2, true);
                tc_fence_after();
                slot_bar = bar(kEmpty0 + slot);
                return base + kOffRing + slot * kSlotBytes;
              };
              const uint64_t aI = smem_desc_sw128(base + kOffA + c * kChunkBytes);
              const uint64_t aT = smem_desc_sw128(base + kOffA + (nkc + c) * kChunkBytes);
              const uint32_t first = (c > 0) ? 1u : 0u;
              if (PASSES == 3) {
                uint32_t a_bar = 0;
                uint64_t aIl, aTl;
                if (kResLo) {
                  aIl = smem_desc_sw128(base + kOffAlo + c * kChunkBytes);
                  aTl = smem_desc_sw128(base + kOffAlo + (nkc + c) * kChunkBytes);
                } else {
                  const uint32_t sa = next_full();
                  a_bar = slot_bar;
                  aIl = smem_desc_sw128(sa);
                  aTl = smem_desc_sw128(sa + kChunkBytes);
                }
                uint32_t sb = next_full();
                {
                  const uint64_t bI = smem_desc_sw128(sb), bIl = smem_desc_sw128(sb + kChunkBytes);
#pragma unroll
                  for (int ks = 0; ks < 4; ++ks) {
                    const uint32_t acc = (first | (ks > 0)) ? 1u : 0u;
                    const uint64_t kI = desc_advance_k(aI, ks), kT = desc_advance_k(aT, ks);
                    const uint64_t kb = desc_advance_k(bI, ks), kbl = desc_advance_k(bIl, ks);
                    if (do_s && PHASE != kRowLoss) {
                      mma_f16_pair(tS, kT, kb, idesc_tile, acc);                       // S  = T_i I_j^T
                      mma_f16_pair(tS, kT, kbl, idesc_tile, 1u);
                      mma_f16_pair(tS, desc_advance_k(aTl, ks), kb, idesc_tile, 1u);
                    }
                    if (do_z && zf) {
                      mma_f16_pair(tZ, kI, kb, idesc_tile, acc);                       // Z += I_i I_j^T
                      if (!zprobe) {
                        mma_f16_pair(tZ, kI, kbl, idesc_tile, 1u);
                        mma_f16_pair(tZ, desc_advance_k(aIl, ks), kb, idesc_tile, 1u);
                      }
                    }
                  }
                }
                mma_commit_pair(slot_bar, 3);
                if (!kW || zf) {   // kBwdW: no T_j slot in the ring for a tile without soft-target mass
                sb = next_full();
                {
                  const uint64_t bT = smem_desc_sw128(sb), bTl = smem_desc_sw128(sb + kChunkBytes);
#pragma unroll
                  for (int ks = 0; ks < 4; ++ks) {
                    const uint32_t acc = (first | (ks > 0)) ? 1u : 0u;
                    const uint64_t kI = desc_advance_k(aI, ks), kT = desc_advance_k(aT, ks);
                    const uint64_t kb = desc_advance_k(bT, ks), kbl = desc_advance_k(bTl, ks);
                    if (do_s) {
                      if (PHASE != kRowLoss && PHASE != kStatsZ && !(PHASE == kStats && p.colpart)) {
                        mma_f16_pair(tSt, kI, kb, idesc_tile, acc);                    // St = I_i T_j^T
                        mma_f16_pair(tSt, kI, kbl, idesc_tile, 1u);
                        mma_f16_pair(tSt, desc_advance_k(aIl, ks), kb, idesc_tile, 1u);
                      }
                    }
                    if (do_z && zf) {
                      mma_f16_pair(tZ, kT, kb, idesc_tile, 1u);                        // Z += T_i T_j^T
                      if (!zprobe) {
                        mma_f16_pair(tZ, kT, kbl, idesc_tile, 1u);
                        mma_f16_pair(tZ, desc_advance_k(aTl, ks), kb, idesc_tile, 1u);
                      }
                    }
                  }
                }
                mma_commit_pair(slot_bar, 3);
                }
                if (!kResLo) mma_commit_pair(a_bar, 3);
              } else {
                const uint32_t sb = next_full();
                const uint64_t bI = smem_desc_sw128(sb), bT = smem_desc_sw128(sb + kChunkBytes);
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                  const uint32_t acc = (first | (ks > 0)) ? 1u : 0u;
                  const uint64_t kI = desc_advance_k(aI, ks), kT = desc_advance_k(aT, ks);
                  const uint64_t kbI = desc_advance_k(bI, ks), kbT = desc_advance_k(bT, ks);
                  if (do_s && PHASE != kRowLoss) {
                    mma_f16_pair(tS, kT, kbI, idesc_tile, acc);
                    if (PHASE != kStatsZ && !(PHASE == kStats && p.colpart) && (!kW || zf)) mma_f16_pair(tSt, kI, kbT, idesc_tile, acc);
                  }
                  if (do_z && zf) {
                    mma_f16_pair(tZ, kI, kbI, idesc_tile, acc);
                    mma_f16_pair(tZ, kT, kbT, idesc_tile, 1u);
                  }
                }
                mma_commit_pair(slot_bar, 3);
              }
            }
            mma_commit_pair(bar(kTmemFull0 + buf), 3);
            if (kIsBwd) {
              if (nproc == 0) {
                mbar_wait_t(bar(kAccEmpty), jpar ^ 1, 5, true);  // the previous job's accumulators were read out
                tc_fence_after();
              } else {
                // kBwdW: nothing is woven - with per-half buffers the whole tile t is issued (and handed to the
                // epilogue) before the issuer waits for the weights of tile t - 1
                if (kW) grad_half(0, nproc == 1);
                grad_half(1, false);
              }
            }
            ++nproc;
            ++tt;
          }
          if (kIsBwd) {
            zg = zf;  // the last tile's own gradient GEMMs
            grad_half(0, nproc == 1);
            grad_half(1, false);
            mma_commit_pair(bar(kAccFull), 3);
          }
          mma_commit_pair(bar(kJobDone), 3);
        }
        MC_PROF_TOTAL(6, prof_t0, true);
      }
    }
    __syncwarp();
  } else {
    // =========================================================== epilogue: two threads per TMEM lane
    // Warps 4-7 take the first 32 TMEM columns of every tile, warps 8-11 the second 32 (column half h).
    // Everything inside exponentials lives in the log2 domain (ex2.approx); the raw accumulators are
    // products of the scaled planes, so S = acc * inv_s2 / tau and Z = acc * inv_s2 * tau / 2.
    const int quarter = warp & 3;
    const int h = (warp - 4) >> 2;
    const int lane_t = quarter * 32 + lane;
    const int m = lane_t & 63, n1 = lane_t >> 6;
    const int tid_e = threadIdx.x - 128;  // 0..255
    const uint32_t lane_field = (uint32_t)(quarter * 32) << 16;
    const int jl0 = 64 * h + 32 * n1;     // first tile column of this thread's 32
    float* const consts = reinterpret_cast<float*>(sbase + kOffConst);  // [2 buffers][8 fields][128 columns]
    const float kL2e = 1.4426950408889634f;
    const float inv_s = p.scale[1], inv_s2 = p.scale[2];
    const float cS2 = inv_s2 * p.inv_tau * kL2e, cZ2 = inv_s2 * p.half_tau * kL2e;  // raw acc -> log2 domain
    const float m2cS2 = -2.f * cS2;
    uint32_t tt = 0, jj = 0, jp = 0;   // jp: processed jobs (sparse phases skip jobs)
    [[maybe_unused]] const bool prof_rec = leader && (threadIdx.x == 128 || threadIdx.x == 256);
    [[maybe_unused]] const int prof_base = threadIdx.x == 128 ? 16 : 24;
    [[maybe_unused]] const long long prof_t0 = MC_PROF_NOW();
    for (int job = pair_id; job < njobs; job += npairs, ++jj) {
      int rb, sp;
      pair_job(p, job, rb, sp);
      const int t0 = sp * p.tiles_per_split, t1 = min(t0 + p.tiles_per_split, p.n_tiles);
      const int lrow = rb * 128 + (int)rank * kRowsCta + m;  // row within this rank's strip
      const int gi = p.row_offset + lrow;
      const bool row_ok = lrow < p.b;
      if (kSparse && p.flags &&
          !job_has_tiles(p.flags + (size_t)rb * p.n_tiles, t0, t1)) {
        // no flagged tile in this (row block, column split): the other roles skip the job too; its partials are empty
        if (kP) continue;   // the caller zeroed the gradient partials
        if (2 * h + n1 == 0) {
          if (PHASE == kStatsZ) {
            float2* out = reinterpret_cast<float2*>(p.part);
            const size_t o = (size_t)sp * 4 * p.bpad + lrow;
            out[o + 2 * (size_t)p.bpad] = make_float2(-INFINITY, 0.f);
            out[o + 3 * (size_t)p.bpad] = make_float2(0.f, 0.f);
          } else {
            const size_t o = (size_t)sp * 2 * p.bpad + lrow;
            p.part[o] = 0.f;
            p.part[o + p.bpad] = 0.f;
          }
        }
        continue;
      }
      // per-row statistics, log2 domain: r2 = r log2(e), ... ; gh = 2B g log2(e)
      float r2_i = 0.f, c2_i = 0.f, rz2_i = 0.f, gh_i = 0.f, q_i = 0.f;
      if (PHASE != kStats && PHASE != kStatsZ && row_ok) { r2_i = p.r[gi] * kL2e; c2_i = p.c[gi] * kL2e; rz2_i = p.rz[gi] * kL2e; }
      if (kIsBwd && row_ok) { gh_i = p.g[gi] * (2.f * (float)p.B) * kL2e; q_i = p.q[gi]; }
      float wS = 0.f, wZ = 0.f;
      bool fast = false;
      float m_rc = 0.f, m_z = 0.f, fA_i = 0.f, fC_i = 0.f, fFQ_i = 0.f;
      if (kIsBwd) {
        const float wsc = p.wscale[0];
        wS = inv_s * p.inv_tau * wsc;              // 2B dS      -> fp16 weight of X_j (scaled plane)
        wZ = inv_s * p.half_tau * wsc * kLn2;      // 2B dZs (log2 units) -> fp16 weight
        fast = p.wscale[1] != 0.f;                 // kernel-uniform: see wscale_kernel
        m_rc = p.wscale[2];
        m_z = p.wscale[3];
        fA_i = ex2f(rz2_i - m_z);                  // P_ji          = P_ij          * fA_i * B_j
        fC_i = ex2f(r2_i - m_rc);                  // e^{S_ij-c_j}  = e^{S_ij-r_i}  * fC_i * D_j
        fFQ_i = ex2f(m_rc - c2_i) * q_i;           // e^{S_ji-c_i} q_i = e^{S_ji-r_j} * E_j * fFQ_i
      }
      float mS = -INFINITY, sS = 0.f, mSt = -INFINITY, sSt = 0.f, mZ = -INFINITY, sZ = 0.f;  // raw-domain max, sums
      float aPS = 0.f;  // sum_j e^{Z_ij - mZ} S_ij in raw accumulator units
      float ps2_i = 0.f;
      if (PHASE == kRowLoss && row_ok) ps2_i = p.ps[lrow] * kL2e;  // sum_j P_ij S_ij, log2 units
      float ag4[4] = {0.f, 0.f, 0.f, 0.f}, aq4[4] = {0.f, 0.f, 0.f, 0.f};
      const uint8_t* frow = p.flags ? p.flags + (size_t)rb * p.n_tiles : nullptr;
      // tile flags (statistics sweep): rz_i >= Z_ii = (|I_i|^2 + |T_i|^2) tau / 2, so a tile whose largest Z_ij stays
      // kFlagTheta2 binades below max(Z_ii, running maximum) cannot hold a P_ij above 2^-44
      float zii2 = 0.f;
      // rounding of the probe: the hi planes carry 2^-11 relative error per element, so |dZ_ij| <= 2^-10 sqrt(Z_ii Z_jj)
      // <= 2^-10 max_k Z_kk, and every |x| is below 2 / s (the planes' scale), i.e. Z_kk < 2 D (2/s)^2 tau/2
      const float zmargin2 = kProbeMargin2 + (1.f / 512.f) * (8.f * (float)D * inv_s2 * p.half_tau * kL2e);
      if (PHASE == kStats && p.flags_out && row_ok) {
        const float ni = p.norm_i[gi], nt = p.norm_t[gi];
        zii2 = (ni * ni + nt * nt) * p.half_tau * kL2e;
      }

      for (int t = t0; t < t1; ++t) {
        if (kSparse && frow) { t = next_flagged(frow, t, t1); if (t >= t1) break; }       // every role skips the same tiles
        const bool zf = !kIsBwd || !frow || frow[t] != 0;          // gradient sweep: does this tile carry P mass?
        // ---- per-column statistics of this tile -> shared memory, one field per 128-float row
        float* cst = consts + (tt & 1) * (8 * 128);
        if (kIsBwd) {
          // the per-column constants of this tile come from warp 3, one tile ahead (no global loads, no block barrier here)
          mbar_wait_t(bar(kCstFull0 + (tt & 1)), (tt >> 1) & 1, prof_base + 0, prof_rec);
        } else if (PHASE != kStats && PHASE != kStatsZ) {
          if (tid_e < 128) {
            const int jcol = t * kTileN + tid_e;
            const bool ok = jcol < p.B;
            const float c2 = ok ? p.c[jcol] * kL2e : 0.f, rz2 = ok ? p.rz[jcol] * kL2e : 0.f;
            cst[1 * 128 + tid_e] = -c2;                                                                 // -c2_j
            cst[2 * 128 + tid_e] = -rz2;                                                                // -rz2_j
          }
          named_bar_sync(1, kEpiThreads);
        }
        const bool ragged = (t + 1) * kTileN > p.B;  // last tile of a batch that is not a multiple of 128
        const int jlim = p.B - t * kTileN;           // columns jl < jlim are real
        const uint32_t buf = tt % kNBuf, use = tt / kNBuf;
        mbar_wait_t(bar(kTmemFull0 + buf), use & 1, prof_base + 1, prof_rec);
        tc_fence_after();
        const uint32_t tS = tmem_base + buf * 192 + lane_field + 32 * h, tSt = tS + 64, tZ = tS + 128;

        // this thread's 32 columns of the three tiles go to registers at once; the tile buffer is
        // handed back to the tensor cores before any arithmetic starts
        float vs[32], vt[32], vz[32];
        if (PHASE != kRowLoss) tmem_ld32(tS, vs);
        const bool colpart = PHASE == kStats && p.colpart != nullptr;
        if (PHASE != kRowLoss && PHASE != kStatsZ && !colpart && (!kW || zf)) tmem_ld32(tSt, vt);
        if (zf) tmem_ld32(tZ, vz);   // a tile without soft-target mass has no Z accumulator at all
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive_cluster(bar(kTmemEmpty0 + buf), 0);

        if (PHASE == kStats || PHASE == kStatsZ) {
#ifndef MC_ABLATE_EPI
          const bool zprobe = PHASE == kStats && p.flags_out != nullptr;
          auto lse_add32 = [&](float* v, float c, float& mx, float& sm) {
            if (ragged) {
#pragma unroll
              for (int e = 0; e < 32; ++e) if (jl0 + e >= jlim) v[e] = -INFINITY;
            }
            float c4[4] = {fmaxf(v[0], v[4]), fmaxf(v[1], v[5]), fmaxf(v[2], v[6]), fmaxf(v[3], v[7])};
#pragma unroll
            for (int e = 8; e < 32; e += 4) {  // four independent chains
#pragma unroll
              for (int u = 0; u < 4; ++u) c4[u] = fmaxf(c4[u], v[e + u]);
            }
            const float cm = fmaxf(fmaxf(c4[0], c4[1]), fmaxf(c4[2], c4[3]));
            const float mn = fmaxf(mx, cm);
            if (mn == -INFINITY) return;
            // (v - mn) * c, not fma(v, c, -mn c): the difference is exact, so an unchanged maximum
            // rescales the running sum by exactly 1 (a rounded offset would compound over the row)
            float a4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int e = 0; e < 32; e += 4) {
#pragma unroll
              for (int u = 0; u < 4; ++u) a4[u] += ex2f((v[e + u] - mn) * c);
            }
            sm = sm * ex2f((mx - mn) * c) + ((a4[0] + a4[1]) + (a4[2] + a4[3]));
            mx = mn;
          };
          {  // Z first: besides its log-sum-exp, accumulate aPS = sum_j e^{Z_ij - max} S_ij (raw S units) so
             // that the row-loss sweep does not have to recompute S.  Padding columns have vz = -inf, vs = 0.
            if (ragged) {
#pragma unroll
              for (int e = 0; e < 32; ++e) if (jl0 + e >= jlim) vz[e] = -INFINITY;
            }
            float c4[4] = {fmaxf(vz[0], vz[4]), fmaxf(vz[1], vz[5]), fmaxf(vz[2], vz[6]), fmaxf(vz[3], vz[7])};
#pragma unroll
            for (int e = 8; e < 32; e += 4) {
#pragma unroll
              for (int u = 0; u < 4; ++u) c4[u] = fmaxf(c4[u], vz[e + u]);
            }
            const float cmz = fmaxf(fmaxf(c4[0], c4[1]), fmaxf(c4[2], c4[3]));
            if (zprobe) {  // rz_i >= Z_ii: a tile whose (hi-plane) Z stays this far below it holds no P_ij >= 2^-44
              const bool hit = row_ok && cmz * cZ2 >= zii2 - kFlagTheta2 - zmargin2;
              if (__any_sync(0xffffffffu, hit) && lane == 0) p.flags_out[(size_t)rb * p.n_tiles + t] = 1;
            }
            const float mn = fmaxf(mZ, cmz);
            if (!zprobe && mn != -INFINITY) {
              float a4[4] = {0.f, 0.f, 0.f, 0.f}, b4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
              for (int e = 0; e < 32; e += 4) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  const float w = ex2f((vz[e + u] - mn) * cZ2);
                  a4[u] += w;
                  b4[u] = fmaf(w, vs[e + u], b4[u]);
                }
              }
              const float resc = ex2f((mZ - mn) * cZ2);
              sZ = sZ * resc + ((a4[0] + a4[1]) + (a4[2] + a4[3]));
              aPS = aPS * resc + ((b4[0] + b4[1]) + (b4[2] + b4[3]));
              mZ = mn;
            }
          }
          if (PHASE == kStats) {
            lse_add32(vs, cS2, mS, sS);
            if (!colpart) {
              lse_add32(vt, cS2, mSt, sSt);
            } else {
              // ---- column LSE without the transposed strip.  This warp holds a 32 x 32 block (lane = row, vs[c] =
              // column jl0 + c).  (1) column maxima by a transpose-reduce: five exchange steps, each halves the values
              // a lane keeps (lane bit set -> upper half), after which lane l owns column l; (2) every lane fetches all
              // 32 maxima through shared memory; (3) exponentials against the column's OWN maximum (exact, no reference
              // shared with other columns can underflow); (4) the same transpose-reduce with a sum; lane l writes
              // max_l + log2(sum_l).  Rows beyond the strip count as -inf.
              float a[32];
#pragma unroll
              for (int e = 0; e < 32; ++e) a[e] = row_ok ? vs[e] : -INFINITY;
#pragma unroll
              for (int s = 16; s >= 1; s >>= 1) {
                const bool up = (lane & s) != 0;
#pragma unroll
                for (int k = 0; k < s; ++k) {
                  const float keep = up ? a[k + s] : a[k], send = up ? a[k] : a[k + s];
                  a[k] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, s));
                }
              }
              float* cmx = consts + (warp - 4) * 32;   // the column constants are not used by this phase
              __syncwarp();
              cmx[lane] = a[0];
              __syncwarp();
              const float cm_own = a[0];
#pragma unroll
              for (int e = 0; e < 32; e += 4) {
                const float4 c4 = *reinterpret_cast<const float4*>(cmx + e);
                const float cmv[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  const float ref = cmv[u] == -INFINITY ? 0.f : cmv[u];
                  a[e + u] = row_ok ? ex2f((vs[e + u] - ref) * cS2) : 0.f;
                }
              }
#pragma unroll
              for (int s = 16; s >= 1; s >>= 1) {
                const bool up = (lane & s) != 0;
#pragma unroll
                for (int k = 0; k < s; ++k) {
                  const float keep = up ? a[k + s] : a[k], send = up ? a[k] : a[k + s];
                  a[k] = keep + __shfl_xor_sync(0xffffffffu, send, s);
                }
              }
              const int g32 = (rb * 128 + (int)rank * kRowsCta + (quarter & 1) * 32) >> 5;   // 32-row group of the strip
              p.colpart[(size_t)g32 * p.Bp + (size_t)t * kTileN + jl0 + lane] =
                  cm_own == -INFINITY ? -INFINITY : fmaf(cm_own, cS2, lg2f(a[0]));
            }
          }
#endif
        } else if (PHASE == kRowLoss) {
          if (ragged) {
#pragma unroll
            for (int e = 0; e < 32; ++e) if (jl0 + e >= jlim) vz[e] = -INFINITY;
          }
#pragma unroll
          for (int e = 0; e < 32; e += 4) {
            const float4 nc = *reinterpret_cast<const float4*>(cst + 1 * 128 + jl0 + e);
            const float4 nrz = *reinterpret_cast<const float4*>(cst + 2 * 128 + jl0 + e);
            const float ncv[4] = {nc.x, nc.y, nc.z, nc.w}, nrzv[4] = {nrz.x, nrz.y, nrz.z, nrz.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {  // four independent accumulation chains
              const float z2 = vz[e + u] * cZ2;
              const float P = ex2f(z2 - rz2_i);
              ag4[u] = fmaf(P, -ncv[u], ag4[u]);   // sum_j P_ij c_j (log2 units)
              aq4[u] += ex2f(z2 + nrzv[u]);        // sum_j e^{Z_ij - rz_j} = colsum(P)_i by symmetry
            }
          }
        } else {
          // ---- gradient sweep: tile -> fp16 weight half-tile h -> tensor cores
          uint32_t wSp[16], wStp[16], wZp[16];
          auto weights32 = [&](auto fast_tag, auto z_tag) {
            constexpr bool kFast = decltype(fast_tag)::value;
            constexpr bool kZ = decltype(z_tag)::value;   // false: P_ij = P_ji = 0 on the whole tile (flag 0)
#pragma unroll
            for (int e = 0; e < 32; e += 4) {
              const float4 f0 = *reinterpret_cast<const float4*>(cst + 0 * 128 + jl0 + e);  // -r2_j
              const float4 f1 = *reinterpret_cast<const float4*>(cst + 1 * 128 + jl0 + e);  // -c2_j
              const float4 f2 = *reinterpret_cast<const float4*>(cst + 2 * 128 + jl0 + e);  // -rz2_j | B_j
              const float4 f3 = *reinterpret_cast<const float4*>(cst + 3 * 128 + jl0 + e);  // gh_j
              const float4 f4 = *reinterpret_cast<const float4*>(cst + 4 * 128 + jl0 + e);  // q_j | D_j q_j
              const float4 f5 = kFast ? *reinterpret_cast<const float4*>(cst + 5 * 128 + jl0 + e)  // E_j
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
              const float nr[4] = {f0.x, f0.y, f0.z, f0.w}, nc[4] = {f1.x, f1.y, f1.z, f1.w};
              const float zc[4] = {f2.x, f2.y, f2.z, f2.w}, gh[4] = {f3.x, f3.y, f3.z, f3.w};
              const float qc[4] = {f4.x, f4.y, f4.z, f4.w}, ej[4] = {f5.x, f5.y, f5.z, f5.w};
              float ms[4], mst[4], mz[4];
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                // kBwdW: the transposed strip exists on flagged tiles only (kZ) and feeds G_ji alone - dS_ji is not formed
                const float a = vs[e + u], bt = (!kW || kZ) ? vt[e + u] : 0.f;
                const float e1 = kP ? 0.f : ex2f(fmaf(a, cS2, -r2_i));     // softmax_row(S)_ij (kBwdP: rowgrad_kernel's part)
                const float e3 = (kW || kP) ? 0.f : ex2f(fmaf(bt, cS2, nr[u]));    // softmax_row(S)_ji
                float P = 0.f, Pt = 0.f, dS, dSt = 0.f;
                if (kZ) {
                  const float z2 = vz[e + u] * cZ2;
                  P = ex2f(z2 - rz2_i);
                  Pt = kFast ? P * (fA_i * zc[u]) : ex2f(z2 + zc[u]);
                }
                if (kFast) {  // three exponentials; the other three are products of per-row / per-column factors
                  dS = fmaf(e1, fmaf(fC_i, qc[u], 1.f), -2.f * P);        // 2B dS_ij
                  if (!kW) dSt = fmaf(e3, fmaf(ej[u], fFQ_i, 1.f), -2.f * Pt);     // 2B dS_ji
                } else {
                  const float e2 = kP ? 0.f : ex2f(fmaf(a, cS2, nc[u]));   // softmax_col(S)_ij
                  dS = fmaf(-2.f, P, fmaf(e2, qc[u], e1));
                  if (!kW) {
                    const float e4 = kP ? 0.f : ex2f(fmaf(bt, cS2, -c2_i));  // softmax_col(S)_ji
                    dSt = fmaf(-2.f, Pt, fmaf(e4, q_i, e3));
                  }
                }
                ms[u] = (kW && !row_ok) ? 0.f : dS * wS;   // kBwdW: rows past the strip must store exact zeros
                mst[u] = dSt * wS;
                if (kZ) {
                  const float G = fmaf(a, m2cS2, r2_i - nc[u]);           // 2B G_ij log2(e)
                  const float Gt = fmaf(bt, m2cS2, c2_i - nr[u]);         // 2B G_ji log2(e)
                  mz[u] = fmaf(P, G - gh_i, Pt * (Gt - gh[u])) * wZ;      // 2B dZs (log2 units) * scale
                } else {
                  mz[u] = 0.f;
                }
              }
#pragma unroll
              for (int u = 0; u < 4; u += 2) {
                __half2 x = __floats2half2_rn(ms[u], ms[u + 1]), y = __floats2half2_rn(mst[u], mst[u + 1]);
                __half2 w = __floats2half2_rn(mz[u], mz[u + 1]);
                wSp[(e + u) >> 1] = *reinterpret_cast<uint32_t*>(&x);
                wStp[(e + u) >> 1] = *reinterpret_cast<uint32_t*>(&y);
                wZp[(e + u) >> 1] = *reinterpret_cast<uint32_t*>(&w);
              }
            }
          };
          if (zf) {
            if (fast) weights32(std::true_type{}, std::true_type{}); else weights32(std::false_type{}, std::true_type{});
          } else {
            if (fast) weights32(std::true_type{}, std::false_type{}); else weights32(std::false_type{}, std::false_type{});
          }
          // The single weight buffer is used by column half 0, then half 1, of every tile: wait until
          // the gradient MMAs of the preceding half have drained it.  One barrier per half keeps every
          // waiter at most one phase behind, which the parity test needs.
          if (h == 0 || (kW && !zf)) mbar_wait_t(bar(kGradDone1), (tt & 1) ^ 1, prof_base + 2, prof_rec);  // half 1 of the previous tile consumed
          else mbar_wait_t(bar(kGradDone), tt & 1, prof_base + 2, prof_rec);                // half 0 of this tile consumed (shared dZ buffer)
          // row m of a 64 x 64 fp16 tile (128 B rows, SWIZZLE_128B): this thread owns K = 32 n1 .. +31
          uint8_t* wrow = sbase + kOffW + m * 128;
          uint8_t* wrow_s = wrow + ((kW && h == 1) ? kChunkBytes : 0);   // kBwdW: half 1 writes the dS^T slot
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int chunk = ((4 * n1 + k) ^ (m & 7)) * 16;
            *reinterpret_cast<uint4*>(wrow_s + chunk) = make_uint4(wSp[4 * k], wSp[4 * k + 1], wSp[4 * k + 2], wSp[4 * k + 3]);
            if (!kW)
              *reinterpret_cast<uint4*>(wrow + kChunkBytes + chunk) =
                  make_uint4(wStp[4 * k], wStp[4 * k + 1], wStp[4 * k + 2], wStp[4 * k + 3]);
            if (zf)
              *reinterpret_cast<uint4*>(wrow + 2 * kChunkBytes + chunk) =
                  make_uint4(wZp[4 * k], wZp[4 * k + 1], wZp[4 * k + 2], wZp[4 * k + 3]);
          }
          if (ragged) {   // padding columns of the last tile: weight zero (the stored strip's copy feeds discarded rows only)
            const int k0 = max(32 * n1, jlim - 64 * h), k1 = 32 * n1 + 32;
            zero_padding_cols(wrow_s, m, k0, k1);
            if (!kW) zero_padding_cols(wrow + kChunkBytes, m, k0, k1);
            if (zf) zero_padding_cols(wrow + 2 * kChunkBytes, m, k0, k1);
          }
          fence_proxy_async_smem();
          mbar_arrive_cluster(bar((kW && h == 1) ? kWFull1 : kWFull), 0);
          if (kW) {
            // the same 32 weights of row lrow, columns t * 128 + jl0 .. + 31, to the stored tile (64 contiguous bytes)
            uint4* wg = reinterpret_cast<uint4*>(p.wout + (size_t)lrow * p.Bp + (size_t)t * kTileN + jl0);
#pragma unroll
            for (int k = 0; k < 4; ++k) wg[k] = make_uint4(wSp[4 * k], wSp[4 * k + 1], wSp[4 * k + 2], wSp[4 * k + 3]);
          }
          mbar_arrive_local(bar(kCstEmpty0 + (tt & 1)));   // this thread is done with the tile's constants
        }
        ++tt;
      }

      // ---- end of job: write this job's partial results
      if (PHASE == kStats || PHASE == kStatsZ || PHASE == kRowLoss) {
        // four threads hold pieces of row m (lane half n1 x column half h): combine through shared memory
        float* scratch = consts;  // [3 partners][7][64] floats; the column constants are dead once the tile loop is over
        OnlineLse2 lS, lSt, lZ;  // log2-domain (max, sum) pairs
        lS.m = mS * cS2; lS.s = sS; lSt.m = mSt * cS2; lSt.s = sSt; lZ.m = mZ * cZ2; lZ.s = sZ;
        float aZ = aPS;          // travels with lZ: rescaled by the same factors
        const float acc_g = (ag4[0] + ag4[1]) + (ag4[2] + ag4[3]), acc_q = (aq4[0] + aq4[1]) + (aq4[2] + aq4[3]);
        const int part = 2 * h + n1;  // 0 = the row's writer
        named_bar_sync(2, kEpiThreads);
        if (part != 0) {
          float* sc = scratch + (part - 1) * 7 * 64;
          if (PHASE == kStats || PHASE == kStatsZ) {
            sc[0 * 64 + m] = lS.m; sc[1 * 64 + m] = lS.s;
            sc[2 * 64 + m] = lSt.m; sc[3 * 64 + m] = lSt.s;
            sc[4 * 64 + m] = lZ.m; sc[5 * 64 + m] = lZ.s;
            sc[6 * 64 + m] = aZ;
          } else {
            sc[0 * 64 + m] = acc_g; sc[1 * 64 + m] = acc_q;
          }
        }
        named_bar_sync(2, kEpiThreads);
        if (part == 0) {
          if (PHASE == kStats || PHASE == kStatsZ) {
            for (int k = 0; k < 3; ++k) {
              const float* sc = scratch + k * 7 * 64;
              lS.merge(sc[0 * 64 + m], sc[1 * 64 + m]);
              lSt.merge(sc[2 * 64 + m], sc[3 * 64 + m]);
              const float m2 = sc[4 * 64 + m], mn = fmaxf(lZ.m, m2);
              if (mn != -INFINITY) aZ = aZ * ex2f(lZ.m - mn) + sc[6 * 64 + m] * ex2f(m2 - mn);
              lZ.merge(m2, sc[5 * 64 + m]);
            }
            float2* out = reinterpret_cast<float2*>(p.part);
            const size_t o = (size_t)sp * 4 * p.bpad + lrow;
            const bool probe = PHASE == kStats && p.flags_out != nullptr;  // the Z half then comes from the kStatsZ sweep
            if (PHASE == kStats) {
              out[o] = make_float2(lS.m, lS.s);
              out[o + p.bpad] = make_float2(lSt.m, lSt.s);
            }
            if (!probe) {
              out[o + 2 * (size_t)p.bpad] = make_float2(lZ.m, lZ.s);
              out[o + 3 * (size_t)p.bpad] = make_float2(aZ * (inv_s2 * p.inv_tau), 0.f);  // natural S units, relative to lZ.m
            }
          } else {
            float pc = acc_g, q = acc_q;
            for (int k = 0; k < 3; ++k) { pc += scratch[k * 7 * 64 + m]; q += scratch[k * 7 * 64 + 64 + m]; }
            const size_t o = (size_t)sp * 2 * p.bpad + lrow;
            p.part[o] = pc * kLn2;  // this split's share of sum_j P_ij c_j
            p.part[o + p.bpad] = q;
          }
        }
      } else {
        // accumulators: lanes 0-63 hold d in [0, D/2), lanes 64-127 hold [D/2, D); this thread reads the
        // column half h of its lane's D/2 columns
        mbar_wait_t(bar(kAccFull), jp & 1, prof_base + 3, prof_rec);
        ++jp;
        tc_fence_after();
        // kBwdW: the dI accumulator is written by flagged tiles only; a job without any holds no dI at all
        const bool di_any = !kW || !frow || job_has_tiles(frow, t0, t1);
        const int half_d = D / 2, quart_d = D / 4;
        float* out_t = p.part + ((size_t)sp * 2 * p.bpad + lrow) * D + n1 * half_d + h * quart_d;
        float* out_i = out_t + (size_t)p.bpad * D;
        for (int c0 = 0; c0 < quart_d; c0 += 32) {
          float v[32];
          tmem_ld32(tmem_base + lane_field + kAccCol + h * quart_d + c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int e = 0; e < 32; e += 4) *reinterpret_cast<float4*>(out_t + c0 + e) = make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]);
          tmem_ld32(tmem_base + lane_field + kAccCol + half_d + h * quart_d + c0, v);
          tmem_ld_wait();
          if (!di_any) {
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = 0.f;
          }
#pragma unroll
          for (int e = 0; e < 32; e += 4) *reinterpret_cast<float4*>(out_i + c0 + e) = make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]);
        }
        tc_fence_before();
        mbar_arrive_cluster(bar(kAccEmpty), 0);
      }
    }
    MC_PROF_TOTAL(prof_base + 4, prof_t0, prof_rec);
  }

  // teardown: nobody leaves while the peer may still touch this CTA's shared memory or TMEM
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc_pair(tmem_base, 512);
}
#ifdef MC_WAIT_PROFILE
}  // namespace tc
}  // namespace mc
extern "C" int mc_debug_wait_profile(unsigned long long* out64, int reset) {
  if (cudaDeviceSynchronize() != cudaSuccess) return 1;
  if (out64 && cudaMemcpyFromSymbol(out64, mc::tc::g_wait_prof, 64 * sizeof(unsigned long long)) != cudaSuccess) return 1;
  if (reset) {
    unsigned long long z[64] = {};
    if (cudaMemcpyToSymbol(mc::tc::g_wait_prof, z, sizeof(z)) != cudaSuccess) return 1;
  }
  return 0;
}
namespace mc {
namespace tc {
#endif

// ------------------------------------------------------------------------------------------
// finalize kernels: merge the per-split partials
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) stats_finalize_kernel(const float2* __restrict__ part, int nsplit, int bpad,
                                                             int b, float* __restrict__ r, float* __restrict__ c,
                                                             float* __restrict__ rz, float* __restrict__ ps) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= b) return;
  float* outs[3] = {r, c, rz};
  for (int k = 0; k < 3; ++k) {
    if (outs[k] == nullptr) continue;   // c comes from the column partials (colpart_merge_kernel)
    OnlineLse2 l;
    l.init();
    float a = 0.f;  // k == 2: sum_j e^{Z_ij - max} S_ij, merged with the same rescaling as the Z sum
    for (int s = 0; s < nsplit; ++s) {
      const float2 v = part[((size_t)s * 4 + k) * bpad + i];
      if (k == 2) {
        const float mn = fmaxf(l.m, v.x);
        if (mn != -INFINITY) a = a * ex2f(l.m - mn) + part[((size_t)s * 4 + 3) * bpad + i].x * ex2f(v.x - mn);
      }
      l.merge(v.x, v.y);
    }
    outs[k][i] = (l.m + log2f(l.s)) * kLn2;
    if (k == 2) ps[i] = a / l.s;
  }
}

// Column LSE from the per-32-row partials of the statistics sweep: c_j = ln2 * log2 sum_g 2^{part[g][j]}.
// A block owns 64 columns; its four thread groups take every fourth row group (eight loads in flight per thread) and
// meet in shared memory in a fixed order.
__global__ void __launch_bounds__(256) colpart_merge_kernel(const float* __restrict__ part, int groups, int Bp, int B,
                                                            float* __restrict__ c) {
  __shared__ float sm_m[4][64], sm_s[4][64];
  const int tx = threadIdx.x & 63, g0 = threadIdx.x >> 6;
  const int j = blockIdx.x * 64 + tx;
  OnlineLse2 l;
  l.init();
  if (j < B) {
    int g = g0;
    for (; g + 28 < groups; g += 32) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = part[(size_t)(g + 4 * u) * Bp + j];
      float mx = v[0];
#pragma unroll
      for (int u = 1; u < 8; ++u) mx = fmaxf(mx, v[u]);
      const float mn = fmaxf(l.m, mx);
      if (mn != -INFINITY) {
        float acc = 0.f;
#pragma unroll
        for (int u = 0; u < 8; ++u) acc += ex2f(v[u] - mn);
        l.s = l.s * ex2f(l.m - mn) + acc;
        l.m = mn;
      }
    }
    for (; g < groups; g += 4) l.merge(part[(size_t)g * Bp + j], 1.f);
  }
  sm_m[g0][tx] = l.m;
  sm_s[g0][tx] = l.s;
  __syncthreads();
  if (g0 == 0 && j < B) {
#pragma unroll
    for (int u = 1; u < 4; ++u) l.merge(sm_m[u][tx], sm_s[u][tx]);
    c[j] = (l.m + log2f(l.s)) * kLn2;
  }
}

// c_j = log sum_q exp(part_q[j]): the ranks' column-LSE vectors (each over that rank's rows) -> the column LSE of S
__global__ void __launch_bounds__(256) ranks_lse_merge_kernel(const float* __restrict__ parts, int n, int64_t stride, int B,
                                                              float* __restrict__ c) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= B) return;
  float m = -INFINITY;
  for (int q = 0; q < n; ++q) m = fmaxf(m, parts[(size_t)q * stride + j]);
  float s = 0.f;
  if (m != -INFINITY)
    for (int q = 0; q < n; ++q) s += __expf(parts[(size_t)q * stride + j] - m);
  c[j] = m == -INFINITY ? -INFINITY : m + __logf(s);
}
int ranks_lse_merge(const float* parts, int n, int64_t stride, int B, float* c, cudaStream_t st) {
  ranks_lse_merge_kernel<<<(B + 255) / 256, 256, 0, st>>>(parts, n, stride, B, c);
  MC_LAUNCH_CHECK();
  return MC_OK;
}

// g_i = (r_i + sum_j P_ij c_j - 2 sum_j P_ij S_ij) / 2B ; q_i = colsum(P)_i
__global__ void __launch_bounds__(256) rowloss_finalize_kernel(const float* __restrict__ part, int nsplit,
                                                               int bpad, int b, float inv_2B,
                                                               const float* __restrict__ r_loc,
                                                               const float* __restrict__ ps_loc,
                                                               float* __restrict__ g, float* __restrict__ q) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= b) return;
  float pc = 0.f, aq = 0.f;
  for (int s = 0; s < nsplit; ++s) {
    pc += part[((size_t)s * 2) * bpad + i];
    aq += part[((size_t)s * 2 + 1) * bpad + i];
  }
  g[i] = (r_loc[i] + pc - 2.f * ps_loc[i]) * inv_2B;
  q[i] = aq;
}

__global__ void __launch_bounds__(1024) sum_kernel(const float* __restrict__ v, int n, float* __restrict__ out) {
  __shared__ double sm[32];
  double acc = 0.0;
  int i0 = 0;
  if ((reinterpret_cast<uintptr_t>(v) & 15) == 0) {  // 16-byte loads: a quarter of the dependent round trips
    const int n4 = n >> 2;
    for (int i = threadIdx.x; i < n4; i += blockDim.x) {
      const float4 x = reinterpret_cast<const float4*>(v)[i];
      acc += ((double)x.x + (double)x.y) + ((double)x.z + (double)x.w);
    }
    i0 = n4 << 2;
  }
  for (int i = i0 + threadIdx.x; i < n; i += blockDim.x) acc += (double)v[i];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    double t = (threadIdx.x < (blockDim.x >> 5)) ? sm[threadIdx.x] : 0.0;
    t = warp_sum(t);
    if (threadIdx.x == 0) *out = (float)t;
  }
}

// Power-of-two scale of the fp16 gradient-weight tiles, from bounds that hold for every element:
//   |2B dS_ij| <= 2 + q_j               (softmax terms in [0,1], P in [0,1], q = colsum(P))
//   0 <= 2B G_ij = r_i + c_j - 2 S_ij <= max r + max c + 2 max||T|| max||I|| / tau   (Cauchy-Schwarz)
//   |2B (dZ_ij + dZ_ji)| <= 2 max(2B G)  (g_i is a P-weighted mean of G_i.)
// The largest possible weight is mapped just below 2^15 so that nothing overflows fp16 and the
// small weights of the soft-target regime stay in the normal range.
__global__ void __launch_bounds__(1024) wscale_kernel(const float* __restrict__ r, const float* __restrict__ c,
                                                      const float* __restrict__ rz, const float* __restrict__ q, int B,
                                                      const float* __restrict__ scale,
                                                      const float* __restrict__ norm_i,
                                                      const float* __restrict__ norm_t, float inv_tau, float tau,
                                                      float* __restrict__ out) {
  // maxima: r, c, q, (unused), ||I||, ||T||, rz, -r, -c, -rz  (the negated ones give the minima)
  __shared__ float sm[10][32];
  float v[10] = {-INFINITY, -INFINITY, 0.f, 0.f, 0.f, 0.f, -INFINITY, -INFINITY, -INFINITY, -INFINITY};
  auto take = [&](float ri, float ci, float zi, float qi, float ni, float nt) {
    v[0] = fmaxf(v[0], ri); v[1] = fmaxf(v[1], ci); v[2] = fmaxf(v[2], qi);
    v[4] = fmaxf(v[4], ni); v[5] = fmaxf(v[5], nt);
    v[6] = fmaxf(v[6], zi); v[7] = fmaxf(v[7], -ri); v[8] = fmaxf(v[8], -ci); v[9] = fmaxf(v[9], -zi);
  };
  int i0 = 0;
  const uintptr_t align = reinterpret_cast<uintptr_t>(r) | reinterpret_cast<uintptr_t>(c) | reinterpret_cast<uintptr_t>(rz) |
                          reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(norm_i) |
                          reinterpret_cast<uintptr_t>(norm_t);
  if ((align & 15) == 0) {  // one block walks six length-B vectors: 16-byte loads, six independent streams in flight
    const int B4 = B >> 2;
    for (int i = threadIdx.x; i < B4; i += blockDim.x) {
      const float4 a = reinterpret_cast<const float4*>(r)[i], b4 = reinterpret_cast<const float4*>(c)[i];
      const float4 z = reinterpret_cast<const float4*>(rz)[i], qq = reinterpret_cast<const float4*>(q)[i];
      const float4 ni = reinterpret_cast<const float4*>(norm_i)[i], nt = reinterpret_cast<const float4*>(norm_t)[i];
      take(a.x, b4.x, z.x, qq.x, ni.x, nt.x);
      take(a.y, b4.y, z.y, qq.y, ni.y, nt.y);
      take(a.z, b4.z, z.z, qq.z, ni.z, nt.z);
      take(a.w, b4.w, z.w, qq.w, ni.w, nt.w);
    }
    i0 = B4 << 2;
  }
  for (int i = i0 + threadIdx.x; i < B; i += blockDim.x) take(r[i], c[i], rz[i], q[i], norm_i[i], norm_t[i]);
  for (int k = 0; k < 10; ++k) {
    v[k] = warp_max(v[k]);
    if ((threadIdx.x & 31) == 0) sm[k][threadIdx.x >> 5] = v[k];
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    for (int k = 0; k < 10; ++k) v[k] = warp_max(sm[k][threadIdx.x]);
    if (threadIdx.x == 0) {
      v[3] = scale[1];  // 1 / s: weights multiply the scaled plane
      const float gmax = fmaxf(v[0] + v[1] + 2.f * v[4] * v[5] * inv_tau, 1.f);
      const float b1 = (2.f + v[2]) * v[3] * inv_tau;
      const float b3 = 2.f * gmax * v[3] * 0.5f * tau;
      const float bound = fmaxf(fmaxf(b1, b3), 1e-30f);
      int e;
      frexpf(bound, &e);  // bound < 2^e
      int k = 15 - e;
      k = k < -60 ? -60 : (k > 60 ? 60 : k);
      out[0] = ldexpf(1.f, k);
      // Fast exponentials: with every row/column statistic within 60 binades of each other,
      // e^{S - c_j} = e^{S - r_i} * 2^{r2_i - M} * 2^{M - c2_j} (and likewise for P_ji) can neither
      // overflow nor lose a term that matters (an underflowed factor implies a term below 2^-66).
      const float kL2e = 1.4426950408889634f;
      const float hi_rc = fmaxf(v[0], v[1]), lo_rc = -fmaxf(v[7], v[8]);
      const float hi_z = v[6], lo_z = -v[9];
      const bool fast = (hi_rc - lo_rc) * kL2e <= 60.f && (hi_z - lo_z) * kL2e <= 60.f;
      out[1] = fast ? 1.f : 0.f;
      out[2] = 0.5f * (hi_rc + lo_rc) * kL2e;  // M_rc, log2 units
      out[3] = 0.5f * (hi_z + lo_z) * kL2e;    // M_z
    }
  }
}

__global__ void __launch_bounds__(256) bwd_finalize_kernel(const float* __restrict__ part, int nsplit, int bpad,
                                                           int b, int D, float inv_2B,
                                                           const float* __restrict__ grad_loss,
                                                           const float* __restrict__ wscale,
                                                           float* __restrict__ dT, float* __restrict__ dI,
                                                           const int* __restrict__ gate = nullptr, int gate_want = 0) {
  if (gate != nullptr && *gate != gate_want) return;
  const float scale = (grad_loss ? *grad_loss : 1.f) * inv_2B / *wscale;
  const size_t n4 = (size_t)b * D / 4;
  const size_t plane = (size_t)bpad * D;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    float4 at = make_float4(0.f, 0.f, 0.f, 0.f), ai = at;
    for (int s = 0; s < nsplit; ++s) {
      const float4 a = reinterpret_cast<const float4*>(part + (size_t)s * 2 * plane)[i];
      const float4 c = reinterpret_cast<const float4*>(part + ((size_t)s * 2 + 1) * plane)[i];
      at.x += a.x; at.y += a.y; at.z += a.z; at.w += a.w;
      ai.x += c.x; ai.y += c.y; ai.z += c.z; ai.w += c.w;
    }
    reinterpret_cast<float4*>(dT)[i] = make_float4(at.x * scale, at.y * scale, at.z * scale, at.w * scale);
    reinterpret_cast<float4*>(dI)[i] = make_float4(ai.x * scale, ai.y * scale, ai.z * scale, ai.w * scale);
  }
}

// ------------------------------------------------------------------------------------------
// Column half of the stored-weights gradient: dI_j (+)= sum_i W_ij T_i over the rows i of a stored weight strip.
//   W  (rows x Bp fp16, written by pair_kernel<kBwdW>)  is the A operand READ TRANSPOSED: a TMA box of {64 j, 64 i}
//      lands in shared memory as 64 rows (i = K) of 128 bytes (64 j = M), which is exactly the canonical MN-major
//      SWIZZLE_128B operand layout (8-row groups 1024 B apart, 64-wide M blocks `LBO` apart) - no transpose anywhere;
//   T^T (the transposed hi plane, rows D..2D)            is the K-major B operand, as in the gradient GEMMs of kBwd.
// A CTA pair owns 256 output rows j (cta_group::2, M = 256: lane = row, N = D columns), streams its K range through a
// ring of 64-row stages and keeps two accumulator buffers in TMEM so that the read-out of one job overlaps the MMAs of
// the next.  Jobs = (256-row block of j) x (K split); every job writes its own partial (deterministic fold afterwards).
// ------------------------------------------------------------------------------------------
constexpr int kCgThreads = 256;   // warp 0 TMA, warp 1 MMA + TMEM, warps 4-7 read-out
constexpr int kCgStageA = 2 * 8192;                  // two 64-wide M blocks x 64 K rows x 128 B
constexpr int kCgStages = 6;
constexpr int kCgMaxSplit = 8;
struct ColGradParams {
  int Bp, D;
  int w_rows;              // rows of the stored strip (multiple of 64)
  int row_offset;          // global row of the strip's first row (column coordinate of T^T)
  int j_first;             // first output row (multiple of 256 ... any multiple of 128)
  int n_jblocks;           // 256-row blocks from j_first on
  int j_end;               // output rows >= j_end are not written
  int ksplit, steps_per_split, steps;   // K steps of 64 rows
  float* part;             // [ksplit][n_jblocks * 256][D]
  const int* gate;         // runs only while *gate == 1 (null: always)
};
// MN-major SWIZZLE_128B operand: [16,30) leading byte offset (between 64-element M blocks), [32,46) stride byte offset
// (between 8-row K groups)
__device__ __forceinline__ uint64_t smem_desc_mn_sw128(uint32_t saddr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(lbo_bytes >> 4) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
__global__ void __launch_bounds__(kCgThreads, 1)
colgrad_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_t,
               const ColGradParams p) {
  if (p.gate != nullptr && *p.gate != 1) return;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* const sbase = smem_raw + (base - raw);
  const int D = p.D;
  const uint32_t b_bytes = (uint32_t)(D / 2) * 128u;           // this CTA's half of the B tile: D/2 rows x 64 K
  const uint32_t stage_bytes = kCgStageA + b_bytes;            // 32 KB at D = 256
  const uint32_t bar0 = base + kCgStages * stage_bytes;
  auto bar = [&](int i) -> uint32_t { return bar0 + 8u * i; };
  enum { kFull = 0, kEmpty = kCgStages, kAccFull = 2 * kCgStages, kAccEmpty = 2 * kCgStages + 2, kBars = 2 * kCgStages + 4 };
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(sbase + kCgStages * stage_bytes + 8 * kBars);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair_id = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int njobs = p.n_jblocks * p.ksplit;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kCgStages; ++s) { mbar_init(bar(kFull + s), 1); mbar_init(bar(kEmpty + s), 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(bar(kAccFull + i), 1); mbar_init(bar(kAccEmpty + i), 2 * 128); }
    fence_mbar_init();
    prefetch_tmap(&map_w);
    prefetch_tmap(&map_t);
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
      uint32_t it = 0;
      for (int job = pair_id; job < njobs; job += npairs) {
        const int jb = job / p.ksplit, ks = job % p.ksplit;
        const int j0 = p.j_first + jb * 256 + (int)rank * 128;
        const int s0 = ks * p.steps_per_split, s1 = min(s0 + p.steps_per_split, p.steps);
        for (int st = s0; st < s1; ++st, ++it) {
          const uint32_t slot = it % kCgStages, par = (it / kCgStages) & 1;
          mbar_wait(bar(kEmpty + slot), par ^ 1);
          const uint32_t fb = bar(kFull + slot), sa = base + slot * stage_bytes;
          if (leader) mbar_arrive_expect_tx(fb, 2u * stage_bytes);
          const int i0 = st * 64;
          tma_load_2d_pair(sa, &map_w, fb, j0, i0);                   // W[i0 .. +64][j0 .. +64]
          tma_load_2d_pair(sa + 8192, &map_w, fb, j0 + 64, i0);       // W[i0 .. +64][j0 + 64 .. +128]
          tma_load_2d_pair(sa + kCgStageA, &map_t, fb, p.row_offset + i0, D + (int)rank * (D / 2));   // T^T[d][i]
        }
      }
    }
  } else if (warp == 1) {
    if (leader && elect_one()) {
      const uint32_t idesc = idesc_f16(256, D) | (1u << 15);   // A is MN-major
      uint32_t it = 0, jj = 0;
      for (int job = pair_id; job < njobs; job += npairs) {
        const int ks = job % p.ksplit;
        const int s0 = ks * p.steps_per_split, s1 = min(s0 + p.steps_per_split, p.steps);
        if (s0 >= s1) continue;            // a split beyond the strip: no accumulator use (jj counts the others)
        const uint32_t buf = jj & 1, use = jj >> 1;
        ++jj;
        mbar_wait(bar(kAccEmpty + buf), (use & 1) ^ 1);
        tc_fence_after();
        const uint32_t tacc = tmem_base + buf * (uint32_t)D;
        for (int st = s0; st < s1; ++st, ++it) {
          const uint32_t slot = it % kCgStages, par = (it / kCgStages) & 1;
          mbar_wait(bar(kFull + slot), par);
          tc_fence_after();
          const uint32_t sa = base + slot * stage_bytes;
          const uint64_t bd = smem_desc_sw128(sa + kCgStageA);
#pragma unroll
          for (int k4 = 0; k4 < 4; ++k4)     // 16 K rows = 2048 bytes of the MN-major tile per MMA
            mma_f16_pair(tacc, smem_desc_mn_sw128(sa + k4 * 2048, 8192), desc_advance_k(bd, k4), idesc,
                         (st > s0 || k4 > 0) ? 1u : 0u);
          mma_commit_pair(bar(kEmpty + slot), 3);
        }
        mma_commit_pair(bar(kAccFull + buf), 3);
      }
    }
  } else if (warp >= 4) {
    const int q = warp - 4;                      // TMEM lane quarter
    uint32_t jj = 0;
    for (int job = pair_id; job < njobs; job += npairs) {
      const int jb = job / p.ksplit, ks = job % p.ksplit;
      const int lrow = jb * 256 + (int)rank * 128 + q * 32 + lane;    // row within the partial
      const bool ok = p.j_first + lrow < p.j_end;
      const int s0 = ks * p.steps_per_split;
      const bool empty = s0 >= p.steps;          // a split beyond the strip: nothing was accumulated
      const uint32_t buf = jj & 1, use = jj >> 1;
      if (!empty) ++jj;
      float* out = p.part + ((size_t)ks * p.n_jblocks * 256 + lrow) * D;
      if (!empty) {
        mbar_wait(bar(kAccFull + buf), use & 1);
        tc_fence_after();
      }
      for (int c0 = 0; c0 < D; c0 += 32) {
        float v[32];
        if (!empty) {
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + buf * (uint32_t)D + c0, v);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int e = 0; e < 32; ++e) v[e] = 0.f;
        }
        if (ok) {
#pragma unroll
          for (int e = 0; e < 32; e += 4)
            *reinterpret_cast<float4*>(out + c0 + e) = make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]);
        }
      }
      if (!empty) {
        tc_fence_before();
        mbar_arrive_cluster(bar(kAccEmpty + buf), 0);
      }
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc_pair(tmem_base, 512);
}

// fold of the row half: dT (final) and the un-scaled soft-target part of dI
__global__ void __launch_bounds__(256) bwd_rows_finalize_kernel(const float* __restrict__ part, int nsplit, int bpad,
                                                                int b, int D, float inv_2B,
                                                                const float* __restrict__ grad_loss,
                                                                const float* __restrict__ wscale,
                                                                float* __restrict__ dT, float* __restrict__ dIz) {
  const float scale = (grad_loss ? *grad_loss : 1.f) * inv_2B / *wscale;
  const size_t n4 = (size_t)b * D / 4;
  const size_t plane = (size_t)bpad * D;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    float4 at = make_float4(0.f, 0.f, 0.f, 0.f), ai = at;
    for (int s = 0; s < nsplit; ++s) {
      const float4 a = reinterpret_cast<const float4*>(part + (size_t)s * 2 * plane)[i];
      const float4 c = reinterpret_cast<const float4*>(part + ((size_t)s * 2 + 1) * plane)[i];
      at.x += a.x; at.y += a.y; at.z += a.z; at.w += a.w;
      ai.x += c.x; ai.y += c.y; ai.z += c.z; ai.w += c.w;
    }
    reinterpret_cast<float4*>(dT)[i] = make_float4(at.x * scale, at.y * scale, at.z * scale, at.w * scale);
    reinterpret_cast<float4*>(dIz)[i] = ai;
  }
}
// fold of the split row half: dT = scale (sum_s rowgrad partials + kBwdP's dT partial), dIz = kBwdP's dI partial
__global__ void __launch_bounds__(256) bwd_rows_split_finalize_kernel(const float* __restrict__ part_r, int nsplit_r,
                                                                      size_t plane_r, const float* __restrict__ part_p,
                                                                      size_t plane_p, int b, int D, float inv_2B,
                                                                      const float* __restrict__ grad_loss,
                                                                      const float* __restrict__ wscale,
                                                                      float* __restrict__ dT, float* __restrict__ dIz,
                                                                      const int* __restrict__ gate) {
  if (gate != nullptr && *gate != 1) return;
  const float scale = (grad_loss ? *grad_loss : 1.f) * inv_2B / *wscale;
  const size_t n4 = (size_t)b * D / 4;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    float4 at = reinterpret_cast<const float4*>(part_p)[i];
    for (int s = 0; s < nsplit_r; ++s) {
      const float4 a = reinterpret_cast<const float4*>(part_r + (size_t)s * plane_r)[i];
      at.x += a.x; at.y += a.y; at.z += a.z; at.w += a.w;
    }
    reinterpret_cast<float4*>(dT)[i] = make_float4(at.x * scale, at.y * scale, at.z * scale, at.w * scale);
    reinterpret_cast<float4*>(dIz)[i] = reinterpret_cast<const float4*>(part_p + plane_p)[i];
  }
}
// fold of the column half: dI_j = scale (dIz_j + sum_k part_k[j])
__global__ void __launch_bounds__(256) bwd_cols_finalize_kernel(const float* __restrict__ part, int ksplit, size_t plane,
                                                                int rows, int D, float inv_2B,
                                                                const float* __restrict__ grad_loss,
                                                                const float* __restrict__ wscale,
                                                                const float* __restrict__ dIz, float* __restrict__ dI,
                                                                const int* __restrict__ gate) {
  if (gate != nullptr && *gate != 1) return;
  const float scale = (grad_loss ? *grad_loss : 1.f) * inv_2B / *wscale;
  const size_t n4 = (size_t)rows * D / 4;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    float4 a = dIz ? reinterpret_cast<const float4*>(dIz)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s = 0; s < ksplit; ++s) {
      const float4 c = reinterpret_cast<const float4*>(part + (size_t)s * plane)[i];
      a.x += c.x; a.y += c.y; a.z += c.z; a.w += c.w;
    }
    reinterpret_cast<float4*>(dI)[i] = make_float4(a.x * scale, a.y * scale, a.z * scale, a.w * scale);
  }
}

// ------------------------------------------------------------------------------------------
// Dense row half of the stored-weights gradient, the softmax part of dS only:
//     2B dS_ij (softmax part) = softmax_row(S)_ij + q_j softmax_col(S)_ij            (the -2 P_ij term and everything
// that depends on Z live on the flagged tiles and are added by pair_kernel<kBwdP>, which visits those tiles only).
// Every tile needs S = T_i I_j^T alone, so this kernel is built around LARGE MMA instructions: tools/mma_issue_bench.cu shows
// that one thread sustains the full tensor rate for every cta_group::2 shape only while it does nothing else - every
// wait, fence or descriptor computation between two 32-cycle (M = 128, N = 128) MMAs is exposed, which is what holds
// pair_kernel at ~50% of the tensor pipe (profiles/r02r_wait_profile_pair_kernel.json, ablation in DESIGN 4.1).
//   * a CTA pair owns 256 rows i (128 per CTA, cta_group::2 with M = 256: TMEM lane = row); S tiles are 256 x 128
//     (64-cycle MMAs), the gradient GEMM dT_i += W I_j is M = 256, N = D (128-cycle MMAs);
//   * T_i hi stays resident (64 KB); a ring slot carries one 64-wide K chunk of {T_i lo, I_j hi, I_j lo} (32 KB);
//   * TMEM: two S tile buffers (2 x 128 columns) + the dT accumulator (D columns);
//   * the fp16 weight tile goes to shared memory (A operand of the gradient GEMM, one buffer per 64-column half, as
//     does the I_j^T tile) and, as full 128-byte rows, to the stored strip W that colgrad_kernel turns into dI.
// Roles: warp 0 ring producer, warp 1 MMA issuer, warp 2 I_j^T producer, warp 3 per-column constants, warps 4-11
// epilogue (lane quarter x column half).
// ------------------------------------------------------------------------------------------
constexpr int kRgThreads = 384;
constexpr int kRgRowsCta = 128;
constexpr int kRgSlotBytes = 32768;
constexpr int kRgSlots = 3;
constexpr int kRgOffA = 0;                                   // T_i hi: D/64 chunks of 128 rows x 128 B
constexpr int kRgOffRing = 65536;
constexpr int kRgOffW = kRgOffRing + kRgSlots * kRgSlotBytes;    // 2 x (128 rows x 64 j) fp16
constexpr int kRgOffXT = kRgOffW + 2 * 16384;                    // 2 x (D/2 rows x 64 j) fp16
constexpr int kRgOffConst = kRgOffXT + 2 * 16384;                // 2 buffers x 2 fields x 128 floats
constexpr int kRgOffBar = kRgOffConst + 2048;
constexpr int kRgSmemBytes = kRgOffBar + 256 + 512;   // the dynamic segment is declared 1024-aligned; 512 bytes of slack are checked
enum RgBar {
  kRgFull0 = 0, kRgEmpty0 = 3, kRgAFull = 6, kRgJobDone = 7, kRgTmemFull0 = 8, kRgTmemEmpty0 = 10, kRgWFull0 = 12,
  kRgXTFull0 = 14, kRgGradDone0 = 16, kRgAccFull = 18, kRgAccEmpty = 19, kRgCstFull0 = 20, kRgCstEmpty0 = 22, kRgNumBars = 24
};
struct RowGradParams {
  int b, B, Bp, D, row_offset;
  int n_row_blocks, n_tiles, nsplit, tiles_per_split, bpad;     // row blocks of 256
  float inv_tau;
  const float* scale;
  const float *r, *c, *q;
  const float* wscale;
  float* part;            // [nsplit][bpad][D]
  __half* wout;           // (bpad x Bp)
  const int* gate;        // runs only while *gate == 1 (null: always)
};
template <int PASSES>
__global__ void __launch_bounds__(kRgThreads, 1)
rowgrad_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
               const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
               const __grid_constant__ CUtensorMap map_t, const RowGradParams p) {
  if (p.gate != nullptr && *p.gate != 1) return;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  if (base - raw > 512u) __trap();   // the map below would run past the allocation
  uint8_t* const sbase = smem_raw + (base - raw);
  const uint32_t bar0 = base + kRgOffBar;
  auto bar = [&](int i) -> uint32_t { return bar0 + 8u * i; };
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(sbase + kRgOffBar + 8 * kRgNumBars);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair_id = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int D = p.D, nkc = D >> 6;
  const int njobs = p.n_row_blocks * p.nsplit;
  const uint32_t xt_bytes = (uint32_t)(D / 2) * 128u;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kRgSlots; ++s) { mbar_init(bar(kRgFull0 + s), 1); mbar_init(bar(kRgEmpty0 + s), 1); }
    mbar_init(bar(kRgAFull), 1);
    mbar_init(bar(kRgJobDone), 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar(kRgTmemFull0 + i), 1);
      mbar_init(bar(kRgTmemEmpty0 + i), 2 * 256);
      mbar_init(bar(kRgWFull0 + i), 2 * 128);
      mbar_init(bar(kRgXTFull0 + i), 1);
      mbar_init(bar(kRgGradDone0 + i), 1);
      mbar_init(bar(kRgCstFull0 + i), 32);
      mbar_init(bar(kRgCstEmpty0 + i), 256);
    }
    mbar_init(bar(kRgAccFull), 1);
    mbar_init(bar(kRgAccEmpty), 2 * 256);
    fence_mbar_init();
    prefetch_tmap(&map_a_hi); prefetch_tmap(&map_a_lo); prefetch_tmap(&map_b_hi); prefetch_tmap(&map_b_lo);
    prefetch_tmap(&map_t);
  }
  if (warp == 1) {
    tmem_alloc_pair(smem_u32(tmem_slot), 512);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  constexpr uint32_t kAcc = 256;   // dT accumulator columns [256, 256 + D)

  if (warp == 0) {
    // ===================================================== ring producer
    if (elect_one()) {
      uint32_t it = 0, jj = 0;
      for (int job = pair_id; job < njobs; job += npairs, ++jj) {
        const int rb = job / p.nsplit, sp = job % p.nsplit;
        const int row_a = p.row_offset + rb * 256 + (int)rank * kRgRowsCta;
        const int t0 = sp * p.tiles_per_split, t1 = min(t0 + p.tiles_per_split, p.n_tiles);
        mbar_wait(bar(kRgJobDone), (jj & 1) ^ 1);
        if (leader) mbar_arrive_expect_tx(bar(kRgAFull), 2u * (uint32_t)nkc * 16384u);
        for (int c = 0; c < nkc; ++c) tma_load_2d_pair(base + kRgOffA + c * 16384, &map_a_hi, bar(kRgAFull), D + c * 64, row_a);
        for (int t = t0; t < t1; ++t) {
          const int j0 = t * kTileN + 64 * (int)rank;
          for (int c = 0; c < nkc; ++c, ++it) {
            const uint32_t slot = it % kRgSlots, par = (it / kRgSlots) & 1;
            mbar_wait(bar(kRgEmpty0 + slot), par ^ 1);
            const uint32_t fb = bar(kRgFull0 + slot), sb = base + kRgOffRing + slot * kRgSlotBytes;
            if (leader) mbar_arrive_expect_tx(fb, PASSES == 3 ? 2u * kRgSlotBytes : 2u * 8192u);
            if (PASSES == 3) tma_load_2d_pair(sb, &map_a_lo, fb, D + c * 64, row_a);            // T_i lo   (128 rows)
            tma_load_2d_pair(sb + 16384, &map_b_hi, fb, c * 64, j0);           // I_j hi   (64 rows)
            if (PASSES == 3) tma_load_2d_pair(sb + 24576, &map_b_lo, fb, c * 64, j0);           // I_j lo
          }
        }
      }
    }
  } else if (warp == 2) {
    // ===================================================== I_j^T half tiles (B operand of dT += W I_j)
    if (elect_one()) {
      uint32_t tt = 0;
      for (int job = pair_id; job < njobs; job += npairs) {
        const int sp = job % p.nsplit;
        const int t0 = sp * p.tiles_per_split, t1 = min(t0 + p.tiles_per_split, p.n_tiles);
        for (int t = t0; t < t1; ++t, ++tt) {
          for (int h = 0; h < 2; ++h) {
            mbar_wait(bar(kRgGradDone0 + h), (tt & 1) ^ 1);     // the previous tile's half-h MMAs have drained the buffer
            const uint32_t fb = bar(kRgXTFull0 + h);
            if (leader) mbar_arrive_expect_tx(fb, 2u * xt_bytes);
            tma_load_2d_pair(base + kRgOffXT + h * 16384, &map_t, fb, t * kTileN + 64 * h, (int)rank * (D / 2));
          }
        }
      }
    }
  } else if (warp == 3) {
    // ===================================================== per-column constants, one tile ahead of the epilogue
    //   fast (statistics within 60 binades, see wscale_kernel): field 0 = 2^(M - c2_j) q_j;  else 0 = -c2_j, 1 = q_j
    float* const consts = reinterpret_cast<float*>(sbase + kRgOffConst);
    const float kL2e = 1.4426950408889634f;
    const bool fast = p.wscale[1] != 0.f;
    const float m_rc = p.wscale[2];
    uint32_t tt = 0;
    for (int job = pair_id; job < njobs; job += npairs) {
      const int sp = job % p.nsplit;
      const int t0 = sp * p.tiles_per_split, t1 = min(t0 + p.tiles_per_split, p.n_tiles);
      for (int t = t0; t < t1; ++t, ++tt) {
        float vc[4], vq[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int jcol = t * kTileN + lane + 32 * u;
          const bool ok = jcol < p.B;
          vc[u] = ok ? p.c[jcol] : 0.f;
          vq[u] = ok ? p.q[jcol] : 0.f;
        }
        mbar_wait(bar(kRgCstEmpty0 + (tt & 1)), ((tt >> 1) & 1) ^ 1);
        float* dst = consts + (tt & 1) * 256;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int col = lane + 32 * u;
          const bool ok = t * kTileN + col < p.B;
          const float c2 = vc[u] * kL2e;
          if (fast) {
            dst[col] = ok ? ex2f(m_rc - c2) * vq[u] : 0.f;
          } else {
            dst[col] = -c2;
            dst[128 + col] = vq[u];
          }
        }
        mbar_arrive_local(bar(kRgCstFull0 + (tt & 1)));
      }
    }
  } else if (warp == 1) {
    // ===================================================== MMA issuer
    if (leader && elect_one()) {
      constexpr uint32_t idesc_s = idesc_f16(256, kTileN);
      const uint32_t idesc_g = idesc_f16(256, D);
      const uint32_t tDT = tmem_base + kAcc;
      uint32_t it = 0, tt = 0, gt = 0, jj = 0;
      auto grad_tile = [&](bool first_of_job) {     // dT += W I_j of the tile whose weights are in the buffers
        for (int h = 0; h < 2; ++h) {
          mbar_wait(bar(kRgWFull0 + h), gt & 1);
          mbar_wait(bar(kRgXTFull0 + h), gt & 1);
          tc_fence_after();
          const uint64_t wd = smem_desc_sw128(base + kRgOffW + h * 16384), xd = smem_desc_sw128(base + kRgOffXT + h * 16384);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
            mma_f16_pair(tDT, desc_advance_k(wd, ks), desc_advance_k(xd, ks), idesc_g, (first_of_job && h == 0 && ks == 0) ? 0u : 1u);
          mma_commit_pair(bar(kRgGradDone0 + h), 3);
        }
        ++gt;
      };
      for (int job = pair_id; job < njobs; job += npairs, ++jj) {
        const int sp = job % p.nsplit;
        const int t0 = sp * p.tiles_per_split, t1 = min(t0 + p.tiles_per_split, p.n_tiles);
        mbar_wait(bar(kRgAFull), jj & 1);
        tc_fence_after();
        for (int t = t0; t < t1; ++t, ++tt) {
          const uint32_t buf = tt & 1, use = tt >> 1;
          mbar_wait(bar(kRgTmemEmpty0 + buf), (use & 1) ^ 1);
          tc_fence_after();
          const uint32_t tS = tmem_base + buf * 128;
          for (int c = 0; c < nkc; ++c, ++it) {
            const uint32_t slot = it % kRgSlots, par = (it / kRgSlots) & 1;
            mbar_wait(bar(kRgFull0 + slot), par);
            tc_fence_after();
            const uint32_t sb = base + kRgOffRing + slot * kRgSlotBytes;
            const uint64_t aT = smem_desc_sw128(base + kRgOffA + c * 16384), aTl = smem_desc_sw128(sb);
            const uint64_t bI = smem_desc_sw128(sb + 16384), bIl = smem_desc_sw128(sb + 24576);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              const uint64_t kT = desc_advance_k(aT, ks), kb = desc_advance_k(bI, ks);
              mma_f16_pair(tS, kT, kb, idesc_s, (c > 0 || ks > 0) ? 1u : 0u);      // S = T_i I_j^T, three passes (or one)
              if (PASSES == 3) {
                mma_f16_pair(tS, kT, desc_advance_k(bIl, ks), idesc_s, 1u);
                mma_f16_pair(tS, desc_advance_k(aTl, ks), kb, idesc_s, 1u);
              }
            }
            mma_commit_pair(bar(kRgEmpty0 + slot), 3);
          }
          mma_commit_pair(bar(kRgTmemFull0 + buf), 3);
          if (t == t0) {
            mbar_wait(bar(kRgAccEmpty), (jj & 1) ^ 1);     // the previous job's accumulator was read out
            tc_fence_after();
          } else {
            grad_tile(t - 1 == t0);
          }
        }
        grad_tile(t1 - 1 == t0);
        mma_commit_pair(bar(kRgAccFull), 3);
        mma_commit_pair(bar(kRgJobDone), 3);
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ===================================================== epilogue: thread = (TMEM lane m, column half h)
    const int q4 = warp & 3, h = (warp - 4) >> 2;
    const int m = q4 * 32 + lane;
    const uint32_t lane_field = (uint32_t)(q4 * 32) << 16;
    const float* const consts = reinterpret_cast<const float*>(sbase + kRgOffConst);
    const float kL2e = 1.4426950408889634f;
    const float inv_s = p.scale[1], inv_s2 = p.scale[2];
    const float cS2 = inv_s2 * p.inv_tau * kL2e;
    const float wS = inv_s * p.inv_tau * p.wscale[0];
    const bool fast = p.wscale[1] != 0.f;
    const float m_rc = p.wscale[2];
    uint32_t tt = 0, jj = 0;
    for (int job = pair_id; job < njobs; job += npairs, ++jj) {
      const int rb = job / p.nsplit, sp = job % p.nsplit;
      const int t0 = sp * p.tiles_per_split, t1 = min(t0 + p.tiles_per_split, p.n_tiles);
      const int lrow = rb * 256 + (int)rank * kRgRowsCta + m;
      const int gi = p.row_offset + lrow;
      const bool row_ok = lrow < p.b;
      const float r2_i = row_ok ? p.r[gi] * kL2e : 0.f;
      const float fC_i = ex2f(r2_i - m_rc);
      const float wrow = row_ok ? wS : 0.f;          // rows past the strip store exact zeros
      for (int t = t0; t < t1; ++t, ++tt) {
        const uint32_t buf = tt & 1, use = tt >> 1;
        mbar_wait(bar(kRgCstFull0 + (tt & 1)), (tt >> 1) & 1);
        const float* cst = consts + (tt & 1) * 256 + 64 * h;
        mbar_wait(bar(kRgTmemFull0 + buf), use & 1);
        tc_fence_after();
        const uint32_t tS = tmem_base + buf * 128 + lane_field + 64 * h;
        const bool ragged = (t + 1) * kTileN > p.B;   // last tile of a batch that is not a multiple of 128
        uint32_t wp[32];
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          float v[32];
          tmem_ld32(tS + 32 * half, v);
          tmem_ld_wait();
          if (half == 1) {
            tc_fence_before();
            mbar_arrive_cluster(bar(kRgTmemEmpty0 + buf), 0);
          }
#pragma unroll
          for (int e = 0; e < 32; e += 4) {
            const float4 f0 = *reinterpret_cast<const float4*>(cst + 32 * half + e);
            const float4 f1 = fast ? make_float4(0.f, 0.f, 0.f, 0.f) : *reinterpret_cast<const float4*>(cst + 128 + 32 * half + e);
            const float k0[4] = {f0.x, f0.y, f0.z, f0.w}, k1[4] = {f1.x, f1.y, f1.z, f1.w};
            float w[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const float a = v[e + u];
              const float e1 = ex2f(fmaf(a, cS2, -r2_i));                       // softmax_row(S)_ij
              float dS;
              if (fast) dS = e1 * fmaf(fC_i, k0[u], 1.f);                       // + q_j softmax_col(S)_ij, factored
              else dS = fmaf(ex2f(fmaf(a, cS2, k0[u])), k1[u], e1);
              w[u] = dS * wrow;
            }
            __half2 x = __floats2half2_rn(w[0], w[1]), y = __floats2half2_rn(w[2], w[3]);
            wp[16 * half + (e >> 1)] = *reinterpret_cast<uint32_t*>(&x);
            wp[16 * half + (e >> 1) + 1] = *reinterpret_cast<uint32_t*>(&y);
          }
        }
        // the half-h weight buffer: drained by the previous tile's gradient MMAs
        mbar_wait(bar(kRgGradDone0 + h), (tt & 1) ^ 1);
        uint8_t* wsm = sbase + kRgOffW + h * 16384 + m * 128;     // row m of a 128 x 64 fp16 tile, SWIZZLE_128B
#pragma unroll
        for (int k = 0; k < 8; ++k)
          *reinterpret_cast<uint4*>(wsm + ((k ^ (m & 7)) * 16)) = make_uint4(wp[4 * k], wp[4 * k + 1], wp[4 * k + 2], wp[4 * k + 3]);
        if (ragged) zero_padding_cols(wsm, m, max(p.B - t * kTileN - 64 * h, 0), 64);   // (the stored strip's copy: see pair_kernel)
        fence_proxy_async_smem();
        mbar_arrive_cluster(bar(kRgWFull0 + h), 0);
        uint4* wg = reinterpret_cast<uint4*>(p.wout + (size_t)lrow * p.Bp + (size_t)t * kTileN + 64 * h);   // one full line
#pragma unroll
        for (int k = 0; k < 8; ++k) wg[k] = make_uint4(wp[4 * k], wp[4 * k + 1], wp[4 * k + 2], wp[4 * k + 3]);
        mbar_arrive_local(bar(kRgCstEmpty0 + (tt & 1)));
      }
      // ---- end of job: this job's partial dT (lane m, columns [h D/2, (h + 1) D/2))
      mbar_wait(bar(kRgAccFull), jj & 1);
      tc_fence_after();
      float* out = p.part + ((size_t)sp * p.bpad + lrow) * D + h * (D / 2);
      for (int c0 = 0; c0 < D / 2; c0 += 32) {
        float v[32];
        tmem_ld32(tmem_base + lane_field + kAcc + h * (D / 2) + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 32; e += 4) *reinterpret_cast<float4*>(out + c0 + e) = make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]);
      }
      tc_fence_before();
      mbar_arrive_cluster(bar(kRgAccEmpty), 0);
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc_pair(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------
// Statistics sweep on large MMA instructions (same skeleton as rowgrad_kernel: CTA pair of 256 rows, cta_group::2 with
// M = 256, TMEM lane = row, 256 x 128 tiles, 64-cycle MMAs).  Two kinds, launched one after the other:
//   kRsS  S = T_i I_j^T in three passes -> row LSE of S (online, one partial per job) and the per-32-row column partials
//         of the column LSE (the transpose-reduce of pair_kernel<kStats>, twice per tile: a thread holds 64 columns).
//         T_i hi resident (64 KB); ring slot = one 64-wide K chunk of {T_i lo, I_j hi, I_j lo} (32 KB, 4 slots).
//   kRsZ  the tile-flag PROBE: Z = (I_i I_j^T + T_i T_j^T) tau/2 from the hi planes only -> flags.  I_i hi and T_i hi
//         resident (128 KB); ring slot = {I_j hi, T_j hi} of one K chunk (16 KB, 5 slots).  Z is symmetric, so a call that
//         owns every row visits the tiles ON OR ABOVE the diagonal only: a warp flags (row block, tile) by the row
//         criterion (max_j Z_ij against Z_ii) and the transposed pair (tile, row block) by the column criterion against
//         the smallest Z_jj of the tile (a superset of the per-column test, as rigorous as the row one).
// Four tile buffers of 128 TMEM columns.  Jobs are (256-row block, column split), optionally filtered by arrival chunk
// (see PairParams::chunk_k).
// ------------------------------------------------------------------------------------------
enum RsKind { kRsS = 0, kRsZ = 1 };
constexpr int kRsThreads = 384;
constexpr int kRsNBuf = 4;
constexpr int kRsOffScratch = 212992;                       // 208 KB: per-warp column maxima / end-of-job merge (2 KB)
constexpr int kRsOffBar = kRsOffScratch + 2048;
constexpr int kRsSmemBytes = kRsOffBar + 256 + 512;
enum RsBar { kRsFull0 = 0, kRsEmpty0 = 5, kRsAFull = 10, kRsJobDone = 11, kRsTmemFull0 = 12, kRsTmemEmpty0 = 16, kRsNumBars = 20 };
struct RowSweepParams {
  int b, B, Bp, D, row_offset;
  int n_row_blocks, n_tiles, nsplit, tiles_per_split, bpad;     // row blocks of 256
  int chunk_k, chunk_blocks, chunk_m;                            // arrival-ordered launches (chunk_k < 0: every job)
  int tri;                                                       // kRsZ: tiles on or above the diagonal only
  float inv_tau, half_tau;
  const float* scale;
  float2* part;             // kRsS: [nsplit][bpad] (row max in log2 units, sum)
  float* colpart;           // kRsS: [(bpad / 32)][Bp]
  uint8_t* flags_out;       // kRsZ: [row blocks of 128][n_tiles]
  const float *norm_i, *norm_t;
  const float* tile_min_zjj2;   // kRsZ, tri: smallest Z_jj (log2 units) of every column tile
  int pk;                       // kRsZ: 64-wide K chunks of each half that are multiplied out (see probe_chunks)
  const float* rho;             // kRsZ: norm of the left-out dimensions of every row (nullptr: nothing is left out)
  const float* tile_max_rho;    // kRsZ: largest rho of every column tile
  const float* tile_max_n;      // kRsZ: largest row norm sqrt(|I_j|^2 + |T_j|^2) of every column tile
  const int* gate;              // kRsZ: optional device word, the launch returns unless it equals gate_want
  int gate_want;                // 1: the full re-probe (probe_gate_kernel's verdict), 0: the partial probe (probe_hopeless_kernel)
};
__device__ __forceinline__ int rs_njobs(const RowSweepParams& p) {
  if (p.chunk_k < 0) return p.n_row_blocks * p.nsplit;
  return p.chunk_blocks * (p.chunk_k + 1) * p.chunk_m + p.chunk_k * p.chunk_blocks * p.chunk_m;
}
__device__ __forceinline__ void rs_job(const RowSweepParams& p, int job, int& rb, int& sp) {
  if (p.chunk_k < 0) { rb = job / p.nsplit; sp = job % p.nsplit; return; }
  const int w = (p.chunk_k + 1) * p.chunk_m, first = p.chunk_blocks * w;
  if (job < first) { rb = p.chunk_k * p.chunk_blocks + job / w; sp = job % w; return; }
  job -= first;
  rb = job / p.chunk_m;
  sp = p.chunk_k * p.chunk_m + job % p.chunk_m;
}
// tile range of a job; kRsZ in triangle mode starts at the row block's own diagonal tile
template <int KIND>
__device__ __forceinline__ void rs_tiles(const RowSweepParams& p, int rb, int sp, int& t0, int& t1) {
  t0 = sp * p.tiles_per_split;
  t1 = min(t0 + p.tiles_per_split, p.n_tiles);
  if (KIND == kRsZ && p.tri) t0 = max(t0, 2 * rb);
}
template <int KIND, int PASSES>
__global__ void __launch_bounds__(kRsThreads, 1)
rowsweep_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
                const RowSweepParams p) {
  constexpr int kSlotBytes_ = KIND == kRsS ? 32768 : 16384;
  constexpr int kSlots = KIND == kRsS ? 4 : 5;
  constexpr int kOffRing = KIND == kRsS ? 65536 : 131072;
  static_assert(kOffRing + kSlots * kSlotBytes_ <= kRsOffScratch, "ring overlaps the scratch");
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  if (base - raw > 512u) __trap();
  uint8_t* const sbase = smem_raw + (base - raw);
  const uint32_t bar0 = base + kRsOffBar;
  auto bar = [&](int i) -> uint32_t { return bar0 + 8u * i; };
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(sbase + kRsOffBar + 8 * kRsNumBars);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair_id = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  if (KIND == kRsZ && p.gate != nullptr && *p.gate != p.gate_want) return;   // kernel-uniform (see RowSweepParams::gate)
  const int D = p.D, nkc = D >> 6;
  const int nkz = KIND == kRsS ? nkc : p.pk;          // K chunks (per half of X) a tile multiplies out
  const int njobs = rs_njobs(p);
  const int n_res = KIND == kRsS ? nkc : 2 * nkz;     // resident 16 KB chunks of this CTA's rows

  if (threadIdx.x == 0) {
    for (int s = 0; s < kSlots; ++s) { mbar_init(bar(kRsFull0 + s), 1); mbar_init(bar(kRsEmpty0 + s), 1); }
    mbar_init(bar(kRsAFull), 1);
    mbar_init(bar(kRsJobDone), 1);
    for (int i = 0; i < kRsNBuf; ++i) { mbar_init(bar(kRsTmemFull0 + i), 1); mbar_init(bar(kRsTmemEmpty0 + i), 2 * 256); }
    fence_mbar_init();
    prefetch_tmap(&map_a_hi); prefetch_tmap(&map_a_lo); prefetch_tmap(&map_b_hi); prefetch_tmap(&map_b_lo);
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
    // ===================================================== producer: resident rows + ring
    if (elect_one()) {
      uint32_t it = 0, jj = 0;
      for (int job = pair_id; job < njobs; job += npairs) {
        int rb, sp, t0, t1;
        rs_job(p, job, rb, sp);
        rs_tiles<KIND>(p, rb, sp, t0, t1);
        if (t0 >= t1) continue;
        const int row_a = p.row_offset + rb * 256 + (int)rank * 128;
        mbar_wait(bar(kRsJobDone), (jj & 1) ^ 1);
        ++jj;
        if (leader) mbar_arrive_expect_tx(bar(kRsAFull), 2u * (uint32_t)n_res * 16384u);
        if (KIND == kRsS) {
          for (int c = 0; c < nkc; ++c) tma_load_2d_pair(base + c * 16384, &map_a_hi, bar(kRsAFull), D + c * 64, row_a);   // T_i hi
        } else {
          for (int c = 0; c < nkz; ++c) {                                                                   // I_i hi, T_i hi
            tma_load_2d_pair(base + c * 16384, &map_a_hi, bar(kRsAFull), c * 64, row_a);
            tma_load_2d_pair(base + (nkc + c) * 16384, &map_a_hi, bar(kRsAFull), D + c * 64, row_a);
          }
        }
        for (int t = t0; t < t1; ++t) {
          const int j0 = t * kTileN + 64 * (int)rank;
          for (int c = 0; c < nkz; ++c, ++it) {
            const uint32_t slot = it % kSlots, par = (it / kSlots) & 1;
            mbar_wait(bar(kRsEmpty0 + slot), par ^ 1);
            const uint32_t fb = bar(kRsFull0 + slot), sb = base + kOffRing + slot * kSlotBytes_;
            if (leader) mbar_arrive_expect_tx(fb, (KIND == kRsS && PASSES != 3) ? 2u * 8192u : 2u * kSlotBytes_);
            if (KIND == kRsS) {
              if (PASSES == 3) tma_load_2d_pair(sb, &map_a_lo, fb, D + c * 64, row_a);            // T_i lo   (128 rows)
              tma_load_2d_pair(sb + 16384, &map_b_hi, fb, c * 64, j0);           // I_j hi   (64 rows)
              if (PASSES == 3) tma_load_2d_pair(sb + 24576, &map_b_lo, fb, c * 64, j0);           // I_j lo
            } else {
              tma_load_2d_pair(sb, &map_b_hi, fb, c * 64, j0);                   // I_j hi
              tma_load_2d_pair(sb + 8192, &map_b_hi, fb, D + c * 64, j0);        // T_j hi
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================== MMA issuer
    if (leader && elect_one()) {
      constexpr uint32_t idesc = idesc_f16(256, kTileN);
      uint32_t it = 0, tt = 0, jj = 0;
      for (int job = pair_id; job < njobs; job += npairs) {
        int rb, sp, t0, t1;
        rs_job(p, job, rb, sp);
        rs_tiles<KIND>(p, rb, sp, t0, t1);
        if (t0 >= t1) continue;
        mbar_wait(bar(kRsAFull), jj & 1);
        ++jj;
        tc_fence_after();
        for (int t = t0; t < t1; ++t, ++tt) {
          const uint32_t buf = tt % kRsNBuf, use = tt / kRsNBuf;
          mbar_wait(bar(kRsTmemEmpty0 + buf), (use & 1) ^ 1);
          tc_fence_after();
          const uint32_t tD = tmem_base + buf * 128;
          for (int c = 0; c < nkz; ++c, ++it) {
            const uint32_t slot = it % kSlots, par = (it / kSlots) & 1;
            mbar_wait(bar(kRsFull0 + slot), par);
            tc_fence_after();
            const uint32_t sb = base + kOffRing + slot * kSlotBytes_;
            if (KIND == kRsS) {
              const uint64_t aT = smem_desc_sw128(base + c * 16384), aTl = smem_desc_sw128(sb);
              const uint64_t bI = smem_desc_sw128(sb + 16384), bIl = smem_desc_sw128(sb + 24576);
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                const uint64_t kT = desc_advance_k(aT, ks), kb = desc_advance_k(bI, ks);
                mma_f16_pair(tD, kT, kb, idesc, (c > 0 || ks > 0) ? 1u : 0u);
                if (PASSES == 3) {
                  mma_f16_pair(tD, kT, desc_advance_k(bIl, ks), idesc, 1u);
                  mma_f16_pair(tD, desc_advance_k(aTl, ks), kb, idesc, 1u);
                }
              }
            } else {
              const uint64_t aI = smem_desc_sw128(base + c * 16384), aT = smem_desc_sw128(base + (nkc + c) * 16384);
              const uint64_t bI = smem_desc_sw128(sb), bT = smem_desc_sw128(sb + 8192);
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                mma_f16_pair(tD, desc_advance_k(aI, ks), desc_advance_k(bI, ks), idesc, (c > 0 || ks > 0) ? 1u : 0u);
                mma_f16_pair(tD, desc_advance_k(aT, ks), desc_advance_k(bT, ks), idesc, 1u);
              }
            }
            mma_commit_pair(bar(kRsEmpty0 + slot), 3);
          }
          mma_commit_pair(bar(kRsTmemFull0 + buf), 3);
        }
        mma_commit_pair(bar(kRsJobDone), 3);
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ===================================================== epilogue: thread = (TMEM lane m, column half h)
    const int q4 = warp & 3, h = (warp - 4) >> 2;
    const int m = q4 * 32 + lane;
    const uint32_t lane_field = (uint32_t)(q4 * 32) << 16;
    float* const scratch = reinterpret_cast<float*>(sbase + kRsOffScratch);
    const float kL2e = 1.4426950408889634f;
    const float inv_s2 = p.scale[2];
    const float cS2 = inv_s2 * p.inv_tau * kL2e, cZ2 = inv_s2 * p.half_tau * kL2e;
    const float zmargin2 = kProbeMargin2 + (1.f / 512.f) * (8.f * (float)D * inv_s2 * p.half_tau * kL2e);
    uint32_t tt = 0;
    for (int job = pair_id; job < njobs; job += npairs) {
      int rb, sp, t0, t1;
      rs_job(p, job, rb, sp);
      const int lrow = rb * 256 + (int)rank * 128 + m;
      const int gi = p.row_offset + lrow;
      const bool row_ok = lrow < p.b;
      rs_tiles<KIND>(p, rb, sp, t0, t1);
      if (t0 >= t1) continue;                                 // kRsZ below the diagonal: nothing to do (kRsS never)
      float mS = -INFINITY, sS = 0.f;
      float zii2 = 0.f, rho2 = 0.f, rnd2 = 0.f;
      if (KIND == kRsZ && row_ok) {
        const float ni = p.norm_i[gi], nt = p.norm_t[gi];
        zii2 = (ni * ni + nt * nt) * p.half_tau * kL2e;
        if (p.rho != nullptr) {
          // left-out dimensions: Z_ij <= E_ij + tau/2 rho_i rho_j (Cauchy-Schwarz; 1.0001 covers the fp32 norms' rounding).
          // The worst-case rounding bound of the full probe (zmargin2: every |x s| < 2) would swallow what the partial
          // probe has left of the threshold, so its rounding term comes from the norms as well: the hi planes are within
          // 2^-11 relative of x (normal halfs), so |E_ij - E_ij(hi)| <= tau/2 2^-10 (1 + 2^-12) |x_i| |x_j| by
          // Cauchy-Schwarz again; the factor 1.05 also covers the truncating fp32 accumulation of the tensor cores over
          // K <= 256 (<= 256 2^-22 = 6% of 2^-10, relative to the same |x_i| |x_j|); subnormal halfs (absolute error
          // 2^-25 each) are covered by the margin at the comparison.
          rho2 = p.rho[gi] * p.half_tau * kL2e * 1.0001f;
          rnd2 = sqrtf(ni * ni + nt * nt) * p.half_tau * kL2e * (1.07f / 1024.f);
        }
      }
      const int rb128 = rb * 2 + (int)rank;                   // this CTA's 128-row block of the strip
      for (int t = t0; t < t1; ++t, ++tt) {
        const uint32_t buf = tt % kRsNBuf, use = tt / kRsNBuf;
        mbar_wait(bar(kRsTmemFull0 + buf), use & 1);
        tc_fence_after();
        const uint32_t tD = tmem_base + buf * 128 + lane_field + 64 * h;
        const bool ragged = (t + 1) * kTileN > p.B;
        float cmz = -INFINITY;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          float v[32];
          tmem_ld32(tD + 32 * half, v);
          tmem_ld_wait();
          if (half == 1) {
            tc_fence_before();
            mbar_arrive_cluster(bar(kRsTmemEmpty0 + buf), 0);
          }
          const int jl0 = 64 * h + 32 * half;                 // first tile column of these 32
          if (ragged) {
            const int jlim = p.B - t * kTileN;
#pragma unroll
            for (int e = 0; e < 32; ++e) if (jl0 + e >= jlim) v[e] = -INFINITY;
          }
          float c4[4] = {fmaxf(v[0], v[4]), fmaxf(v[1], v[5]), fmaxf(v[2], v[6]), fmaxf(v[3], v[7])};
#pragma unroll
          for (int e = 8; e < 32; e += 4) {
#pragma unroll
            for (int u = 0; u < 4; ++u) c4[u] = fmaxf(c4[u], v[e + u]);
          }
          const float cm = fmaxf(fmaxf(c4[0], c4[1]), fmaxf(c4[2], c4[3]));
          if (KIND == kRsZ) {
            cmz = fmaxf(cmz, cm);
          } else {
            // ---- row LSE of S, online.  The 32 exponentials are taken against the chunk's OWN row maximum cm (exact: the
            // largest term is 1) and shared with the column partials below; the chunk's sum joins the running (mS, sS)
            // with two more exponentials per row (an unchanged maximum rescales by exactly 1).
            float a[32];
            if (cm != -INFINITY) {
              float a4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
              for (int e = 0; e < 32; e += 4) {
#pragma unroll
                for (int u = 0; u < 4; ++u) { a[e + u] = ex2f((v[e + u] - cm) * cS2); a4[u] += a[e + u]; }
              }
              const float mn = fmaxf(mS, cm);
              sS = sS * ex2f((mS - mn) * cS2) + ((a4[0] + a4[1]) + (a4[2] + a4[3])) * ex2f((cm - mn) * cS2);
              mS = mn;
            } else {
#pragma unroll
              for (int e = 0; e < 32; ++e) a[e] = 0.f;
            }
            // ---- column partials: this warp's 32 x 32 block (lane = row) -> LSE over its rows of each column, from a
            // transpose-reduce in registers (five exchange steps, lane l ends up owning column l).
            // Common case (every row of the warp real, every column of the tile too): the SAME exponentials, weighted per
            // row by w_i = 2^((cm_i - M) c) against the block maximum M (one CREDUX, one exponential per row): column j's
            // sum is sum_i a_ij w_i = sum_i 2^((S_ij - M) c).  A column whose every entry lies so far below M that its sum
            // leaves the safe range (< 2^-100: a term that underflowed could then matter by more than 2^-26 of it) sends
            // the block down the exact path below - per-column maxima from redux.sync.max.f32 (one CREDUX per column,
            // warp-uniform result), exponentials against the column's OWN maximum.
            const int g32 = (rb * 256 + (int)rank * 128 + q4 * 32) >> 5;
            float* const cp_out = p.colpart + (size_t)g32 * p.Bp + (size_t)t * kTileN + jl0 + lane;
            bool col_done = false;
            if (!ragged && __all_sync(0xffffffffu, row_ok)) {
              float M;
              asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(M) : "f"(cm));
              const float w = ex2f((cm - M) * cS2);
#pragma unroll
              for (int e = 0; e < 32; ++e) a[e] *= w;
#pragma unroll
              for (int s2 = 16; s2 >= 1; s2 >>= 1) {
                const bool up = (lane & s2) != 0;
#pragma unroll
                for (int k = 0; k < s2; ++k) {
                  const float keep = up ? a[k + s2] : a[k], send = up ? a[k] : a[k + s2];
                  a[k] = keep + __shfl_xor_sync(0xffffffffu, send, s2);
                }
              }
              if (__all_sync(0xffffffffu, a[0] >= 7.8886e-31f)) {       // 2^-100
                *cp_out = fmaf(M, cS2, lg2f(a[0]));
                col_done = true;
              }
            }
            if (!col_done) {
              float* cmx = scratch + (warp - 4) * 32;
              __syncwarp();
#pragma unroll
              for (int e = 0; e < 32; ++e) {
                float cme;
                const float in = row_ok ? v[e] : -INFINITY;
                asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(cme) : "f"(in));
                if (lane == 0) cmx[e] = cme;
                const float ref = cme == -INFINITY ? 0.f : cme;
                a[e] = row_ok ? ex2f((v[e] - ref) * cS2) : 0.f;
              }
              __syncwarp();
              const float cm_own = cmx[lane];
#pragma unroll
              for (int s2 = 16; s2 >= 1; s2 >>= 1) {
                const bool up = (lane & s2) != 0;
#pragma unroll
                for (int k = 0; k < s2; ++k) {
                  const float keep = up ? a[k + s2] : a[k], send = up ? a[k] : a[k + s2];
                  a[k] = keep + __shfl_xor_sync(0xffffffffu, send, s2);
                }
              }
              *cp_out = cm_own == -INFINITY ? -INFINITY : fmaf(cm_own, cS2, lg2f(a[0]));
            }
          }
        }
        if (KIND == kRsZ) {
          // row criterion: rz_i >= Z_ii, so a row whose largest (hi-plane) Z stays 44 binades + the rounding bound below it
          // holds no P_ij >= 2^-44 in this tile
          float z2 = -INFINITY, zm2 = zmargin2;
          if (row_ok) {
            z2 = cmz * cZ2;
            if (p.rho != nullptr) {
              z2 += fmaf(rho2, p.tile_max_rho[t], rnd2 * p.tile_max_n[t]);
              zm2 = kProbeMargin2 + 8.f * (float)D * 2.98e-8f * cZ2;      // slack + 2 D products of |x s| < 2 with a 2^-25 error, twice
            }
          }
          const bool hit = z2 >= zii2 - kFlagTheta2 - zm2;
          if (__any_sync(0xffffffffu, hit) && lane == 0) p.flags_out[(size_t)rb128 * p.n_tiles + t] = 1;
          if (p.tri && t != rb128) {
            // column criterion for the transposed tile (rows of tile t, columns of this row block), by Z_ij = Z_ji
            const float wm = warp_max(z2);
            if (lane == 0 && wm >= p.tile_min_zjj2[t] - kFlagTheta2 - zm2) p.flags_out[(size_t)t * p.n_tiles + rb128] = 1;
          }
        }
      }
      if (KIND == kRsS) {
        // ---- end of job: the two column halves of a row meet in shared memory (h = 1 hands over, h = 0 writes)
        named_bar_sync(2, 256);
        float* sc = scratch + 256;       // behind the per-warp column maxima: [2][128]
        if (h == 1) { sc[m] = mS * cS2; sc[128 + m] = sS; }
        named_bar_sync(2, 256);
        if (h == 0) {
          OnlineLse2 l;
          l.m = mS * cS2; l.s = sS;
          l.merge(sc[m], sc[128 + m]);
          p.part[(size_t)sp * p.bpad + lrow] = make_float2(l.m, l.s);
        }
      }
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc_pair(tmem_base, 512);
}

// smallest Z_jj (log2 units) of every 128-column tile (kRsZ, triangle mode)
// and the largest rho (norm of the dimensions the probe leaves out) of the same tile
__global__ void __launch_bounds__(128) tile_min_zjj_kernel(const float* __restrict__ norm_i, const float* __restrict__ norm_t,
                                                           const float* __restrict__ rho, int B, float half_tau,
                                                           float* __restrict__ out, float* __restrict__ out_rho,
                                                           float* __restrict__ out_n) {
  __shared__ float sm[4], sr[4], sn[4];
  const int j = blockIdx.x * 128 + threadIdx.x;
  float z = INFINITY, r = 0.f, n = 0.f;
  if (j < B) {
    const float ni = norm_i[j], nt = norm_t[j];
    z = (ni * ni + nt * nt) * half_tau * 1.4426950408889634f;
    r = rho[j];
    n = sqrtf(ni * ni + nt * nt);
  }
  for (int o = 16; o > 0; o >>= 1) {
    z = fminf(z, __shfl_xor_sync(0xffffffffu, z, o));
    r = fmaxf(r, __shfl_xor_sync(0xffffffffu, r, o));
    n = fmaxf(n, __shfl_xor_sync(0xffffffffu, n, o));
  }
  if ((threadIdx.x & 31) == 0) { sm[threadIdx.x >> 5] = z; sr[threadIdx.x >> 5] = r; sn[threadIdx.x >> 5] = n; }
  __syncthreads();
  if (threadIdx.x == 0) {
    out[blockIdx.x] = fminf(fminf(sm[0], sm[1]), fminf(sm[2], sm[3]));
    out_rho[blockIdx.x] = fmaxf(fmaxf(sr[0], sr[1]), fmaxf(sr[2], sr[3]));
    out_n[blockIdx.x] = fmaxf(fmaxf(sn[0], sn[1]), fmaxf(sn[2], sn[3]));
  }
}
// Before the partial probe: a batch for which the bound ALONE (E_ij = 0) already reaches the threshold inside most tiles
// (small norms - the soft regime - or all the energy in the left-out dimensions) cannot be served by it; *hopeless is set
// (sticky over the arrival-ordered launches of one statistics sweep: stats_begin clears it) and the partial probe returns
// at once.  Only the first n_valid tiles have their rows staged yet.
__global__ void __launch_bounds__(256) probe_hopeless_kernel(const float* __restrict__ tile_min_zjj2,
                                                             const float* __restrict__ tile_max_rho, int n_valid,
                                                             float half_tau, int* __restrict__ hopeless) {
  __shared__ int cnt;
  if (threadIdx.x == 0) cnt = 0;
  __syncthreads();
  int c = 0;
  for (int t = threadIdx.x; t < n_valid; t += blockDim.x) {
    const float r = tile_max_rho[t];
    c += r * r * half_tau * 1.4426950408889634f >= tile_min_zjj2[t] - kFlagTheta2 - kProbeMargin2;
  }
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(&cnt, c);
  __syncthreads();
  if (threadIdx.x == 0 && 2 * cnt > n_valid) *hopeless = 1;
}
// The partial probe's verdict: with more flagged tiles than a concentrated batch can have (its diagonal + 1/64 of all
// tiles) the Cauchy-Schwarz bound was too loose for this batch - clear the bitmap and let the full probe run (*gate = 1);
// likewise when the partial probe was skipped as hopeless (gate[1]).
__global__ void __launch_bounds__(1024) probe_gate_kernel(uint8_t* __restrict__ flags, int n, int limit, int* __restrict__ gate) {
  __shared__ int cnt;
  if (threadIdx.x == 0) cnt = 0;
  __syncthreads();
  int c = 0;
  const bool vec = (reinterpret_cast<uintptr_t>(flags) & 15) == 0 && n % 16 == 0;   // flag bytes are 0 / 1
  if (vec) {
    for (int i = threadIdx.x; i < n / 16; i += blockDim.x) {
      const uint4 w = reinterpret_cast<const uint4*>(flags)[i];
      c += __popc(w.x) + __popc(w.y) + __popc(w.z) + __popc(w.w);
    }
  } else {
    for (int i = threadIdx.x; i < n; i += blockDim.x) c += flags[i] != 0;
  }
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(&cnt, c);
  __syncthreads();
  const bool redo = cnt > limit || gate[1] != 0;
  if (redo) {
    if (vec) for (int i = threadIdx.x; i < n / 16; i += blockDim.x) reinterpret_cast<uint4*>(flags)[i] = make_uint4(0u, 0u, 0u, 0u);
    else for (int i = threadIdx.x; i < n; i += blockDim.x) flags[i] = 0;
  }
  if (threadIdx.x == 0) *gate = redo ? 1 : 0;
}
// row LSE of S from rowsweep_kernel<kRsS>'s partials
__global__ void __launch_bounds__(256) rowsweep_finalize_kernel(const float2* __restrict__ part, int nsplit, int bpad, int b,
                                                                float* __restrict__ r) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= b) return;
  OnlineLse2 l;
  l.init();
  for (int s = 0; s < nsplit; ++s) {
    const float2 v = part[(size_t)s * bpad + i];
    l.merge(v.x, v.y);
  }
  r[i] = (l.m + log2f(l.s)) * kLn2;
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(f);
  }
  return fn;
}

// 2-D fp16 tensor [rows][cols] (cols contiguous), box {64 cols, box_rows}, 128-byte swizzle
static int make_map(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  EncodeTiledFn fn = encode_fn();
  MC_REQUIRE(fn != nullptr, MC_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * sizeof(__half)};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  MC_REQUIRE(r == CUDA_SUCCESS, MC_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return MC_OK;
}

struct Split {
  int n_row_blocks, n_tiles, nsplit, tiles_per_split, bpad;
};
// Per-job overhead of a sweep, in tiles (fitted to the 4096-row strip of B = 32768, tools/strip_sweep.py: the gradient
// sweep pays the load of its resident rows, the pipeline fill of its weight tiles and the read-out of 2 x 64 x D
// accumulators per job, and every extra split adds a set of partial gradients to fold: 0.578 ms with 16 splits, 0.505
// with 2; the statistics sweep is cheap per job)
constexpr double kOvhStats = 1.5, kOvhRowLoss = 0.5, kOvhBwd = 6.0;
template <int PHASE> constexpr double phase_ovh() { return (PHASE == kBwd || PHASE == kBwdW || PHASE == kBwdP) ? kOvhBwd : (PHASE == kRowLoss ? kOvhRowLoss : kOvhStats); }
static Split choose_split(int b, int B, double ovh = kOvhRowLoss, int align = 1) {
  Split s;
  s.n_row_blocks = (b + 127) / 128;
  s.bpad = s.n_row_blocks * 128;
  s.n_tiles = (int)(round_up((size_t)B, 128) / 128);
  const int npairs = num_sms() / 2;
  int best = 1;
  double best_cost = 1e30;
  const int max_split = s.n_tiles < kMaxSplit ? s.n_tiles : kMaxSplit;
  for (int ns = align; ns <= max_split; ns += align) {   // align > 1: the column splits must not straddle a row chunk
    const int tps = (s.n_tiles + ns - 1) / ns;
    if ((long)(ns - 1) * tps >= s.n_tiles) continue;     // the last split would be empty (the gradient roles assume >= 1 tile per job)
    double cost = 0.02 * ns;
    if (align > 1) {
      // arrival-ordered launches (PairParams::chunk_k): every launch pays its own partly filled last round
      if (s.n_tiles % ns != 0 || s.n_row_blocks % align != 0) continue;
      const long cb = s.n_row_blocks / align, cm = ns / align;
      for (int k = 0; k < align; ++k) {
        const long jobs = cb * (k + 1) * cm + (long)k * cb * cm;
        cost += (double)((jobs + npairs - 1) / npairs) * (tps + ovh);
      }
    } else {
      const long jobs = (long)s.n_row_blocks * ns;
      cost += (double)((jobs + npairs - 1) / npairs) * (tps + ovh);
    }
    if (cost < best_cost - 1e-9) { best_cost = cost; best = ns; }
  }
  static const int forced = getenv("MAE_CLIP_NSPLIT") ? atoi(getenv("MAE_CLIP_NSPLIT")) : 0;   // experiments only
  if (forced >= 1 && forced <= max_split && align == 1) best = forced;
  s.nsplit = best;
  s.tiles_per_split = (s.n_tiles + best - 1) / best;
  return s;
}

size_t planes_bytes(int B, int D, int /*mode*/) { return supported(D) ? planes_layout(B, D).total : 0; }

// can the statistics sweep of a whole batch (b == B) run as `chunks` arrival-ordered launches?
bool stats_chunkable(int B, int D, int chunks) {
  if (!supported(D) || chunks < 2 || B % 128 != 0) return false;
  const int nb = B / 128;
  if (nb % chunks != 0 || chunks > kMaxSplit) return false;
  Split sp = choose_split(B, B, kOvhStats, chunks);
  return sp.nsplit % chunks == 0 && sp.n_tiles % sp.nsplit == 0 && sp.n_tiles == sp.n_row_blocks;
}

// Column LSE of S.  Two forms (SURVEY section 7 hard part c):
//   transposed strip  the statistics sweep also computes S^T-strip = I_i T_j^T (3 more tensor-core passes per tile)
//                     and takes its row LSE: c of the OWNED rows, nothing to merge
//   column partials   no transposed strip: every epilogue warp reduces its 32 x 32 block along the rows with two
//                     transpose-reduces in registers (exact: exponentials against each column's own maximum) and writes
//                     one log-sum-exp per column and 32-row group; colpart_merge_kernel folds the (b / 32) x B partials.
// Measured at B = 32768 (profiles/r02_*): statistics sweep 3.19 -> see DESIGN.  The partials describe ALL columns over
// the OWNED rows, so under row sharding they would have to be merged across ranks; they are used when one call owns
// every row (b == B: the single-GPU step); MAE_CLIP_COLPART=0 keeps the transposed strip (A/B switch).
static bool use_colpart(int b, int B) {
  static const bool off = getenv("MAE_CLIP_COLPART") != nullptr && getenv("MAE_CLIP_COLPART")[0] == '0';
  return !off && b == B;
}
static size_t colpart_bytes(int b, int B, bool forced = false) {
  if (!forced && !use_colpart(b, B)) return 0;
  return round_up((round_up((size_t)b, 256) / 32) * round_up((size_t)B, 128) * sizeof(float), 256);   // rowsweep_kernel pads to 256 rows
}
// workspace of the sharded column-partials form (stats with c_part_all): the phase partials + the (b / 32) x B partials
size_t stats_colpart_workspace_bytes(int b, int B, int D, int mode) {
  return core_workspace_bytes(b, B, D, mode) - colpart_bytes(b, B) + colpart_bytes(b, B, true);
}

static size_t rowsweep_extra_bytes(int b, int B) {
  return round_up((size_t)kMaxSplit * round_up((size_t)b, 256) * sizeof(float2), 256) + round_up(3 * (round_up((size_t)B, 128) / 128) * sizeof(float) + 16, 256);   // tile min Z_jj, tile max rho / norm, the probe gate
}
// rowgrad_kernel: row blocks of 256, tiles of 256 x 128; same cost model as choose_split (a job pays ~3 tiles of overhead)
static Split choose_split_rows256(int b, int B, int align = 1, double ovh = 3.0) {
  Split s;
  s.n_row_blocks = (b + 255) / 256;
  s.bpad = s.n_row_blocks * 256;
  s.n_tiles = (int)(round_up((size_t)B, 128) / 128);
  const int npairs = num_sms() / 2;
  int best = 1;
  double best_cost = 1e30;
  const int max_split = s.n_tiles < kMaxSplit ? s.n_tiles : kMaxSplit;
  for (int ns = align; ns <= max_split; ns += align) {
    const int tps = (s.n_tiles + ns - 1) / ns;
    if ((long)(ns - 1) * tps >= s.n_tiles) continue;     // no empty last split: rowgrad_kernel's roles assume >= 1 tile per job
    double cost = 0.04 * ns;
    if (align > 1) {   // arrival-ordered launches: see choose_split
      if (s.n_tiles % ns != 0 || s.n_row_blocks % align != 0) continue;
      const long cb = s.n_row_blocks / align, cm = ns / align;
      for (int k = 0; k < align; ++k) {
        const long jobs = cb * (k + 1) * cm + (long)k * cb * cm;
        cost += (double)((jobs + npairs - 1) / npairs) * (tps + ovh);
      }
    } else {
      const long jobs = (long)s.n_row_blocks * ns;
      cost += (double)((jobs + npairs - 1) / npairs) * (tps + ovh);
    }
    if (cost < best_cost - 1e-9) { best_cost = cost; best = ns; }
  }
  s.nsplit = best;
  s.tiles_per_split = (s.n_tiles + best - 1) / best;
  return s;
}
static size_t rowgrad_part_bytes(int b, int B, int D) {
  Split s = choose_split_rows256(b, B);
  return round_up((size_t)s.nsplit * s.bpad * D * sizeof(float), 256);
}

size_t core_workspace_bytes(int b, int B, int D, int /*mode*/) {
  Split s = choose_split(b, B, kOvhStats), sr = choose_split(b, B, kOvhRowLoss), sb = choose_split(b, B, kOvhBwd);
  (void)sr;
  size_t stats = (size_t)kMaxSplit * 4 * s.bpad * sizeof(float2);   // any split count (the chunked launches align theirs)
  stats += rowsweep_extra_bytes(b, B);                               // rowsweep_kernel: row-LSE partials + per-tile min Z_jj
  size_t bwdp = (size_t)sb.nsplit * 2 * s.bpad * D * sizeof(float);
  {  // the split gradient: rowgrad_kernel's dT partials (row blocks of 256) + kBwdP's single (dT, dI) partial
    const size_t split_part = rowgrad_part_bytes(b, B, D) + (size_t)2 * s.bpad * D * sizeof(float);
    if (split_part > bwdp) bwdp = split_part;
  }
  return round_up(stats > bwdp ? stats : bwdp, 256) + 256 + colpart_bytes(b, B);  // + the weight-scale slot + column partials
}
static float* colpart_slot(void* ws, int b, int B, int D) {
  return reinterpret_cast<float*>(static_cast<char*>(ws) + core_workspace_bytes(b, B, D, 0) - colpart_bytes(b, B));
}
static float* wscale_slot(void* ws, int b, int B, int D) {
  return reinterpret_cast<float*>(static_cast<char*>(ws) + core_workspace_bytes(b, B, D, 0) - colpart_bytes(b, B) - 256);
}


// ------------------------------------------------------------------------------------------
// Peer-memory staging (row-sharded loss, one process per GPU): the embedding all-gather is fused
// into the operand staging.  Rank q keeps its (b, D) fp32 shards in a region every peer has
// mapped over NVLink; each rank pulls every row straight from its owner with 16-byte loads while
// it writes its local fp16 hi / lo planes, so the fp32 global batch is never assembled in HBM and
// no collective library call sits between the towers and the first sweep.
// ------------------------------------------------------------------------------------------
constexpr int kMaxPeers = 16;
struct PeerRows {
  const float* I[kMaxPeers];
  const float* T[kMaxPeers];
};

// local part of the global scale: largest magnitude of this rank's shards (+ optional copy of the
// shards into the exchange region, so the towers' output is read once)
__global__ void __launch_bounds__(256) amax_copy_kernel(const float4* __restrict__ I, const float4* __restrict__ T,
                                                        size_t n4, float4* __restrict__ I_copy,
                                                        float4* __restrict__ T_copy,
                                                        unsigned int* __restrict__ amax_bits) {
  float a = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 x = I[i], y = T[i];
    if (I_copy) I_copy[i] = x;
    if (T_copy) T_copy[i] = y;
    a = fmaxf(a, fmaxf(fmaxf(fabsf(x.x), fabsf(x.y)), fmaxf(fabsf(x.z), fabsf(x.w))));
    a = fmaxf(a, fmaxf(fmaxf(fabsf(y.x), fabsf(y.y)), fmaxf(fabsf(y.z), fabsf(y.w))));
  }
  a = warp_max(a);
  if ((threadIdx.x & 31) == 0 && a > 0.f) atomicMax(amax_bits, __float_as_uint(a));
}

// Fused staging: a block owns 32 global rows.  Each warp pulls four rows of [I_i || T_i] (16-byte
// loads, all in flight before the first use: they may cross NVLink), writes the scaled fp16 hi / lo
// planes and the row norms, and parks hi in a shared tile from which the block writes its
// 32-column slice of the transposed plane (64-byte runs) - fp32 rows are read once and the hi
// plane is never re-read.  Row gi belongs to rank gi / b (src.I[q] / src.T[q] = rank q's rows).
template <int D>
__global__ void __launch_bounds__(256) stage_fused_kernel(PeerRows src, int b, int B, int Bp,
                                                          const unsigned int* amax_slots, int nslots,
                                                          __half* __restrict__ Xh, __half* __restrict__ Xl,
                                                          __half* __restrict__ XhT, float* hdr,
                                                          float* __restrict__ norm_i, float* __restrict__ norm_t,
                                                          int blk0 /* first 32-row block of this launch */,
                                                          float* __restrict__ rho, int tail_c0 /* first float4 of a half the probe leaves out */) {
  constexpr int K2 = 2 * D, kVec = K2 / 128, kRows = 32, kPitch = K2 + 2;  // pitch in halfs: odd word count
  __shared__ __align__(16) __half tile[kRows * kPitch];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int j0 = (blockIdx.x + blk0) * kRows;
  unsigned int abits = 0;
  for (int q = 0; q < nslots; ++q) abits = max(abits, amax_slots[q]);
  const float amax = __uint_as_float(abits);
  float s = 1.f;
  if (amax > 0.f && amax < INFINITY) {
    int e;
    frexpf(amax, &e);        // amax = f * 2^e, f in [0.5, 1)
    s = ldexpf(1.f, 1 - e);  // amax * s in [1, 2)
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    reinterpret_cast<unsigned int*>(hdr)[0] = abits;
    hdr[1] = s; hdr[2] = 1.f / s; hdr[3] = (1.f / s) * (1.f / s);
  }
  float4 v[4][kVec];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gi = j0 + warp * 4 + i;
    if (gi < B) {
      const int q = gi / b, lr = gi - q * b;
      const float4* pi = reinterpret_cast<const float4*>(src.I[q] + (size_t)lr * D);
      const float4* pt = reinterpret_cast<const float4*>(src.T[q] + (size_t)lr * D);
#pragma unroll
      for (int u = 0; u < kVec; ++u) {
        const int c = lane + 32 * u;
        v[i][u] = (c < D / 4) ? pi[c] : pt[c - D / 4];
      }
    } else {
#pragma unroll
      for (int u = 0; u < kVec; ++u) v[i][u] = make_float4(0.f, 0.f, 0.f, 0.f);  // zero padding rows B .. Bp-1
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = warp * 4 + i, gi = j0 + r;
    if (gi >= Bp) continue;
    uint2* xh = reinterpret_cast<uint2*>(Xh + (size_t)gi * K2);
    uint2* xl = reinterpret_cast<uint2*>(Xl + (size_t)gi * K2);
    uint32_t* trow = reinterpret_cast<uint32_t*>(tile + r * kPitch);
    float ni = 0.f, nt = 0.f, nr = 0.f;
#pragma unroll
    for (int u = 0; u < kVec; ++u) {
      const int c = lane + 32 * u;
      const float raw[4] = {v[i][u].x, v[i][u].y, v[i][u].z, v[i][u].w};
      __half h[4], l[4];
      float nn = 0.f;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        nn = fmaf(raw[e], raw[e], nn);
        const float x = raw[e] * s;
        h[e] = __float2half_rn(x);
        l[e] = __float2half_rn(x - __half2float(h[e]));
      }
      if (c < D / 4) ni += nn; else nt += nn;
      if ((c < D / 4 ? c : c - D / 4) >= tail_c0) nr += nn;
      __half2 h01 = __halves2half2(h[0], h[1]), h23 = __halves2half2(h[2], h[3]);
      __half2 l01 = __halves2half2(l[0], l[1]), l23 = __halves2half2(l[2], l[3]);
      const uint32_t a0 = *reinterpret_cast<uint32_t*>(&h01), a1 = *reinterpret_cast<uint32_t*>(&h23);
      xh[c] = make_uint2(a0, a1);
      xl[c] = make_uint2(*reinterpret_cast<uint32_t*>(&l01), *reinterpret_cast<uint32_t*>(&l23));
      trow[2 * c] = a0;
      trow[2 * c + 1] = a1;
    }
    ni = warp_sum(ni);
    nt = warp_sum(nt);
    nr = warp_sum(nr);
    if (lane == 0) { norm_i[gi] = sqrtf(ni); norm_t[gi] = sqrtf(nt); rho[gi] = sqrtf(nr); }
  }
  __syncthreads();
  // transposed slice: XhT[k][j0 .. j0+32).  A warp instruction covers two k rows: lanes 0-15 -> k, 16-31 -> k+1,
  // each lane the pair of rows (2l, 2l+1); the odd word pitch keeps the column reads conflict-free.
  if (j0 + kRows > Bp) return;  // Bp is a multiple of 128: never taken, keeps the stores in range by construction
  const int l16 = lane & 15, kk = lane >> 4;
  for (int k = warp * 2 + kk; k < K2; k += 16) {
    const __half lo = tile[(2 * l16) * kPitch + k], hi = tile[(2 * l16 + 1) * kPitch + k];
    __half2 pr = __halves2half2(lo, hi);
    *reinterpret_cast<uint32_t*>(XhT + (size_t)k * Bp + j0 + 2 * l16) = *reinterpret_cast<uint32_t*>(&pr);
  }
}

// Push variant of the exchange: every rank writes its shards into ALL ranks' (B, D) fp32 images
// of the global batch (posted NVLink stores, no round trip) while it reduces its local amax; the
// last block to finish publishes that amax into every rank's slot and re-arms the scratch words.
struct PushDst {
  float* I[kMaxPeers];
  float* T[kMaxPeers];
  unsigned int* slots[kMaxPeers];
};
__global__ void __launch_bounds__(256) push_shards_kernel(const float4* __restrict__ I, const float4* __restrict__ T,
                                                          size_t n4, size_t dst_off4, PushDst dst, int rank, int world,
                                                          unsigned int* __restrict__ scratch /* {amax, blocks done} */) {
  float a = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 x = I[i], y = T[i];
    for (int q = 0; q < world; ++q) {
      reinterpret_cast<float4*>(dst.I[q])[dst_off4 + i] = x;
      reinterpret_cast<float4*>(dst.T[q])[dst_off4 + i] = y;
    }
    a = fmaxf(a, fmaxf(fmaxf(fabsf(x.x), fabsf(x.y)), fmaxf(fabsf(x.z), fabsf(x.w))));
    a = fmaxf(a, fmaxf(fmaxf(fabsf(y.x), fabsf(y.y)), fmaxf(fabsf(y.z), fabsf(y.w))));
  }
  a = warp_max(a);
  if ((threadIdx.x & 31) == 0 && a > 0.f) atomicMax(scratch, __float_as_uint(a));
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int done = atomicAdd(scratch + 1, 1u) + 1u;
    if (done == gridDim.x) {
      __threadfence();
      const unsigned int bits = atomicExch(scratch, 0u);  // read the final maximum and re-arm
      scratch[1] = 0u;
      for (int q = 0; q < world; ++q) dst.slots[q][rank] = bits;
    }
  }
}

static void launch_stage_fused(const PeerRows& src, int b, int B, int D, const PlanesLayout& l,
                               const unsigned int* amax_slots, int nslots, __half* Xh, __half* Xl, __half* XhT,
                               float* hdr, float* norm_i, float* norm_t, cudaStream_t st) {
  const int blocks = l.Bp / 32;
  if (D == 256)
    stage_fused_kernel<256><<<blocks, 256, 0, st>>>(src, b, B, l.Bp, amax_slots, nslots, Xh, Xl, XhT, hdr, norm_i, norm_t, 0,
                                                    norm_i + (l.off_rho - l.off_norm_i) / 4, 16 * probe_chunks(D));
  else
    stage_fused_kernel<128><<<blocks, 256, 0, st>>>(src, b, B, l.Bp, amax_slots, nslots, Xh, Xl, XhT, hdr, norm_i, norm_t, 0,
                                                    norm_i + (l.off_rho - l.off_norm_i) / 4, 16 * probe_chunks(D));
}

int push_shards(const float* I_loc, const float* T_loc, int b, int D, int rank, int world, float* const* I_dst,
                float* const* T_dst, unsigned int* const* amax_slots, unsigned int* scratch, cudaStream_t st) {
  MC_REQUIRE(world >= 1 && world <= kMaxPeers && rank >= 0 && rank < world, MC_ERR_BAD_ARG,
             "clip_push_shards: rank %d / world %d outside [1, %d]", rank, world, kMaxPeers);
  MC_REQUIRE(D % 4 == 0 && aligned(I_loc, 16) && aligned(T_loc, 16), MC_ERR_ALIGN,
             "clip_push_shards: shards must be 16-byte aligned with D %% 4 == 0");
  PushDst dst;
  for (int q = 0; q < kMaxPeers; ++q) { dst.I[q] = nullptr; dst.T[q] = nullptr; dst.slots[q] = nullptr; }
  for (int q = 0; q < world; ++q) {
    MC_REQUIRE(I_dst[q] && T_dst[q] && amax_slots[q] && aligned(I_dst[q], 16) && aligned(T_dst[q], 16), MC_ERR_ALIGN,
               "clip_push_shards: destination of rank %d null or not 16-byte aligned", q);
    dst.I[q] = I_dst[q]; dst.T[q] = T_dst[q]; dst.slots[q] = amax_slots[q];
  }
  const size_t n4 = (size_t)b * D / 4;
  int nb = (int)((n4 + 255) / 256);
  if (nb > num_sms() * 4) nb = num_sms() * 4;
  push_shards_kernel<<<nb, 256, 0, st>>>(reinterpret_cast<const float4*>(I_loc), reinterpret_cast<const float4*>(T_loc), n4,
                                         (size_t)rank * n4, dst, rank, world, scratch);
  MC_LAUNCH_CHECK();
  return MC_OK;
}

int amax_copy(const float* I_loc, const float* T_loc, int b, int D, float* I_copy, float* T_copy,
              unsigned int* amax_bits, cudaStream_t st) {
  MC_REQUIRE(D % 4 == 0 && aligned(I_loc, 16) && aligned(T_loc, 16) && (!I_copy || aligned(I_copy, 16)) &&
                 (!T_copy || aligned(T_copy, 16)),
             MC_ERR_ALIGN, "clip_amax: embeddings must be 16-byte aligned with D %% 4 == 0");
  MC_CUDA(cudaMemsetAsync(amax_bits, 0, 4, st));
  const size_t n4 = (size_t)b * D / 4;
  int ab = (int)((n4 + 255) / 256);
  if (ab > num_sms() * 8) ab = num_sms() * 8;
  amax_copy_kernel<<<ab, 256, 0, st>>>(reinterpret_cast<const float4*>(I_loc), reinterpret_cast<const float4*>(T_loc), n4,
                                       reinterpret_cast<float4*>(I_copy), reinterpret_cast<float4*>(T_copy), amax_bits);
  MC_LAUNCH_CHECK();
  return MC_OK;
}

int prepare_peers(const float* const* I_peers, const float* const* T_peers, int world, int b, int D, int /*mode*/,
                  const unsigned int* amax_slots, void* planes_all, cudaStream_t st) {
  MC_REQUIRE(supported(D), MC_ERR_UNSUPPORTED, "tcgen05 engine needs D in {128, 256} (got %d)", D);
  MC_REQUIRE(world >= 1 && world <= kMaxPeers, MC_ERR_BAD_ARG, "clip_prepare_peers: world %d outside [1, %d]", world,
             kMaxPeers);
  MC_REQUIRE(aligned(planes_all, 256), MC_ERR_ALIGN, "clip_prepare_peers: planes buffer must be 256-byte aligned");
  PeerRows src;
  for (int q = 0; q < kMaxPeers; ++q) { src.I[q] = nullptr; src.T[q] = nullptr; }
  for (int q = 0; q < world; ++q) {
    MC_REQUIRE(I_peers[q] && T_peers[q] && aligned(I_peers[q], 16) && aligned(T_peers[q], 16), MC_ERR_ALIGN,
               "clip_prepare_peers: shard pointers of rank %d null or not 16-byte aligned", q);
    src.I[q] = I_peers[q];
    src.T[q] = T_peers[q];
  }
  const int B = world * b;
  PlanesLayout l = planes_layout(B, D);
  char* base = static_cast<char*>(planes_all);
  __half* Xh = reinterpret_cast<__half*>(base + l.off_hi);
  __half* Xl = reinterpret_cast<__half*>(base + l.off_lo);
  __half* XhT = reinterpret_cast<__half*>(base + l.off_hiT);
  float* hdr = reinterpret_cast<float*>(base + l.off_hdr);
  float* norm_i = reinterpret_cast<float*>(base + l.off_norm_i);
  float* norm_t = reinterpret_cast<float*>(base + l.off_norm_t);
  launch_stage_fused(src, b, B, D, l, amax_slots, world, Xh, Xl, XhT, hdr, norm_i, norm_t, st);
  MC_LAUNCH_CHECK();
  return MC_OK;
}

int prepare(const float* I_loc, const float* T_loc, int b, int B, int D, int row_offset, int /*mode*/,
            void* planes_all, cudaStream_t st) {
  MC_REQUIRE(supported(D), MC_ERR_UNSUPPORTED, "tcgen05 engine needs D in {128, 256} (got %d)", D);
  MC_REQUIRE(b == B && row_offset == 0, MC_ERR_UNSUPPORTED,
             "tcgen05 engine stages all B rows in one call (the scale is global): got b=%d B=%d row_offset=%d", b, B,
             row_offset);
  MC_REQUIRE(aligned(planes_all, 256), MC_ERR_ALIGN, "clip_prepare: planes buffer must be 256-byte aligned");
  PlanesLayout l = planes_layout(B, D);
  char* base = static_cast<char*>(planes_all);
  __half* Xh = reinterpret_cast<__half*>(base + l.off_hi);
  __half* Xl = reinterpret_cast<__half*>(base + l.off_lo);
  __half* XhT = reinterpret_cast<__half*>(base + l.off_hiT);
  float* hdr = reinterpret_cast<float*>(base + l.off_hdr);
  float* norm_i = reinterpret_cast<float*>(base + l.off_norm_i);
  float* norm_t = reinterpret_cast<float*>(base + l.off_norm_t);
  MC_CUDA(cudaMemsetAsync(hdr, 0, 16, st));
  const size_t n = (size_t)B * D;
  int ab = (int)((n + 255) / 256);
  if (ab > num_sms() * 8) ab = num_sms() * 8;
  amax_kernel<<<ab, 256, 0, st>>>(I_loc, T_loc, n, reinterpret_cast<unsigned int*>(hdr));
  MC_LAUNCH_CHECK();
  PeerRows src;
  for (int q = 0; q < kMaxPeers; ++q) { src.I[q] = nullptr; src.T[q] = nullptr; }
  src.I[0] = I_loc;
  src.T[0] = T_loc;
  MC_REQUIRE(aligned(I_loc, 16) && aligned(T_loc, 16), MC_ERR_ALIGN, "clip_prepare: embeddings must be 16-byte aligned");
  launch_stage_fused(src, B, B, D, l, reinterpret_cast<const unsigned int*>(hdr), 1, Xh, Xl, XhT, hdr, norm_i, norm_t, st);
  MC_LAUNCH_CHECK();
  return MC_OK;
}

template <int PHASE, int PASSES>
static int launch_pair(const ClipProblem& p, const ClipStatsAll& s, const float* ps_loc, float* part,
                       const float* wscale, cudaStream_t st, float* colpart = nullptr, int chunk_k = -1, int chunks = 1,
                       __half* wout = nullptr) {
  MC_REQUIRE(supported(p.D), MC_ERR_UNSUPPORTED, "tcgen05 engine needs D in {128, 256} (got %d)", p.D);
  MC_REQUIRE(p.row_offset % 128 == 0, MC_ERR_UNSUPPORTED, "tcgen05 engine needs row_offset %% 128 == 0 (got %d)",
             p.row_offset);
  MC_REQUIRE(p.planes_all != nullptr && aligned(p.planes_all, 256), MC_ERR_BAD_ARG,
             "tcgen05 engine: planes buffer missing or not 256-byte aligned (call mc_clip_prepare first)");
  PlanesLayout l = planes_layout(p.B, p.D);
  const char* base = static_cast<const char*>(p.planes_all);
  const void* Xh = base + l.off_hi;
  const void* Xl = base + l.off_lo;
  const void* XhT = base + l.off_hiT;
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo, mt;
  int rc;
  if ((rc = make_map(&ma_hi, Xh, l.Bp, 2 * p.D, 64))) return rc;
  if ((rc = make_map(&ma_lo, Xl, l.Bp, 2 * p.D, 64))) return rc;
  if ((rc = make_map(&mb_hi, Xh, l.Bp, 2 * p.D, 32))) return rc;
  if ((rc = make_map(&mb_lo, Xl, l.Bp, 2 * p.D, 32))) return rc;
  if ((rc = make_map(&mt, XhT, 2 * p.D, l.Bp, p.D / 2))) return rc;

  const bool chunked = chunks > 1 && (PHASE == kStats || PHASE == kStatsZ);
  Split sp = choose_split(p.b, p.B, phase_ovh<PHASE>(), chunked ? chunks : 1);
  if (PHASE == kBwdP) { sp.nsplit = 1; sp.tiles_per_split = sp.n_tiles; }   // a handful of flagged tiles per row block
  PairParams pp;
  pp.b = p.b; pp.B = p.B; pp.Bp = l.Bp; pp.D = p.D; pp.row_offset = p.row_offset;
  pp.n_row_blocks = sp.n_row_blocks; pp.n_tiles = sp.n_tiles; pp.nsplit = sp.nsplit;
  pp.tiles_per_split = sp.tiles_per_split; pp.bpad = sp.bpad;
  pp.inv_tau = 1.f / p.tau; pp.half_tau = 0.5f * p.tau; pp.inv_2B = 0.5f / (float)p.B;
  pp.scale = reinterpret_cast<const float*>(base + l.off_hdr) + 1;
  pp.r = s.r; pp.c = s.c; pp.rz = s.rz; pp.g = s.g; pp.q = s.q;
  pp.ps = ps_loc;
  pp.part = part;
  pp.wscale = wscale;
  pp.flags_out = (PHASE == kStats) ? p.tile_flags_out : nullptr;
  pp.flags = (PHASE == kStatsZ) ? p.tile_flags_out : (PHASE != kStats ? p.tile_flags : nullptr);  // kStatsZ: the probe's raw flags
  pp.norm_i = reinterpret_cast<const float*>(base + l.off_norm_i);
  pp.norm_t = reinterpret_cast<const float*>(base + l.off_norm_t);
  pp.colpart = (PHASE == kStats) ? colpart : nullptr;
  pp.wout = wout;
  pp.gate = (PHASE == kBwd || PHASE == kBwdW || PHASE == kBwdP) ? p.gate : nullptr;
  pp.gate_want = PHASE == kBwd ? 0 : 1;
  pp.chunk_k = (PHASE == kStats && chunked) ? chunk_k : -1;
  pp.chunk_blocks = chunked ? sp.n_row_blocks / chunks : sp.n_row_blocks;
  pp.chunk_m = chunked ? sp.nsplit / chunks : sp.nsplit;
  if (chunked)
    MC_REQUIRE(sp.n_row_blocks % chunks == 0 && sp.nsplit % chunks == 0 && sp.n_tiles % sp.nsplit == 0 &&
                   sp.n_tiles == sp.n_row_blocks,
               MC_ERR_UNSUPPORTED, "chunked statistics sweep: %d row blocks / %d splits do not divide into %d chunks",
               sp.n_row_blocks, sp.nsplit, chunks);

  auto kern = pair_kernel<PHASE, PASSES>;
  static std::atomic<unsigned long long> attr_done{0};  // per template instantiation, one bit per device
  MC_CUDA(ensure_dynamic_smem(kern, kSmemBytes, attr_done));
  long njobs = (long)sp.n_row_blocks * sp.nsplit;
  if (pp.chunk_k >= 0) njobs = (long)pp.chunk_blocks * (pp.chunk_k + 1) * pp.chunk_m + (long)pp.chunk_k * pp.chunk_blocks * pp.chunk_m;
  int npairs = num_sms() / 2;
  if (njobs < npairs) npairs = (int)njobs;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * npairs);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  MC_CUDA(cudaLaunchKernelEx(&cfg, kern, ma_hi, ma_lo, mb_hi, mb_lo, mt, pp));
  count_launch();
  return MC_OK;
}

template <int PHASE>
static int launch_phase(int mode, const ClipProblem& p, const ClipStatsAll& s, const float* ps_loc, float* part,
                        const float* wscale, cudaStream_t st, float* colpart = nullptr, int chunk_k = -1, int chunks = 1,
                        __half* wout = nullptr) {
  if (mode == MC_GEMM_TC_F16X3) return launch_pair<PHASE, 3>(p, s, ps_loc, part, wscale, st, colpart, chunk_k, chunks, wout);
  return launch_pair<PHASE, 1>(p, s, ps_loc, part, wscale, st, colpart, chunk_k, chunks, wout);
}

// ------------------------------------------------------------------------------------------
// tile flags: flag(I, J) = 1 when some P_ij or P_ji of the 128 x 128 tile (row block I, column tile J) may exceed
// 2^-44.  The statistics sweep decides the row side for its own row blocks; the column side of (I, J) is the row
// side of (J, I) (Z is symmetric), which belongs to whoever owns row block J - hence the gather + transpose here.
// ------------------------------------------------------------------------------------------
size_t tile_flags_bytes(int b, int B) {
  Split s = choose_split(b, B);
  return (size_t)s.n_row_blocks * s.n_tiles;
}

// flags_all: [n_tiles][n_tiles] (all row blocks of the global batch), flags_loc: [own row blocks][n_tiles]
__global__ void __launch_bounds__(256) flags_finalize_kernel(const uint8_t* __restrict__ flags_all, int n_tiles, int rb0,
                                                             int nrb_loc, uint8_t* __restrict__ flags_loc) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= nrb_loc * n_tiles) return;
  const int il = idx / n_tiles, j = idx - il * n_tiles, ig = rb0 + il;
  flags_loc[idx] = (flags_all[(size_t)ig * n_tiles + j] | flags_all[(size_t)j * n_tiles + ig]) ? 1 : 0;
}

int flags_finalize(const uint8_t* flags_all, int B, int b, int row_offset, uint8_t* flags_loc, cudaStream_t st) {
  MC_REQUIRE(row_offset % 128 == 0, MC_ERR_UNSUPPORTED, "clip_flags_finalize: row_offset %% 128 != 0");
  Split s = choose_split(b, B);
  const int total = s.n_row_blocks * s.n_tiles;
  flags_finalize_kernel<<<(total + 255) / 256, 256, 0, st>>>(flags_all, s.n_tiles, row_offset / 128, s.n_row_blocks,
                                                             flags_loc);
  MC_LAUNCH_CHECK();
  return MC_OK;
}

// c_part_all (optional, B floats): the column-partials form under row sharding - receives LSE_{i in the owned rows} S_ij
// for EVERY column j (natural log); c_loc is then not written and the caller merges the ranks' vectors (ranks_lse_merge).
// chunks > 1 (b == B only): the probe sweep is launched once per arrived row chunk (stats_chunk), see PairParams.
static float* stats_colpart_ptr(const ClipProblem& p, int mode, void* ws, float* c_part_all) {
  if (c_part_all)
    return reinterpret_cast<float*>(static_cast<char*>(ws) + core_workspace_bytes(p.b, p.B, p.D, mode) - colpart_bytes(p.b, p.B));
  return use_colpart(p.b, p.B) ? colpart_slot(ws, p.b, p.B, p.D) : nullptr;
}
// ---- statistics sweep on rowsweep_kernel (probe form with column partials, 3-pass engine, from 4096 x 4096 logits on)
static bool rowsweep_ok(const ClipProblem& p, int mode, const float* colpart, int chunks) {
  static const bool off = getenv("MAE_CLIP_STATS_ROWSWEEP") != nullptr && getenv("MAE_CLIP_STATS_ROWSWEEP")[0] == '0';
  if (off || (mode != MC_GEMM_TC_F16X3 && mode != MC_GEMM_TC_F16) || colpart == nullptr || p.tile_flags_out == nullptr) return false;
  if ((double)p.b * (double)p.B < 4096.0 * 4096.0 || p.row_offset % 128 != 0) return false;
  if (chunks > 1) {
    Split s = choose_split_rows256(p.b, p.B, chunks, 2.0);
    if (s.n_row_blocks % chunks != 0 || s.nsplit % chunks != 0 || s.n_tiles % s.nsplit != 0 || p.b != p.B) return false;
  }
  return true;
}
static float2* rowsweep_part(const ClipProblem& p, void* ws) {
  Split s = choose_split(p.b, p.B, kOvhStats);
  return reinterpret_cast<float2*>(static_cast<char*>(ws) + (size_t)kMaxSplit * 4 * s.bpad * sizeof(float2));
}
static float* rowsweep_tile_min(const ClipProblem& p, void* ws) {
  return reinterpret_cast<float*>(reinterpret_cast<char*>(rowsweep_part(p, ws)) +
                                  round_up((size_t)kMaxSplit * round_up((size_t)p.b, 256) * sizeof(float2), 256));
}
static float* rowsweep_tile_max_rho(const ClipProblem& p, void* ws) {
  return rowsweep_tile_min(p, ws) + round_up((size_t)p.B, 128) / 128;
}
static float* rowsweep_tile_max_n(const ClipProblem& p, void* ws) {
  return rowsweep_tile_max_rho(p, ws) + round_up((size_t)p.B, 128) / 128;
}
static int* rowsweep_probe_gate(const ClipProblem& p, void* ws) {
  return reinterpret_cast<int*>(rowsweep_tile_max_n(p, ws) + round_up((size_t)p.B, 128) / 128);
}
// full_reprobe (kRsZ): every K chunk multiplied out, gated on the device by probe_gate_kernel's verdict
template <int KIND, int PASSES>
static int launch_rowsweep(const ClipProblem& p, void* ws, float* colpart, int chunk_k, int chunks, cudaStream_t st,
                           bool full_reprobe = false) {
  PlanesLayout l = planes_layout(p.B, p.D);
  const char* base = static_cast<const char*>(p.planes_all);
  const void* Xh = base + l.off_hi;
  const void* Xl = base + l.off_lo;
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
  int rc;
  if ((rc = make_map(&ma_hi, Xh, l.Bp, 2 * p.D, 128))) return rc;
  if ((rc = make_map(&ma_lo, Xl, l.Bp, 2 * p.D, 128))) return rc;
  if ((rc = make_map(&mb_hi, Xh, l.Bp, 2 * p.D, 64))) return rc;
  if ((rc = make_map(&mb_lo, Xl, l.Bp, 2 * p.D, 64))) return rc;
  const bool chunked = chunks > 1;
  Split sp = choose_split_rows256(p.b, p.B, chunked ? chunks : 1, 2.0);
  RowSweepParams rp;
  rp.b = p.b; rp.B = p.B; rp.Bp = l.Bp; rp.D = p.D; rp.row_offset = p.row_offset;
  rp.n_row_blocks = sp.n_row_blocks; rp.n_tiles = sp.n_tiles; rp.nsplit = sp.nsplit;
  rp.tiles_per_split = sp.tiles_per_split; rp.bpad = sp.bpad;
  rp.chunk_k = chunked ? chunk_k : -1;
  rp.chunk_blocks = chunked ? sp.n_row_blocks / chunks : sp.n_row_blocks;
  rp.chunk_m = chunked ? sp.nsplit / chunks : sp.nsplit;
  rp.tri = (p.b == p.B && p.row_offset == 0) ? 1 : 0;
  rp.inv_tau = 1.f / p.tau; rp.half_tau = 0.5f * p.tau;
  rp.scale = reinterpret_cast<const float*>(base + l.off_hdr) + 1;
  rp.part = rowsweep_part(p, ws);
  rp.colpart = colpart;
  rp.flags_out = p.tile_flags_out;
  rp.norm_i = reinterpret_cast<const float*>(base + l.off_norm_i);
  rp.norm_t = reinterpret_cast<const float*>(base + l.off_norm_t);
  rp.tile_min_zjj2 = rowsweep_tile_min(p, ws);
  rp.pk = full_reprobe ? p.D / 64 : probe_chunks(p.D);
  rp.rho = rp.pk < p.D / 64 ? reinterpret_cast<const float*>(base + l.off_rho) : nullptr;
  rp.tile_max_rho = rowsweep_tile_max_rho(p, ws);
  rp.tile_max_n = rowsweep_tile_max_n(p, ws);
  // gate words: [0] probe_gate_kernel's verdict (1 = re-probe in full), [1] probe_hopeless_kernel's (1 = skip the partial probe)
  rp.gate = full_reprobe ? rowsweep_probe_gate(p, ws) : (rp.rho != nullptr ? rowsweep_probe_gate(p, ws) + 1 : nullptr);
  rp.gate_want = full_reprobe ? 1 : 0;
  auto kern = rowsweep_kernel<KIND, PASSES>;
  static std::atomic<unsigned long long> attr_done{0};
  MC_CUDA(ensure_dynamic_smem(kern, kRsSmemBytes, attr_done));
  long njobs = (long)sp.n_row_blocks * sp.nsplit;
  if (rp.chunk_k >= 0) njobs = (long)rp.chunk_blocks * (rp.chunk_k + 1) * rp.chunk_m + (long)rp.chunk_k * rp.chunk_blocks * rp.chunk_m;
  int npairs = num_sms() / 2;
  if (njobs < npairs) npairs = (int)njobs;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * npairs);
  cfg.blockDim = dim3(kRsThreads);
  cfg.dynamicSmemBytes = kRsSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  MC_CUDA(cudaLaunchKernelEx(&cfg, kern, ma_hi, ma_lo, mb_hi, mb_lo, rp));
  count_launch();
  return MC_OK;
}

int stats_begin(const ClipProblem& p, cudaStream_t st) {
  if (p.tile_flags_out) MC_CUDA(cudaMemsetAsync(p.tile_flags_out, 0, tile_flags_bytes(p.b, p.B), st));
  return MC_OK;
}
int stats_chunk(const ClipProblem& p, int mode, int k, int chunks, void* ws, cudaStream_t st, float* c_part_all) {
  ClipStatsAll none{nullptr, nullptr, nullptr, nullptr, nullptr};
  float* colpart_rs = stats_colpart_ptr(p, mode, ws, c_part_all);
  if (rowsweep_ok(p, mode, colpart_rs, chunks)) {
    // S statistics and the Z probe as two launches of rowsweep_kernel (large MMA shapes); the per-tile minima of Z_jj are
    // recomputed at every arrival (the norms of a chunk's rows exist once it is staged)
    PlanesLayout l = planes_layout(p.B, p.D);
    const char* base = static_cast<const char*>(p.planes_all);
    const int n_tiles = (int)(round_up((size_t)p.B, 128) / 128);
    tile_min_zjj_kernel<<<n_tiles, 128, 0, st>>>(reinterpret_cast<const float*>(base + l.off_norm_i),
                                                 reinterpret_cast<const float*>(base + l.off_norm_t),
                                                 reinterpret_cast<const float*>(base + l.off_rho), p.B, 0.5f * p.tau,
                                                 rowsweep_tile_min(p, ws), rowsweep_tile_max_rho(p, ws), rowsweep_tile_max_n(p, ws));
    MC_LAUNCH_CHECK();
    if (probe_chunks(p.D) < p.D / 64) {
      if (k <= 0) MC_CUDA(cudaMemsetAsync(rowsweep_probe_gate(p, ws), 0, 2 * sizeof(int), st));   // first launch of this sweep
      const int n_valid = chunks > 1 ? (int)((long)n_tiles * (k + 1) / chunks) : n_tiles;
      probe_hopeless_kernel<<<1, 256, 0, st>>>(rowsweep_tile_min(p, ws), rowsweep_tile_max_rho(p, ws), n_valid, 0.5f * p.tau,
                                               rowsweep_probe_gate(p, ws) + 1);
      MC_LAUNCH_CHECK();
    }
    int rc = mode == MC_GEMM_TC_F16X3 ? launch_rowsweep<kRsS, 3>(p, ws, colpart_rs, k, chunks, st)
                                      : launch_rowsweep<kRsS, 1>(p, ws, colpart_rs, k, chunks, st);
    if (rc) return rc;
    return launch_rowsweep<kRsZ, 3>(p, ws, colpart_rs, k, chunks, st);   // the probe reads the hi planes only in either engine
  }
  return launch_phase<kStats>(mode, p, none, nullptr, static_cast<float*>(ws), nullptr, st,
                              stats_colpart_ptr(p, mode, ws, c_part_all), k, chunks);
}
int stats_end(const ClipProblem& p, int mode, int chunks, float* r_loc, float* c_loc, float* rz_loc, float* ps_loc, void* ws,
              cudaStream_t st, float* c_part_all) {
  ClipStatsAll none{nullptr, nullptr, nullptr, nullptr, nullptr};
  float* colpart = stats_colpart_ptr(p, mode, ws, c_part_all);
  if (c_part_all) c_loc = c_part_all;
  int rc;
  // a partial probe (probe_chunks) whose bound was too loose for this batch flags far more tiles than a concentrated
  // batch has: the device decides, clears the bitmap and re-probes with every K chunk (both launches are always enqueued)
  if (rowsweep_ok(p, mode, colpart, chunks) && probe_chunks(p.D) < p.D / 64) {
    const int nflag = (int)tile_flags_bytes(p.b, p.B);
    probe_gate_kernel<<<1, 1024, 0, st>>>(p.tile_flags_out, nflag, (p.b + 127) / 128 + nflag / 64, rowsweep_probe_gate(p, ws));
    MC_LAUNCH_CHECK();
    if ((rc = launch_rowsweep<kRsZ, 3>(p, ws, colpart, -1, 1, st, true))) return rc;
  }
  // with tile flags the sweep above was the probe form (S exact, Z from the hi planes -> flags); the exact Z and
  // sum_j P_ij S_ij follow on the flagged tiles only
  if (p.tile_flags_out &&
      (rc = launch_phase<kStatsZ>(mode, p, none, nullptr, static_cast<float*>(ws), nullptr, st, nullptr, -1, chunks)))
    return rc;
  Split sp = choose_split(p.b, p.B, kOvhStats, chunks);
  const bool rs = rowsweep_ok(p, mode, colpart, chunks);
  int col_groups = sp.bpad / 32;
  if (rs) {   // r comes from rowsweep_kernel<kRsS>'s own partials (row blocks of 256, its own split)
    Split sr = choose_split_rows256(p.b, p.B, chunks > 1 ? chunks : 1, 2.0);
    rowsweep_finalize_kernel<<<(p.b + 255) / 256, 256, 0, st>>>(rowsweep_part(p, ws), sr.nsplit, sr.bpad, p.b, r_loc);
    MC_LAUNCH_CHECK();
    col_groups = sr.bpad / 32;
  }
  stats_finalize_kernel<<<(p.b + 255) / 256, 256, 0, st>>>(static_cast<const float2*>(ws), sp.nsplit, sp.bpad, p.b,
                                                          rs ? nullptr : r_loc, colpart ? nullptr : c_loc, rz_loc, ps_loc);
  MC_LAUNCH_CHECK();
  if (colpart) {
    // rows b .. bpad of the last row block wrote -inf partials; c_loc has B entries here (every column, over the owned rows)
    const int Bp = (int)round_up((size_t)p.B, 128);
    colpart_merge_kernel<<<(p.B + 63) / 64, 256, 0, st>>>(colpart, col_groups, Bp, p.B, c_loc);
    MC_LAUNCH_CHECK();
  }
  return MC_OK;
}
int stats(const ClipProblem& p, int mode, float* r_loc, float* c_loc, float* rz_loc, float* ps_loc, void* ws,
          size_t ws_bytes, cudaStream_t st, float* c_part_all) {
  const size_t need = c_part_all ? stats_colpart_workspace_bytes(p.b, p.B, p.D, mode) : core_workspace_bytes(p.b, p.B, p.D, mode);
  MC_REQUIRE(ws_bytes >= need, MC_ERR_WORKSPACE, "clip_stats(tc): workspace %zu < %zu", ws_bytes, need);
  int rc;
  if ((rc = stats_begin(p, st))) return rc;
  if ((rc = stats_chunk(p, mode, -1, 1, ws, st, c_part_all))) return rc;
  return stats_end(p, mode, 1, r_loc, c_loc, rz_loc, ps_loc, ws, st, c_part_all);
}

// ---- chunked staging (host-buffer entry): rows [row0, row0 + rows) of a batch that is still arriving.  The planes share
// ONE power-of-two scale, so the first chunk fixes it with a binade of headroom (slot = 2 max|chunk 0|) and every chunk
// adds to the true maximum; verify_scale() afterwards flags the (rare) batch whose later rows exceed the headroom - the
// caller then redoes the step the plain way.  The bound the tile-flag probe relies on (|x| s < 2) holds whenever the
// flag is clear.
__global__ void scale_slot_kernel(const unsigned int* __restrict__ true_bits, unsigned int* __restrict__ slot) {
  const float a = __uint_as_float(*true_bits);
  *slot = __float_as_uint(a > 0.f && a < INFINITY ? 2.f * a : 0.f);
}
__global__ void scale_verify_kernel(const unsigned int* __restrict__ true_bits, const unsigned int* __restrict__ slot,
                                    int* __restrict__ bad) {
  *bad = (__uint_as_float(*true_bits) > __uint_as_float(*slot)) ? 1 : 0;
}
int prepare_chunk(const float* I, const float* T, int B, int D, int row0, int rows, void* planes_all, unsigned int* words,
                  cudaStream_t st) {
  // words: [0] true max so far (zeroed by the caller before the first chunk), [1] the scale slot, [2] the "bad" flag
  MC_REQUIRE(supported(D) && row0 % 32 == 0 && rows % 32 == 0 && row0 + rows <= (int)round_up((size_t)B, 128), MC_ERR_UNSUPPORTED,
             "clip_prepare_chunk: D %d / rows [%d, +%d) not supported", D, row0, rows);
  MC_REQUIRE(aligned(I, 16) && aligned(T, 16) && aligned(planes_all, 256), MC_ERR_ALIGN, "clip_prepare_chunk: alignment");
  PlanesLayout l = planes_layout(B, D);
  char* base = static_cast<char*>(planes_all);
  const int real_rows = row0 + rows <= B ? rows : (B > row0 ? B - row0 : 0);
  if (real_rows > 0) {
    const size_t n = (size_t)real_rows * D;
    int ab = (int)((n + 255) / 256);
    if (ab > num_sms() * 8) ab = num_sms() * 8;
    amax_kernel<<<ab, 256, 0, st>>>(I + (size_t)row0 * D, T + (size_t)row0 * D, n, words);
    MC_LAUNCH_CHECK();
  }
  if (row0 == 0) {
    scale_slot_kernel<<<1, 1, 0, st>>>(words, words + 1);
    MC_LAUNCH_CHECK();
  }
  PeerRows src;
  for (int q = 0; q < kMaxPeers; ++q) { src.I[q] = nullptr; src.T[q] = nullptr; }
  src.I[0] = I;
  src.T[0] = T;
  const int blocks = rows / 32, blk0 = row0 / 32;
  __half* Xh = reinterpret_cast<__half*>(base + l.off_hi);
  __half* Xl = reinterpret_cast<__half*>(base + l.off_lo);
  __half* XhT = reinterpret_cast<__half*>(base + l.off_hiT);
  float* hdr = reinterpret_cast<float*>(base + l.off_hdr);
  float* norm_i = reinterpret_cast<float*>(base + l.off_norm_i);
  float* norm_t = reinterpret_cast<float*>(base + l.off_norm_t);
  if (D == 256)
    stage_fused_kernel<256><<<blocks, 256, 0, st>>>(src, B, B, l.Bp, words + 1, 1, Xh, Xl, XhT, hdr, norm_i, norm_t, blk0,
                                                    norm_i + (l.off_rho - l.off_norm_i) / 4, 16 * probe_chunks(D));
  else
    stage_fused_kernel<128><<<blocks, 256, 0, st>>>(src, B, B, l.Bp, words + 1, 1, Xh, Xl, XhT, hdr, norm_i, norm_t, blk0,
                                                    norm_i + (l.off_rho - l.off_norm_i) / 4, 16 * probe_chunks(D));
  MC_LAUNCH_CHECK();
  return MC_OK;
}
int verify_scale(unsigned int* words, cudaStream_t st) {
  scale_verify_kernel<<<1, 1, 0, st>>>(words, words + 1, reinterpret_cast<int*>(words + 2));
  MC_LAUNCH_CHECK();
  return MC_OK;
}

int rowloss(const ClipProblem& p, int mode, const ClipStatsAll& s, const float* ps_loc, float* g_loc, float* q_loc,
            float* loss_part, void* ws, size_t ws_bytes, cudaStream_t st) {
  MC_REQUIRE(ws_bytes >= core_workspace_bytes(p.b, p.B, p.D, mode), MC_ERR_WORKSPACE, "clip_rowloss(tc): workspace too small");
  int rc = launch_phase<kRowLoss>(mode, p, s, ps_loc, static_cast<float*>(ws), nullptr, st);
  if (rc) return rc;
  Split sp = choose_split(p.b, p.B, kOvhRowLoss);
  rowloss_finalize_kernel<<<(p.b + 255) / 256, 256, 0, st>>>(static_cast<const float*>(ws), sp.nsplit, sp.bpad, p.b,
                                                            0.5f / (float)p.B, s.r + p.row_offset, ps_loc, g_loc, q_loc);
  MC_LAUNCH_CHECK();
  sum_kernel<<<1, 1024, 0, st>>>(g_loc, p.b, loss_part);
  MC_LAUNCH_CHECK();
  return MC_OK;
}

int bwd(const ClipProblem& p, int mode, const ClipStatsAll& s, const float* grad_loss, float* dI, float* dT, void* ws,
        size_t ws_bytes, cudaStream_t st) {
  const bool use_stored = p.b == p.B && p.row_offset == 0 && stored_form_enabled(p.b, p.B, p.D) && p.tile_flags != nullptr &&
                          (mode == MC_GEMM_TC_F16X3 || mode == MC_GEMM_TC_F16);
  MC_REQUIRE(ws_bytes >= (use_stored ? workspace_bytes(p.b, p.B, p.D, mode) : core_workspace_bytes(p.b, p.B, p.D, mode)),
             MC_ERR_WORKSPACE, "clip_bwd(tc): workspace too small");
  MC_REQUIRE(aligned(dI, 16) && aligned(dT, 16), MC_ERR_ALIGN, "clip_bwd(tc): gradients must be 16-byte aligned");
  MC_REQUIRE(p.planes_all != nullptr, MC_ERR_BAD_ARG, "clip_bwd(tc): planes buffer missing");
  if (use_stored) {
    // a call that owns every row and has tile flags: the stored-weights form (row half + column half) while the soft
    // targets are concentrated, the own-rows sweep otherwise - decided on the device from the flag density
    StoredLayout sl = stored_layout(p.B, p.D, mode);
    char* base = static_cast<char*>(ws);
    ClipProblem pg = p;
    int* gate = reinterpret_cast<int*>(wscale_slot(ws, p.b, p.B, p.D) + 16);
    int rc = bwd_gate(p.tile_flags, tile_flags_bytes(p.b, p.B), gate, st);
    if (rc) return rc;
    pg.gate = gate;
    rc = bwd_rows(pg, mode, s, grad_loss, dT, reinterpret_cast<float*>(base + sl.off_diz), base + sl.off_w, ws, sl.off_w, st, dI);
    if (rc) return rc;
    return bwd_cols(pg, mode, s, grad_loss, base + sl.off_w, p.B, 0, 0, p.B, reinterpret_cast<const float*>(base + sl.off_diz), dI,
                    base + sl.off_cols, sl.cols_bytes, st, wscale_slot(ws, p.b, p.B, p.D));
  }
  PlanesLayout l = planes_layout(p.B, p.D);
  const char* pbase = static_cast<const char*>(p.planes_all);
  float* wsc = wscale_slot(ws, p.b, p.B, p.D);
  wscale_kernel<<<1, 1024, 0, st>>>(s.r, s.c, s.rz, s.q, p.B, reinterpret_cast<const float*>(pbase + l.off_hdr) + 1,
                                   reinterpret_cast<const float*>(pbase + l.off_norm_i),
                                   reinterpret_cast<const float*>(pbase + l.off_norm_t), 1.f / p.tau, p.tau, wsc);
  MC_LAUNCH_CHECK();
  int rc = launch_phase<kBwd>(mode, p, s, nullptr, static_cast<float*>(ws), wsc, st);
  if (rc) return rc;
  Split sp = choose_split(p.b, p.B, kOvhBwd);
  size_t n4 = (size_t)p.b * p.D / 4;
  int blocks = (int)((n4 + 255) / 256);
  int cap = num_sms() * 8;
  if (blocks > cap) blocks = cap;
  bwd_finalize_kernel<<<blocks, 256, 0, st>>>(static_cast<const float*>(ws), sp.nsplit, sp.bpad, p.b, p.D,
                                              0.5f / (float)p.B, grad_loss, wsc, dT, dI);
  MC_LAUNCH_CHECK();
  return MC_OK;
}

// ---- stored-weights gradient (see kBwdW / colgrad_kernel) -------------------------------------------------
static int launch_wscale(const ClipProblem& p, const ClipStatsAll& s, float* wsc, cudaStream_t st) {
  PlanesLayout l = planes_layout(p.B, p.D);
  const char* pbase = static_cast<const char*>(p.planes_all);
  wscale_kernel<<<1, 1024, 0, st>>>(s.r, s.c, s.rz, s.q, p.B, reinterpret_cast<const float*>(pbase + l.off_hdr) + 1,
                                   reinterpret_cast<const float*>(pbase + l.off_norm_i),
                                   reinterpret_cast<const float*>(pbase + l.off_norm_t), 1.f / p.tau, p.tau, wsc);
  MC_LAUNCH_CHECK();
  return MC_OK;
}
struct ColSplit { int n_jblocks, steps, ksplit, steps_per_split; };
static ColSplit choose_col_split(int w_rows, int n_cols) {
  ColSplit c;
  c.n_jblocks = (n_cols + 255) / 256;
  c.steps = (w_rows + 63) / 64;
  const int npairs = num_sms() / 2;
  int best = 1;
  double best_cost = 1e30;
  for (int k = 1; k <= kCgMaxSplit && k <= c.steps; ++k) {
    const int per = (c.steps + k - 1) / k;
    const long jobs = (long)c.n_jblocks * k;
    const double cost = (double)((jobs + npairs - 1) / npairs) * (per + 16.0) + 4.0 * k;   // + the partial each split adds
    if (cost < best_cost - 1e-9) { best_cost = cost; best = k; }
  }
  c.ksplit = best;
  c.steps_per_split = (c.steps + best - 1) / best;
  return c;
}
const float* bwd_rows_wscale(void* ws, int b, int B, int D) { return wscale_slot(ws, b, B, D); }
size_t stored_weights_bytes(int b, int B) { return round_up(round_up((size_t)b, 256) * round_up((size_t)B, 128) * sizeof(__half), 256); }
size_t bwd_cols_workspace_bytes(int /*w_rows*/, int n_cols, int D) {
  return round_up((size_t)kCgMaxSplit * ((size_t)(n_cols + 255) / 256 * 256) * D * sizeof(float), 256) + 256;
}
StoredLayout stored_layout(int B, int D, int mode) {
  StoredLayout l;
  l.off_w = round_up(core_workspace_bytes(B, B, D, mode), 1024);
  l.off_diz = l.off_w + stored_weights_bytes(B, B);
  l.off_cols = l.off_diz + round_up(round_up((size_t)B, 128) * D * sizeof(float), 256);
  l.cols_bytes = bwd_cols_workspace_bytes(B, B, D);
  l.total = l.off_cols + l.cols_bytes;
  return l;
}
size_t workspace_bytes(int b, int B, int D, int mode) {
  if (b == B && stored_form_enabled(b, B, D)) return stored_layout(B, D, mode).total;
  return core_workspace_bytes(b, B, D, mode);
}
bool stored_form_enabled(int b, int B, int D) {
  static const bool off = getenv("MAE_CLIP_BWD_FORM") != nullptr && strcmp(getenv("MAE_CLIP_BWD_FORM"), "ownrows") == 0;
  // small problems are launch-bound: the own-rows sweep is one kernel + one fold (C2's B = 1024: 0.18 ms against 0.25 ms for
  // the ten launches of the stored form); from 4096 x 4096 logits on the saved tensor work dominates
  return !off && supported(D) && (double)b * (double)B >= 4096.0 * 4096.0 && stored_weights_bytes(b, B) <= ((size_t)16 << 30);
}

static int launch_rowgrad(const ClipProblem& p, int mode, const ClipStatsAll& s, float* part, const float* wscale,
                          __half* wout, cudaStream_t st) {
  MC_REQUIRE(p.row_offset % 128 == 0, MC_ERR_UNSUPPORTED, "rowgrad: row_offset %% 128 != 0 (%d)", p.row_offset);
  PlanesLayout l = planes_layout(p.B, p.D);
  const char* base = static_cast<const char*>(p.planes_all);
  const void* Xh = base + l.off_hi;
  const void* Xl = base + l.off_lo;
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo, mt;
  int rc;
  if ((rc = make_map(&ma_hi, Xh, l.Bp, 2 * p.D, 128))) return rc;
  if ((rc = make_map(&ma_lo, Xl, l.Bp, 2 * p.D, 128))) return rc;
  if ((rc = make_map(&mb_hi, Xh, l.Bp, 2 * p.D, 64))) return rc;
  if ((rc = make_map(&mb_lo, Xl, l.Bp, 2 * p.D, 64))) return rc;
  if ((rc = make_map(&mt, base + l.off_hiT, 2 * p.D, l.Bp, p.D / 2))) return rc;
  Split sp = choose_split_rows256(p.b, p.B);
  RowGradParams rp;
  rp.b = p.b; rp.B = p.B; rp.Bp = l.Bp; rp.D = p.D; rp.row_offset = p.row_offset;
  rp.n_row_blocks = sp.n_row_blocks; rp.n_tiles = sp.n_tiles; rp.nsplit = sp.nsplit;
  rp.tiles_per_split = sp.tiles_per_split; rp.bpad = sp.bpad;
  rp.inv_tau = 1.f / p.tau;
  rp.scale = reinterpret_cast<const float*>(base + l.off_hdr) + 1;
  rp.r = s.r; rp.c = s.c; rp.q = s.q;
  rp.wscale = wscale;
  rp.part = part;
  rp.wout = wout;
  rp.gate = p.gate;
  const bool three = mode == MC_GEMM_TC_F16X3;
  static std::atomic<unsigned long long> attr_done3{0}, attr_done1{0};
  if (three) MC_CUDA(ensure_dynamic_smem(rowgrad_kernel<3>, kRgSmemBytes, attr_done3));
  else MC_CUDA(ensure_dynamic_smem(rowgrad_kernel<1>, kRgSmemBytes, attr_done1));
  const long njobs = (long)sp.n_row_blocks * sp.nsplit;
  int npairs = num_sms() / 2;
  if (njobs < npairs) npairs = (int)njobs;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * npairs);
  cfg.blockDim = dim3(kRgThreads);
  cfg.dynamicSmemBytes = kRgSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (three) MC_CUDA(cudaLaunchKernelEx(&cfg, rowgrad_kernel<3>, ma_hi, ma_lo, mb_hi, mb_lo, mt, rp));
  else MC_CUDA(cudaLaunchKernelEx(&cfg, rowgrad_kernel<1>, ma_hi, ma_lo, mb_hi, mb_lo, mt, rp));
  count_launch();
  return MC_OK;
}

// Row half over the strip p.row_offset .. + p.b: dT_loc (final), dIz_loc (b x D, un-scaled soft-target part of dI of the
// strip's rows) and the strip's rows of W (pointer to the strip's first row, row pitch Bp).
// 1 = concentrated soft targets (few flagged tiles): the stored-weights / split form pays; 0 = own-rows sweep
__global__ void __launch_bounds__(1024) bwd_gate_kernel(const uint8_t* __restrict__ flags, size_t n, float thresh, int* __restrict__ gate) {
  __shared__ unsigned int sm[32];
  unsigned int cnt = 0;
  size_t i0 = 0;
  if ((reinterpret_cast<uintptr_t>(flags) & 15) == 0) {   // 16 flags per load
    const size_t n16 = n >> 4;
    for (size_t i = threadIdx.x; i < n16; i += blockDim.x) {
      const uint4 v = reinterpret_cast<const uint4*>(flags)[i];
      cnt += (__popc(__vcmpne4(v.x, 0u)) + __popc(__vcmpne4(v.y, 0u)) + __popc(__vcmpne4(v.z, 0u)) + __popc(__vcmpne4(v.w, 0u))) >> 3;
    }
    i0 = n16 << 4;
  }
  for (size_t i = i0 + threadIdx.x; i < n; i += blockDim.x) cnt += flags[i] != 0;
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = cnt;
  __syncthreads();
  if (threadIdx.x < 32) {
    cnt = sm[threadIdx.x];
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (threadIdx.x == 0) *gate = ((float)cnt <= thresh * (float)n) ? 1 : 0;
  }
}
int bwd_gate(const uint8_t* flags, size_t n_flags, int* gate_out, cudaStream_t st) {
  // break-even of the two forms (DESIGN 4.1): the split form executes 5 + 16 d GEMM units, the flagged part at about half
  // the efficiency of the dense kernels; the own-rows sweep 8 + 8 d
  static const float thresh = getenv("MAE_CLIP_BWD_GATE") ? (float)atof(getenv("MAE_CLIP_BWD_GATE")) : 0.15f;
  bwd_gate_kernel<<<1, 1024, 0, st>>>(flags, n_flags, thresh, gate_out);
  MC_LAUNCH_CHECK();
  return MC_OK;
}

int bwd_rows(const ClipProblem& p, int mode, const ClipStatsAll& s, const float* grad_loss, float* dT_loc, float* dIz_loc,
             void* W_rows, void* ws, size_t ws_bytes, cudaStream_t st, float* dI_loc_ownrows) {
  MC_REQUIRE(ws_bytes >= core_workspace_bytes(p.b, p.B, p.D, mode), MC_ERR_WORKSPACE, "clip_bwd_rows: workspace too small");
  MC_REQUIRE(aligned(dT_loc, 16) && aligned(dIz_loc, 16) && aligned(W_rows, 256), MC_ERR_ALIGN, "clip_bwd_rows: alignment");
  MC_REQUIRE(p.planes_all != nullptr, MC_ERR_BAD_ARG, "clip_bwd_rows: planes buffer missing");
  float* wsc = wscale_slot(ws, p.b, p.B, p.D);
  int rc;
  if ((rc = launch_wscale(p, s, wsc, st))) return rc;
  size_t n4 = (size_t)p.b * p.D / 4;
  int blocks = (int)((n4 + 255) / 256);
  int cap = num_sms() * 8;
  if (blocks > cap) blocks = cap;
  // With tile flags the sweep splits: rowgrad_kernel (softmax part of dS on every tile, large MMA shapes) + kBwdP
  // (soft-target part on the flagged tiles).  Without flags every tile carries soft-target mass and kBwdW does both at
  // once.  MAE_CLIP_BWD_SPLIT=0 keeps the single sweep (A/B switch).
  static const bool split_off = getenv("MAE_CLIP_BWD_SPLIT") != nullptr && getenv("MAE_CLIP_BWD_SPLIT")[0] == '0';
  if (p.tile_flags != nullptr && !split_off && (mode == MC_GEMM_TC_F16X3 || mode == MC_GEMM_TC_F16)) {
    Split sr = choose_split_rows256(p.b, p.B), sp = choose_split(p.b, p.B, kOvhBwd);
    float* part_r = static_cast<float*>(ws);
    float* part_p = reinterpret_cast<float*>(static_cast<char*>(ws) + rowgrad_part_bytes(p.b, p.B, p.D));
    const size_t plane_p = (size_t)sp.bpad * p.D;
    MC_CUDA(cudaMemsetAsync(part_p, 0, 2 * plane_p * sizeof(float), st));   // row blocks without a flagged tile write nothing
    if ((rc = launch_phase<kBwdP>(mode, p, s, nullptr, part_p, wsc, st))) return rc;
    if ((rc = launch_rowgrad(p, mode, s, part_r, wsc, static_cast<__half*>(W_rows), st))) return rc;
    bwd_rows_split_finalize_kernel<<<blocks, 256, 0, st>>>(part_r, sr.nsplit, (size_t)sr.bpad * p.D, part_p, plane_p, p.b, p.D,
                                                          0.5f / (float)p.B, grad_loss, wsc, dT_loc, dIz_loc, p.gate);
    MC_LAUNCH_CHECK();
    if (p.gate != nullptr) {
      // the own-rows sweep of the same strip, for the batches whose soft targets are NOT concentrated (gate == 0): it
      // shares the partial-sum buffer (only one of the two forms executes) and writes dT_loc and the caller's dI rows
      MC_REQUIRE(dI_loc_ownrows != nullptr && aligned(dI_loc_ownrows, 16), MC_ERR_BAD_ARG,
                 "clip_bwd_rows: a gated call needs the dI rows of the own-rows form");
      if ((rc = launch_phase<kBwd>(mode, p, s, nullptr, static_cast<float*>(ws), wsc, st))) return rc;
      bwd_finalize_kernel<<<blocks, 256, 0, st>>>(static_cast<const float*>(ws), sp.nsplit, sp.bpad, p.b, p.D,
                                                  0.5f / (float)p.B, grad_loss, wsc, dT_loc, dI_loc_ownrows, p.gate, 0);
      MC_LAUNCH_CHECK();
    }
    return MC_OK;
  }
  MC_REQUIRE(p.gate == nullptr, MC_ERR_BAD_ARG, "clip_bwd_rows: the form switch needs tile flags");
  if ((rc = launch_phase<kBwdW>(mode, p, s, nullptr, static_cast<float*>(ws), wsc, st, nullptr, -1, 1,
                                static_cast<__half*>(W_rows))))
    return rc;
  Split sp = choose_split(p.b, p.B, kOvhBwd);
  bwd_rows_finalize_kernel<<<blocks, 256, 0, st>>>(static_cast<const float*>(ws), sp.nsplit, sp.bpad, p.b, p.D,
                                                   0.5f / (float)p.B, grad_loss, wsc, dT_loc, dIz_loc);
  MC_LAUNCH_CHECK();
  return MC_OK;
}

// Column half: dI of the rows j0 .. j1 (j0 a multiple of 128) from the stored strip W (w_rows rows whose first is the
// global row w_row_offset): dI_out[j - j0] = scale (dIz[j - j0] + sum_i W_ij T_i).  dIz may be null (a rank that does
// not own those rows contributes the W part only).
int bwd_cols(const ClipProblem& p, int mode, const ClipStatsAll& s, const float* grad_loss, const void* W, int w_rows,
             int w_row_offset, int j0, int j1, const float* dIz, float* dI_out, void* ws, size_t ws_bytes, cudaStream_t st,
             const float* wscale_ready) {
  (void)mode;
  MC_REQUIRE(supported(p.D), MC_ERR_UNSUPPORTED, "clip_bwd_cols: D %d", p.D);
  MC_REQUIRE(j0 % 128 == 0 && j0 >= 0 && j1 > j0 && j1 <= p.B && w_rows > 0 && w_row_offset % 64 == 0, MC_ERR_BAD_ARG,
             "clip_bwd_cols: bad ranges (j %d..%d, rows %d at %d)", j0, j1, w_rows, w_row_offset);
  MC_REQUIRE(ws_bytes >= bwd_cols_workspace_bytes(w_rows, j1 - j0, p.D), MC_ERR_WORKSPACE, "clip_bwd_cols: workspace too small");
  MC_REQUIRE(aligned(W, 256) && aligned(dI_out, 16) && (!dIz || aligned(dIz, 16)), MC_ERR_ALIGN, "clip_bwd_cols: alignment");
  PlanesLayout l = planes_layout(p.B, p.D);
  const char* base = static_cast<const char*>(p.planes_all);
  const int w_rows_pad = (int)round_up((size_t)w_rows, 128);
  CUtensorMap mw, mt;
  int rc;
  if ((rc = make_map(&mw, W, w_rows_pad, l.Bp, 64))) return rc;
  if ((rc = make_map(&mt, base + l.off_hiT, 2 * p.D, l.Bp, p.D / 2))) return rc;
  ColSplit cs = choose_col_split(w_rows_pad, j1 - j0);
  const size_t part_bytes = round_up((size_t)kCgMaxSplit * ((size_t)cs.n_jblocks * 256) * p.D * sizeof(float), 256);
  // the power-of-two scale of the stored weights: the row half's own word when the caller still has it (same stream),
  // else recomputed from the statistics (deterministic: the same value)
  const float* wsc = wscale_ready;
  if (wsc == nullptr) {
    float* w2 = reinterpret_cast<float*>(static_cast<char*>(ws) + part_bytes);
    if ((rc = launch_wscale(p, s, w2, st))) return rc;
    wsc = w2;
  }
  ColGradParams cp;
  cp.Bp = l.Bp; cp.D = p.D; cp.w_rows = w_rows_pad; cp.row_offset = w_row_offset;
  cp.j_first = j0; cp.n_jblocks = cs.n_jblocks; cp.j_end = j1;
  cp.ksplit = cs.ksplit; cp.steps_per_split = cs.steps_per_split; cp.steps = cs.steps;
  cp.part = static_cast<float*>(ws);
  cp.gate = p.gate;
  const int smem = kCgStages * (kCgStageA + (p.D / 2) * 128) + 8 * 32 + 16 + 1024;
  // the opt-in is set once per device: ask for the largest layout (D = 256) whatever this call's width is
  const int smem_max = kCgStages * (kCgStageA + 128 * 128) + 8 * 32 + 16 + 1024;
  static std::atomic<unsigned long long> attr_done{0};
  MC_CUDA(ensure_dynamic_smem(colgrad_kernel, smem_max, attr_done));
  const long njobs = (long)cs.n_jblocks * cs.ksplit;
  int npairs = num_sms() / 2;
  if (njobs < npairs) npairs = (int)njobs;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * npairs);
  cfg.blockDim = dim3(kCgThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  MC_CUDA(cudaLaunchKernelEx(&cfg, colgrad_kernel, mw, mt, cp));
  count_launch();
  const int rows = j1 - j0;
  size_t n4 = (size_t)rows * p.D / 4;
  int blocks = (int)((n4 + 255) / 256);
  int cap = num_sms() * 8;
  if (blocks > cap) blocks = cap;
  bwd_cols_finalize_kernel<<<blocks, 256, 0, st>>>(static_cast<const float*>(ws), cs.ksplit, (size_t)cs.n_jblocks * 256 * p.D,
                                                   rows, p.D, 0.5f / (float)p.B, grad_loss, wsc, dIz, dI_out, p.gate);
  MC_LAUNCH_CHECK();
  return MC_OK;
}

}  // namespace tc
}  // namespace mc

// "Next" row 3 (SURVEY.md section 8 f): inference-side similarity + top-k retrieval.
// Replaces /root/reference inference.py:42-46 (find_matches) and the same pattern in
// CIFAR.ipynb / classifier.ipynb:
//     image_n = F.normalize(image_embeddings, p=2, dim=-1); text_n = F.normalize(text_embeddings, p=2, dim=-1)
//     dot_similarity = text_n @ image_n.T;  values, indices = torch.topk(dot_similarity, k)
// Eager PyTorch writes a normalised copy of the whole image bank, then a GEMM, then a sort-based
// top-k.  Here the bank is streamed ONCE (HBM-bound: N*D*4 bytes): one warp per image row computes
// the row norm and its dot product with every (pre-normalised, shared-memory resident) query; the
// (Q, N) scores then go through an exact radix select per query.  Keys are 64-bit
// (order-preserving score bits << 32 | ~index), hence unique: the k-th largest key is an exact
// threshold, ties resolve to the LOWER index, and the result is deterministic.
//
// Retrieval evaluation (mc_retrieval_ranks, below): text->image and image->text ranks of every caption and image over
// the whole (Q, N) score matrix, counted inside the epilogue of the resident tcgen05 pair kernel (head_tc.cu,
// kAresRanks), so the matrix is never stored.
//
// Retrieval top-k (mc_retrieval_topk, below): the exact top-k of the same engine scores for a batch of queries, in
// workspace that does not grow with queries x bank.  The bank is swept in chunks of C entries; the epilogue of the
// resident pair kernel (kAresTopk) appends every score at or above its query's running k-th best to that query's C
// slots, and a selection kernel per query merges them into the running top-k and tightens the threshold.
#include <assert.h>

#include "common.cuh"
#include "head_tc.cuh"

namespace mc {

constexpr int kMaxQ = 32;      // queries per streaming pass (host loops over larger Q)
constexpr int kMaxK = 1024;    // top-k kept in shared memory
constexpr float kNormEps = 1e-12f;  // F.normalize default eps

__device__ __forceinline__ uint32_t desc_bits(float f) {  // larger float -> larger unsigned; NaN largest (torch.topk)
  if (f != f) return 0xFFFFFFFFu;
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// text (Q, D) -> normalised queries (Q, D): one warp per query
__global__ void __launch_bounds__(256) normalize_rows_kernel(const float* __restrict__ x, int rows, int D,
                                                             float* __restrict__ out) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= rows) return;
  float s = 0.f;
  for (int k = lane; k < D; k += 32) { const float v = x[(size_t)r * D + k]; s = fmaf(v, v, s); }
  const float inv = 1.f / fmaxf(sqrtf(warp_sum(s)), kNormEps);
  for (int k = lane; k < D; k += 32) out[(size_t)r * D + k] = x[(size_t)r * D + k] * inv;
}

// scores[q][n] = <t_n[q], x[n]> / max(||x[n]||, eps).  kVec float4 per lane cover a row (D = 128 * kVec).
template <int kVec>
__global__ void __launch_bounds__(256) sim_scores_kernel(const float* __restrict__ tn, int Q, const float* __restrict__ x,
                                                         long long N, float* __restrict__ scores) {
  constexpr int D = 128 * kVec;
  extern __shared__ __align__(16) float sq[];  // [Q][D] normalised queries
  for (int i = threadIdx.x; i < Q * D / 4; i += blockDim.x)
    reinterpret_cast<float4*>(sq)[i] = reinterpret_cast<const float4*>(tn)[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long n = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; n < N; n += warps) {
    float4 v[kVec];
#pragma unroll
    for (int u = 0; u < kVec; ++u) v[u] = ld_stream(reinterpret_cast<const float4*>(x + n * D) + lane + 32 * u);
    float nn = 0.f;
#pragma unroll
    for (int u = 0; u < kVec; ++u) nn += (v[u].x * v[u].x + v[u].y * v[u].y) + (v[u].z * v[u].z + v[u].w * v[u].w);
    const float inv = 1.f / fmaxf(sqrtf(warp_sum(nn)), kNormEps);
    for (int q = 0; q < Q; ++q) {
      float d = 0.f;
#pragma unroll
      for (int u = 0; u < kVec; ++u) {
        const float4 t = reinterpret_cast<const float4*>(sq + q * D)[lane + 32 * u];
        d += (v[u].x * t.x + v[u].y * t.y) + (v[u].z * t.z + v[u].w * t.w);
      }
      d = warp_sum(d);
      if (lane == 0) scores[(size_t)q * N + n] = d * inv;
    }
  }
}

// generic D (any multiple of 4 is not required): scalar loads
__global__ void __launch_bounds__(256) sim_scores_generic_kernel(const float* __restrict__ tn, int Q, int D,
                                                                 const float* __restrict__ x, long long N,
                                                                 float* __restrict__ scores) {
  const int lane = threadIdx.x & 31;
  const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long n = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; n < N; n += warps) {
    float nn = 0.f;
    for (int k = lane; k < D; k += 32) { const float v = x[n * D + k]; nn = fmaf(v, v, nn); }
    const float inv = 1.f / fmaxf(sqrtf(warp_sum(nn)), kNormEps);
    for (int q = 0; q < Q; ++q) {
      float d = 0.f;
      for (int k = lane; k < D; k += 32) d = fmaf(x[n * D + k], tn[(size_t)q * D + k], d);
      d = warp_sum(d);
      if (lane == 0) scores[(size_t)q * N + n] = d * inv;
    }
  }
}

__device__ __forceinline__ unsigned long long topk_key(float s, long long n) {
  return ((unsigned long long)desc_bits(s) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)n);
}

// one block per query: exact k-th largest 64-bit key by 8 radix passes, then gather + bitonic sort of the k winners
__global__ void __launch_bounds__(1024) topk_kernel(const float* __restrict__ scores, long long N, int k, int kpad,
                                                    float* __restrict__ out_vals, int64_t* __restrict__ out_idx) {
  __shared__ unsigned int hist[256];
  __shared__ unsigned long long prefix_s;
  __shared__ unsigned int remaining_s, count_s;
  extern __shared__ unsigned long long winners[];  // [kpad]
  const float* row = scores + (size_t)blockIdx.x * N;
  if (threadIdx.x == 0) { prefix_s = 0ull; remaining_s = (unsigned)k; count_s = 0u; }
  __syncthreads();
  for (int pass = 0; pass < 8; ++pass) {
    const int shift = 56 - 8 * pass;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0u;
    __syncthreads();
    const unsigned long long prefix = prefix_s;
    const unsigned long long himask = pass == 0 ? 0ull : (~0ull << (shift + 8));
    for (long long n = threadIdx.x; n < N; n += blockDim.x) {
      const unsigned long long key = topk_key(row[n], n);
      if ((key & himask) == prefix) atomicAdd(&hist[(unsigned)(key >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned int rem = remaining_s;
      int d = 255;
      for (; d > 0; --d) {
        if (hist[d] >= rem) break;
        rem -= hist[d];
      }
      remaining_s = rem;  // the k-th largest is the rem-th largest inside digit d
      prefix_s = prefix | ((unsigned long long)d << shift);
    }
    __syncthreads();
  }
  const unsigned long long thr = prefix_s;  // exactly k keys are >= thr
  for (int i = threadIdx.x; i < kpad; i += blockDim.x) winners[i] = 0ull;
  __syncthreads();
  for (long long n = threadIdx.x; n < N; n += blockDim.x) {
    const unsigned long long key = topk_key(row[n], n);
    if (key >= thr) {
      const unsigned int slot = atomicAdd(&count_s, 1u);
      if (slot < (unsigned)kpad) winners[slot] = key;
    }
  }
  __syncthreads();
  for (int kk = 2; kk <= kpad; kk <<= 1) {  // bitonic, descending
    for (int j = kk >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < (kpad >> 1); t += blockDim.x) {
        const int i = ((t / j) * 2 * j) + (t % j), l = i + j;
        const bool desc = ((i & kk) == 0);
        const unsigned long long a = winners[i], b = winners[l];
        if ((a < b) == desc) { winners[i] = b; winners[l] = a; }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    const long long n = (long long)(0xFFFFFFFFu - (uint32_t)(winners[i] & 0xFFFFFFFFull));
    out_idx[(size_t)blockIdx.x * k + i] = n;
    out_vals[(size_t)blockIdx.x * k + i] = row[n];
  }
}

// ------------------------------------------------------------------------------------------------ retrieval ranks
// t_key[q] = ord(<tn[q], xn[g(q)]>): the score of each caption with its own image (one warp per caption, fp32), and
// u_key[g(q)] = max over the captions of that image (order-preserving integer atomicMax; u_key zeroed = no caption)
__global__ void __launch_bounds__(256) pair_thresholds_kernel(const float* __restrict__ tn, const float* __restrict__ xn,
                                                              int Q, int D, const int64_t* __restrict__ text_to_image,
                                                              unsigned int* __restrict__ t_key,
                                                              unsigned int* __restrict__ u_key) {
  const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (q >= Q) return;
  const int64_t g = text_to_image ? text_to_image[q] : q;
  const float4* a = reinterpret_cast<const float4*>(tn + (size_t)q * D);
  const float4* b = reinterpret_cast<const float4*>(xn + (size_t)g * D);
  float d = 0.f;
  for (int k = lane; k < D / 4; k += 32) {
    const float4 x = a[k], y = b[k];
    d = fmaf(x.x, y.x, d); d = fmaf(x.y, y.y, d); d = fmaf(x.z, y.z, d); d = fmaf(x.w, y.w, d);
  }
  d = warp_sum(d);
  if (lane == 0) {
    const unsigned int key = float_to_ord(d);
    t_key[q] = key;
    atomicMax(u_key + g, key);
  }
}

// images without a caption: rank -1 (their column / row counted nothing: threshold +inf)
__global__ void __launch_bounds__(256) uncaptioned_kernel(const unsigned int* __restrict__ u_key, int N,
                                                          int32_t* __restrict__ i2t_rank) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n < N && u_key[n] == 0u) i2t_rank[n] = -1;
}

// Score prologue shared by mc_retrieval_ranks and mc_retrieval_topk, so that both see the same score bits: both sides
// normalised into the workspace (tn, xn), the LARGER side resident (the rows of the pair kernel: it spreads row blocks
// over the CTA pairs) with its max |.| in *amax, the other side staged as fp16 planes in `planes`.
struct ScoreSides {
  bool text_rows;   // the captions / queries are the rows
  const float* A;   // resident side (M, D)
  int M, N;
  tcg::Planes W;    // streamed side (N, D)
};
static int score_prologue(const float* text, int Q, const float* image, int N, int D, float* tn, float* xn,
                          unsigned int* amax, void* planes, ScoreSides* o, cudaStream_t st) {
  normalize_rows_kernel<<<(Q + 7) / 8, 256, 0, st>>>(text, Q, D, tn);
  MC_LAUNCH_CHECK();
  normalize_rows_kernel<<<(N + 7) / 8, 256, 0, st>>>(image, N, D, xn);
  MC_LAUNCH_CHECK();
  o->text_rows = Q >= N;
  o->M = o->text_rows ? Q : N;
  o->N = o->text_rows ? N : Q;
  o->A = o->text_rows ? tn : xn;
  o->W = tcg::carve_planes(planes, o->N, D);
  int rc;
  if ((rc = tcg::amax(o->A, o->M, D, D, amax, st))) return rc;
  return tcg::stage(o->text_rows ? xn : tn, o->N, D, D, 0, o->W, st);
}

struct RanksLayout {
  size_t tn, xn, t_key, u_key, amax, planes, total;
};
static RanksLayout ranks_layout(int Q, int N, int D) {
  RanksLayout l;
  const int streamed = Q >= N ? N : Q;
  l.tn = 0;
  l.xn = l.tn + round_up((size_t)Q * D * 4, 256);
  l.t_key = l.xn + round_up((size_t)N * D * 4, 256);
  l.u_key = l.t_key + round_up((size_t)Q * 4, 256);
  l.amax = l.u_key + round_up((size_t)N * 4, 256);
  l.planes = l.amax + 256;
  l.total = l.planes + round_up(tcg::planes_bytes(streamed, D), 256);
  return l;
}

// ------------------------------------------------------------------------------------------------ retrieval top-k
// Chunk capacity C (bank entries per launch of the pair kernel = survivor slots per query): the survivor buffer
// Q * C * 8 bytes stays within kSurvivorBudget, C is a whole number of the kernel's bank units (128-column tiles when
// the queries are the rows, 256-row blocks when the bank is), at most kMaxChunk and at most the bank.  With the bank as
// the rows (Q < N) a chunk of C rows gives C / 256 row blocks to the 74 CTA pairs: all of them from C = 18 944, which
// the budget allows up to Q = 1 770 queries.  Above that the budget wins and a chunk leaves pairs idle.
constexpr size_t kSurvivorBudget = size_t(256) << 20;
constexpr int kMaxChunk = 65536;
constexpr int kSelThreads = 512;
constexpr int kSortCap = 4096;   // k + survivors up to this: one shared-memory bitonic sort

static int topk_chunk(int Q, int N) {
  const int unit = Q >= N ? 128 : 256;
  size_t c = kSurvivorBudget / ((size_t)Q * 8) / unit * unit;
  if (c < (size_t)unit) c = unit;
  if (c > (size_t)kMaxChunk) c = kMaxChunk;
  const size_t bank = ((size_t)N + unit - 1) / unit * unit;
  return (int)(c < bank ? c : bank);
}

struct TopkLayout {
  size_t tn, xn, amax, planes, run, theta, cnt, surv, total;
  int cap;
};
static TopkLayout topk_layout(int Q, int N, int D, int k) {
  TopkLayout l;
  l.cap = topk_chunk(Q, N);
  l.tn = 0;
  l.xn = l.tn + round_up((size_t)Q * D * 4, 256);
  l.amax = l.xn + round_up((size_t)N * D * 4, 256);
  l.planes = l.amax + 256;
  l.run = l.planes + round_up(tcg::planes_bytes(Q >= N ? N : Q, D), 256);
  l.theta = l.run + round_up((size_t)Q * k * 8, 256);
  l.cnt = l.theta + round_up((size_t)Q * 4, 256);
  l.surv = l.cnt + round_up((size_t)Q * 4, 256);
  l.total = l.surv + (size_t)Q * l.cap * 8;
  return l;
}

// descending bitonic sort of a[0, P) in shared memory, P a power of two
__device__ void bitonic_desc(unsigned long long* a, int P) {
  for (int kk = 2; kk <= P; kk <<= 1) {
    for (int j = kk >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < (P >> 1); t += blockDim.x) {
        const int i = ((t / j) * 2 * j) + (t % j), l = i + j;
        const bool desc = ((i & kk) == 0);
        const unsigned long long x = a[i], y = a[l];
        if ((x < y) == desc) { a[i] = y; a[l] = x; }
      }
      __syncthreads();
    }
  }
}

// One block per query: the running top-k run[q] (k keys, descending, 0 = empty) and the query's cnt[q] survivors of
// the last chunk -> the top-k of their union, theta[q] = score bits of the k-th key (0 while fewer than k exist),
// cnt[q] = 0.  Survivor keys are unique and a key's rank does not depend on where it sits, so the result does not
// depend on the order in which the survivors arrived.
__global__ void __launch_bounds__(kSelThreads) topk_merge_kernel(unsigned long long* __restrict__ run, int k,
                                                                 const unsigned long long* __restrict__ surv, int cap,
                                                                 unsigned int* __restrict__ cnt,
                                                                 unsigned int* __restrict__ theta) {
  __shared__ unsigned long long a[kSortCap];
  __shared__ unsigned int hist[256];
  __shared__ unsigned long long prefix_s;
  __shared__ unsigned int remaining_s, count_s;
  const int q = blockIdx.x;
  const unsigned int n_raw = cnt[q];
#ifdef MC_DEBUG_ASSERTS
  assert(n_raw <= (unsigned int)cap);
#endif
  const int n = (int)min(n_raw, (unsigned int)cap);
  if (n == 0) return;
  unsigned long long* const r = run + (size_t)q * k;
  const unsigned long long* const s = surv + (size_t)q * cap;
  const int total = k + n;
  if (total <= kSortCap) {
    int P = 2;
    while (P < total) P <<= 1;
    for (int i = threadIdx.x; i < P; i += blockDim.x) a[i] = i < k ? r[i] : (i < total ? s[i - k] : 0ull);
    __syncthreads();
    bitonic_desc(a, P);
  } else {
    // exact k-th largest key of the union by 8 radix passes (keys are unique except the empty 0s)
    if (threadIdx.x == 0) { prefix_s = 0ull; remaining_s = (unsigned)k; count_s = 0u; }
    __syncthreads();
    for (int pass = 0; pass < 8; ++pass) {
      const int shift = 56 - 8 * pass;
      for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0u;
      __syncthreads();
      const unsigned long long prefix = prefix_s;
      const unsigned long long himask = pass == 0 ? 0ull : (~0ull << (shift + 8));
      for (int i = threadIdx.x; i < total; i += blockDim.x) {
        const unsigned long long key = i < k ? r[i] : s[i - k];
        if ((key & himask) == prefix) atomicAdd(&hist[(unsigned)(key >> shift) & 255u], 1u);
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        unsigned int rem = remaining_s;
        int d = 255;
        for (; d > 0; --d) {
          if (hist[d] >= rem) break;
          rem -= hist[d];
        }
        remaining_s = rem;
        prefix_s = prefix | ((unsigned long long)d << shift);
      }
      __syncthreads();
    }
    const unsigned long long thr = prefix_s;   // the k-th largest key: fewer than k keys lie above it
    int P = 2;
    while (P < k) P <<= 1;
    for (int i = threadIdx.x; i < P; i += blockDim.x) a[i] = i < k ? thr : 0ull;
    __syncthreads();
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
      const unsigned long long key = i < k ? r[i] : s[i - k];
      if (key > thr) a[atomicAdd(&count_s, 1u)] = key;   // the rest of [0, k) keeps thr
    }
    __syncthreads();
    bitonic_desc(a, P);
  }
  for (int i = threadIdx.x; i < k; i += blockDim.x) r[i] = a[i];
  if (threadIdx.x == 0) {
    theta[q] = (unsigned int)(a[k - 1] >> 32);
    cnt[q] = 0u;
  }
}

struct TopkMerge {
  unsigned long long* run;
  int Q, k, cap;
  const unsigned long long* surv;
  unsigned int* cnt;
  unsigned int* theta;
};
static int topk_merge(void* ctx, cudaStream_t st) {
  const TopkMerge& m = *static_cast<const TopkMerge*>(ctx);
  topk_merge_kernel<<<m.Q, kSelThreads, 0, st>>>(m.run, m.k, m.surv, m.cap, m.cnt, m.theta);
  MC_LAUNCH_CHECK();
  return MC_OK;
}

// keys -> the engine's fp32 scores and int64 bank indices
__global__ void __launch_bounds__(256) topk_out_kernel(const unsigned long long* __restrict__ run, size_t total,
                                                       float* __restrict__ out_vals, int64_t* __restrict__ out_idx) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const unsigned long long key = run[i];
  out_vals[i] = ord_to_float((unsigned int)(key >> 32));
  out_idx[i] = (int64_t)(~(uint32_t)key);
}

}  // namespace mc

using namespace mc;

extern "C" {

size_t mc_similarity_topk_workspace_bytes(int Q, long long N, int D) {
  if (Q <= 0 || N <= 0 || D <= 0) return 0;
  return round_up((size_t)Q * D * sizeof(float), 256) + (size_t)Q * (size_t)N * sizeof(float);
}

int mc_similarity_topk(const float* text, int Q, const float* image, long long N, int D, int k, float* out_vals,
                       int64_t* out_idx, float* scores_out, void* ws, size_t ws_bytes, void* stream) {
  MC_ARCH_GUARD();
  MC_REQUIRE(text && image && ws && (k == 0 || (out_vals && out_idx)), MC_ERR_BAD_ARG, "similarity_topk: null pointer");
  MC_REQUIRE(Q > 0 && N > 0 && D > 0 && k >= 0, MC_ERR_BAD_ARG, "similarity_topk: bad sizes Q=%d N=%lld D=%d k=%d", Q, N, D, k);
  MC_REQUIRE(k <= N, MC_ERR_BAD_ARG, "similarity_topk: k=%d exceeds the %lld candidates (torch.topk raises too)", k, N);
  MC_REQUIRE(k <= kMaxK, MC_ERR_UNSUPPORTED, "similarity_topk: k=%d > %d", k, kMaxK);
  MC_REQUIRE(N < 0xFFFFFFFFll, MC_ERR_UNSUPPORTED, "similarity_topk: more than 2^32 - 1 candidates");
  MC_REQUIRE(ws_bytes >= mc_similarity_topk_workspace_bytes(Q, N, D), MC_ERR_WORKSPACE, "similarity_topk: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* tn = static_cast<float*>(ws);
  float* scores = scores_out ? scores_out : reinterpret_cast<float*>(static_cast<char*>(ws) + round_up((size_t)Q * D * 4, 256));
  normalize_rows_kernel<<<(Q + 7) / 8, 256, 0, st>>>(text, Q, D, tn);
  MC_LAUNCH_CHECK();
  long long nb = (N + 7) / 8;
  const long long cap = (long long)num_sms() * 8;
  if (nb > cap) nb = cap;
  const bool vec = (D == 128 || D == 256 || D == 512) && aligned(image, 16);
  for (int q0 = 0; q0 < Q; q0 += kMaxQ) {
    const int qn = Q - q0 < kMaxQ ? Q - q0 : kMaxQ;
    const float* tq = tn + (size_t)q0 * D;
    float* sc = scores + (size_t)q0 * N;
    const size_t smem = (size_t)qn * D * sizeof(float);
    if (vec && D == 128) sim_scores_kernel<1><<<(int)nb, 256, smem, st>>>(tq, qn, image, N, sc);
    else if (vec && D == 256) sim_scores_kernel<2><<<(int)nb, 256, smem, st>>>(tq, qn, image, N, sc);
    else if (vec && D == 512) {
      MC_CUDA(ensure_dynamic_smem<sim_scores_kernel<4>>(kMaxQ * 512 * 4));
      sim_scores_kernel<4><<<(int)nb, 256, smem, st>>>(tq, qn, image, N, sc);
    } else sim_scores_generic_kernel<<<(int)nb, 256, 0, st>>>(tq, qn, D, image, N, sc);
    MC_LAUNCH_CHECK();
  }
  if (k > 0) {
    int kpad = 2;
    while (kpad < k) kpad <<= 1;
    topk_kernel<<<Q, 1024, (size_t)kpad * 8, st>>>(scores, N, k, kpad, out_vals, out_idx);
    MC_LAUNCH_CHECK();
  }
  return MC_OK;
}

size_t mc_retrieval_ranks_workspace_bytes(int Q, int N, int D, int mode) {
  (void)mode;
  if (Q <= 0 || N <= 0 || D <= 0) return 0;
  return ranks_layout(Q, N, D).total;
}

// One pass of the resident pair kernel over the (Q, N) cosine scores, which are never stored.  The LARGER side is the
// resident (row) operand: the kernel spreads row blocks over the CTA pairs, so a 1 000-image bank against 25 000
// captions still fills the GPU.  Rows and columns swap their thresholds and positive-pair keys with the orientation.
int mc_retrieval_ranks(const float* text, int Q, const float* image, int N, int D, const int64_t* text_to_image, int mode,
                       int32_t* t2i_rank, int32_t* i2t_rank, void* ws, size_t ws_bytes, void* stream) {
  MC_ARCH_GUARD();
  MC_REQUIRE(text && image && t2i_rank && i2t_rank && ws, MC_ERR_BAD_ARG, "retrieval_ranks: null pointer");
  MC_REQUIRE(Q > 0 && N > 0 && D > 0, MC_ERR_BAD_ARG, "retrieval_ranks: bad sizes Q=%d N=%d D=%d", Q, N, D);
  MC_REQUIRE(text_to_image || Q == N, MC_ERR_BAD_ARG,
             "retrieval_ranks: without text_to_image caption q pairs with image q, so Q (%d) must equal N (%d)", Q, N);
  MC_REQUIRE(mode == MC_GEMM_TC_F16X3 || mode == MC_GEMM_TC_F16 || mode == MC_GEMM_SIMT_FP32, MC_ERR_BAD_ARG,
             "retrieval_ranks: unknown mode %d", mode);
  MC_REQUIRE(mode != MC_GEMM_SIMT_FP32, MC_ERR_UNSUPPORTED, "retrieval_ranks: runs on the tensor cores only (tc_f16x3 or tc_f16)");
  MC_REQUIRE(D <= 256 && D % 4 == 0, MC_ERR_UNSUPPORTED, "retrieval_ranks: needs D <= 256 and D %% 4 == 0 (D=%d)", D);
  MC_REQUIRE(aligned(ws, 256), MC_ERR_ALIGN, "retrieval_ranks: workspace must be 256-byte aligned");
  MC_REQUIRE(ws_bytes >= mc_retrieval_ranks_workspace_bytes(Q, N, D, mode), MC_ERR_WORKSPACE,
             "retrieval_ranks: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const RanksLayout l = ranks_layout(Q, N, D);
  char* base = static_cast<char*>(ws);
  float* tn = reinterpret_cast<float*>(base + l.tn);
  float* xn = reinterpret_cast<float*>(base + l.xn);
  unsigned int* t_key = reinterpret_cast<unsigned int*>(base + l.t_key);
  unsigned int* u_key = reinterpret_cast<unsigned int*>(base + l.u_key);
  unsigned int* amax = reinterpret_cast<unsigned int*>(base + l.amax);
  ScoreSides sides;
  int rc;
  if ((rc = score_prologue(text, Q, image, N, D, tn, xn, amax, base + l.planes, &sides, st))) return rc;
  MC_CUDA(cudaMemsetAsync(u_key, 0, (size_t)N * 4, st));
  MC_CUDA(cudaMemsetAsync(t2i_rank, 0, (size_t)Q * 4, st));
  MC_CUDA(cudaMemsetAsync(i2t_rank, 0, (size_t)N * 4, st));
  pair_thresholds_kernel<<<(Q + 7) / 8, 256, 0, st>>>(tn, xn, Q, D, text_to_image, t_key, u_key);
  MC_LAUNCH_CHECK();

  const bool text_rows = sides.text_rows;
  hg::AresRankArgs a = {};
  a.M = sides.M;
  a.N = sides.N;
  a.K = D;
  a.passes = mode == MC_GEMM_TC_F16X3 ? 3 : 1;
  a.A = sides.A;
  a.a_amax = amax;
  a.W = sides.W;
  a.thr_row = text_rows ? t_key : u_key;
  a.thr_col = text_rows ? u_key : t_key;
  a.key_row = text_rows ? text_to_image : nullptr;   // positive pair: text_to_image[q] == n
  a.key_col = text_rows ? nullptr : text_to_image;
  a.cnt_row = text_rows ? t2i_rank : i2t_rank;
  a.cnt_col = text_rows ? i2t_rank : t2i_rank;
  if ((rc = hg::ares_ranks(a, st))) return rc;
  uncaptioned_kernel<<<(N + 255) / 256, 256, 0, st>>>(u_key, N, i2t_rank);
  MC_LAUNCH_CHECK();
  return MC_OK;
}

size_t mc_retrieval_topk_workspace_bytes(int Q, int N, int D, int k, int mode) {
  (void)mode;
  if (Q <= 0 || N <= 0 || D <= 0 || k <= 0) return 0;
  return topk_layout(Q, N, D, k).total;
}

int mc_retrieval_topk(const float* text, int Q, const float* image, int N, int D, int k, int mode, float* out_vals,
                      int64_t* out_idx, void* ws, size_t ws_bytes, void* stream) {
  MC_ARCH_GUARD();
  MC_REQUIRE(text && image && out_vals && out_idx && ws, MC_ERR_BAD_ARG, "retrieval_topk: null pointer");
  MC_REQUIRE(Q > 0 && N > 0 && D > 0 && k > 0, MC_ERR_BAD_ARG, "retrieval_topk: bad sizes Q=%d N=%d D=%d k=%d", Q, N, D,
             k);
  MC_REQUIRE(k <= N, MC_ERR_BAD_ARG, "retrieval_topk: k=%d exceeds the %d candidates (torch.topk raises too)", k, N);
  MC_REQUIRE(k <= kMaxK, MC_ERR_UNSUPPORTED, "retrieval_topk: k=%d > %d", k, kMaxK);
  MC_REQUIRE(mode == MC_GEMM_TC_F16X3 || mode == MC_GEMM_TC_F16 || mode == MC_GEMM_SIMT_FP32, MC_ERR_BAD_ARG,
             "retrieval_topk: unknown mode %d", mode);
  MC_REQUIRE(mode != MC_GEMM_SIMT_FP32, MC_ERR_UNSUPPORTED, "retrieval_topk: runs on the tensor cores only (tc_f16x3 or tc_f16)");
  MC_REQUIRE(D <= 256 && D % 4 == 0, MC_ERR_UNSUPPORTED, "retrieval_topk: needs D <= 256 and D %% 4 == 0 (D=%d)", D);
  MC_REQUIRE(aligned(ws, 256), MC_ERR_ALIGN, "retrieval_topk: workspace must be 256-byte aligned");
  MC_REQUIRE(ws_bytes >= mc_retrieval_topk_workspace_bytes(Q, N, D, k, mode), MC_ERR_WORKSPACE,
             "retrieval_topk: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const TopkLayout l = topk_layout(Q, N, D, k);
  char* base = static_cast<char*>(ws);
  float* tn = reinterpret_cast<float*>(base + l.tn);
  float* xn = reinterpret_cast<float*>(base + l.xn);
  unsigned int* amax = reinterpret_cast<unsigned int*>(base + l.amax);
  ScoreSides sides;
  int rc;
  if ((rc = score_prologue(text, Q, image, N, D, tn, xn, amax, base + l.planes, &sides, st))) return rc;
  MC_CUDA(cudaMemsetAsync(base + l.run, 0, l.surv - l.run, st));   // running keys, thresholds and counters

  TopkMerge merge;
  merge.run = reinterpret_cast<unsigned long long*>(base + l.run);
  merge.Q = Q; merge.k = k; merge.cap = l.cap;
  merge.surv = reinterpret_cast<unsigned long long*>(base + l.surv);
  merge.cnt = reinterpret_cast<unsigned int*>(base + l.cnt);
  merge.theta = reinterpret_cast<unsigned int*>(base + l.theta);
  hg::AresTopkArgs a = {};
  a.A = sides.A;
  a.a_amax = amax;
  a.W = sides.W;
  a.M = sides.M;
  a.N = sides.N;
  a.K = D;
  a.passes = mode == MC_GEMM_TC_F16X3 ? 3 : 1;
  a.query_rows = sides.text_rows ? 1 : 0;
  a.cap = l.cap;
  a.theta = merge.theta;
  a.surv = reinterpret_cast<unsigned long long*>(base + l.surv);
  a.cnt = merge.cnt;
  a.after_chunk = topk_merge;
  a.ctx = &merge;
  if ((rc = hg::ares_topk(a, st))) return rc;
  const size_t total = (size_t)Q * k;
  topk_out_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(merge.run, total, out_vals, out_idx);
  MC_LAUNCH_CHECK();
  return MC_OK;
}

}  // extern "C"

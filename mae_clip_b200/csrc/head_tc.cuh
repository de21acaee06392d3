// ProjectionHead GEMMs, second generation (modules.py:63-75 and their autograd): CTA-pair tcgen05 kernels that take
// the ACTIVATION operand as it lies in HBM (fp32, row-major) and split it into fp16 hi/lo inside the kernel, so no
// operand plane of an activation is ever staged in HBM.  See head_tc.cu for the execution model.
#pragma once
#include "common.cuh"
#include "gemm_tc.cuh"

namespace mc {
namespace hg {

enum RowEpilogue {
  kEpiPlain = 0,    // C = acc (+ bias)
  kEpiBiasGelu = 1, // out0 = acc + bias ; out1 = gelu(out0) ; out_amax = max |out1|          (x Wp^T, modules.py:70-71)
  kEpiLN = 2,       // z = keep * (acc + bias) / (1-p) + in0 ; out0 = LayerNorm(z) ; out1 = z   (modules.py:72-75)
  kEpiGeluBwd = 3   // out0 = acc * gelu'(in0) + in1 ; out_amax = max |out0| ; column partials  (backward of :70-71)
};

struct RowArgs {
  const float* A;             // (M, K) fp32 row-major, row stride lda floats (16-byte aligned rows)
  int64_t lda;
  const unsigned int* a_amax; // device word: bit pattern of max |A| (the producer of A reduced it)
  tcg::Planes W;              // (256, K) staged weight planes (fp16 hi / lo, K-major)
  int M, K;
  int passes;                 // 3: hi*hi + hi*lo + lo*hi (fp32-class) ; 1: hi*hi
  int epilogue;
  const float* bias;          // length 256 or null
  float* out0;
  float* out1;
  const float* in0;
  const float* in1;
  const uint8_t* keep;        // kEpiLN: (M, 256) 0/1 bytes or null (eval mode)
  float drop_scale, eps;
  const float* gamma;
  const float* beta;
  float* mean;
  float* rstd;
  unsigned int* out_amax;     // or null
  float* colpart;             // kEpiGeluBwd: (colpart_rows(M), 256) per-warp column sums of out0, or null
  // Scale protocol.  The fp16 planes need a power-of-two scale from max |A|; reducing it first costs a whole pass over A
  // (45 us for the 268 MB image features).  A power-of-two scale only matters at the ends of the fp16 range, so the
  // scale of the PREVIOUS call is as good - provided it is checked:
  //   vmode 1  run with the previous call's max |A| (*v_stale) while the converters reduce the true one into *a_live
  //   vmode 2  the same launch again: every CTA returns at once when *v_live was inside the safe window of *v_stale
  //            (no fp16 overflow, lo plane not starved), else the GEMM is redone with the exact scale
  //   vmode 3  a consumer of what those two produced: its own operand's max is *a_amax when the first attempt stood,
  //            *a_alt when it was redone; *amax_publish receives the one chosen
  //   vmode 0  plain: *a_amax
  int vmode;
  const unsigned int* a_alt;
  const unsigned int* v_stale;
  const unsigned int* v_live;
  unsigned int* a_live;
  unsigned int* amax_publish;
};
int colpart_rows(int M);      // rows of RowArgs::colpart for a problem with M rows
// C-like: out(M, 256) = A(M, K) . W(256, K)^T with the epilogue fused.  K % 4 == 0.
int rows_gemm(const RowArgs& a, cudaStream_t st);

// C(M, N) = A(M, K) . W(N, K)^T for a SHORT K (K <= 256, K % 4 == 0): the converted row block of A stays resident in
// tensor memory while the column tiles of W stream by (dx = dp Wp, modules.py:70 backward).  N % 4 == 0.
struct AresArgs {
  const float* A;
  int64_t lda;
  const unsigned int* a_amax;
  tcg::Planes W;              // (N, K)
  int M, N, K, passes;
  float* C;
  int64_t ldc;
};
int ares_gemm(const AresArgs& a, cudaStream_t st);

// The same kernel with a counting epilogue instead of the store (retrieval ranks, retrieval.cu): S = A . W^T is never
// written.  For every row r and column c that are not a positive pair (key_row[r] != key_col[c]; a null key array is
// the identity r / c):
//   cnt_row[r] += 1 when S[r][c] > thr_row[r]        cnt_col[c] += 1 when S[r][c] > thr_col[c]
// Thresholds are order-preserving integers of floats (float_to_ord; 0 = +inf, nothing counts).  The counts are
// added with integer atomics (zero them first): exact and identical run to run.  A is (M, K) dense, K <= 256.
struct AresRankArgs {
  const float* A;
  const unsigned int* a_amax;
  tcg::Planes W;              // (N, K)
  int M, N, K, passes;
  const unsigned int* thr_row;
  const unsigned int* thr_col;
  const int64_t* key_row;
  const int64_t* key_col;
  int* cnt_row;
  int* cnt_col;
};
int ares_ranks(const AresRankArgs& a, cudaStream_t st);

// The same kernel with a top-k epilogue (retrieval top-k, retrieval.cu): S = A . W^T is never written.  One side holds
// the queries, the other the bank; query_rows = 1: the M rows are the queries and the N columns the bank, 0: the other
// way round.  The bank is covered in chunks of `cap` entries (whole 128-column tiles / 256-row blocks), one launch per
// chunk, all from the same tensor maps.  In a launch, every score s of a query with ord(s) >= theta[query]
// (float_to_ord bits; 0 = no threshold yet) is appended as the key (ord(s) << 32 | ~bank index) to
// surv[query * cap + cnt[query]++]; a chunk holds at most cap bank entries, so no query's slots can overflow.  After
// each launch after_chunk(ctx, st) runs on the stream: it consumes the survivors, tightens theta and zeroes cnt.
struct AresTopkArgs {
  const float* A;
  const unsigned int* a_amax;
  tcg::Planes W;              // (N, K)
  int M, N, K, passes;
  int query_rows;
  int cap;
  const unsigned int* theta;
  unsigned long long* surv;   // (queries, cap)
  unsigned int* cnt;          // (queries,), zero on entry
  int (*after_chunk)(void* ctx, cudaStream_t st);
  void* ctx;
};
int ares_topk(const AresTopkArgs& a, cudaStream_t st);

// C(Mo, No) = A^T . B with A (K, Mo) and B (K, No) both fp32 row-major (the weight gradients: K is the batch).  Both
// operands are converted AND transposed inside the kernel.  Mo == 256.  Split-K partials go to `ws`; a second kernel
// reduces them deterministically.
struct TtArgs {
  const float* A;
  int64_t lda;
  const unsigned int* a_amax;
  const float* B;
  int64_t ldb;
  const unsigned int* b_amax;
  int K, No, passes;
  float* C;                   // (256, No), row stride ldc
  int64_t ldc;
};
size_t tt_workspace_bytes(int No, int K);
int tt_gemm(const TtArgs& a, void* ws, size_t ws_bytes, cudaStream_t st);

bool supported(int P);        // the pair kernels cover projection_dim == 256 (the reference's default, config.py:23)

}  // namespace hg
}  // namespace mc

// C-ABI entry points of the contrastive soft-target loss (L3-L6): argument checks, engine
// dispatch (SIMT fp32 strips vs tcgen05 fused tiles) and the single-GPU fused / host-buffer
// conveniences.  Reference: /root/reference CLIP.py:34-43 (+ autograd at main.py:58).
#include <stdlib.h>

#include <mutex>
#include <string>
#include <vector>

#include "clip_loss.cuh"

namespace mc {

static int check_problem(const char* who, const float* I_all, const float* T_all, int b, int B, int D,
                         int row_offset, float tau, int mode) {
  MC_REQUIRE(b > 0 && B > 0 && D > 0 && b <= B, MC_ERR_BAD_ARG, "%s: bad sizes b=%d B=%d D=%d", who,
             b, B, D);
  MC_REQUIRE(row_offset >= 0 && row_offset + b <= B, MC_ERR_BAD_ARG, "%s: row_offset %d out of range",
             who, row_offset);
  MC_REQUIRE(tau > 0.f, MC_ERR_BAD_ARG, "%s: temperature must be positive (got %g)", who, tau);
  MC_REQUIRE(mode >= MC_GEMM_SIMT_FP32 && mode <= MC_GEMM_TC_F16, MC_ERR_BAD_ARG, "%s: bad mode %d",
             who, mode);
  // the tcgen05 engine reads the staged planes only; the fp32 embeddings may then be absent
  // (peer-memory staging never assembles them)
  MC_REQUIRE((I_all && T_all) || (mode != MC_GEMM_SIMT_FP32 && tc::supported(D)), MC_ERR_BAD_ARG,
             "%s: null embedding pointer", who);
  return MC_OK;
}

// Shapes the tcgen05 engine does not cover (D other than 128 / 256) run on the fp32 SIMT
// engine: same device, same ABI, true-fp32 arithmetic - never a CPU path.
static int eff_mode(int mode, int D) {
  return (mode != MC_GEMM_SIMT_FP32 && !tc::supported(D)) ? (int)MC_GEMM_SIMT_FP32 : mode;
}

struct FusedLayout {
  size_t off_vec, off_flags, off_planes, off_phase, total;
  size_t vec_stride, flags_bytes;
  // stored-weights gradient (tc::bwd_rows / tc::bwd_cols): the fp16 weights of all B x B pairs, the un-scaled soft-target
  // part of dI and the column half's partials; all zero when that form is off
  size_t off_w, off_diz, off_cols, cols_bytes, phase_bytes;
};
static FusedLayout fused_layout(int B, int D, int mode) {
  mode = eff_mode(mode, D);
  FusedLayout l;
  l.vec_stride = round_up((size_t)B * 4, 256);
  l.off_vec = 0;
  l.flags_bytes = (mode == MC_GEMM_SIMT_FP32) ? 0 : round_up(tc::tile_flags_bytes(B, B), 256);
  l.off_flags = round_up(6 * l.vec_stride + 256, 256);    // raw flags of the statistics sweep, then the symmetrised ones
  l.off_planes = round_up(l.off_flags + 2 * l.flags_bytes, 1024);  // planes 1024-aligned
  size_t planes = (mode == MC_GEMM_SIMT_FP32) ? 0 : tc::planes_bytes(B, D, mode);
  l.off_phase = l.off_planes + round_up(planes, 256);
  size_t phase = (mode == MC_GEMM_SIMT_FP32) ? simt::workspace_bytes(B, B, D)
                                             : tc::workspace_bytes(B, B, D, mode);
  l.phase_bytes = round_up(phase, 256);
  l.total = l.off_phase + l.phase_bytes;
  l.off_w = l.off_diz = l.off_cols = l.cols_bytes = 0;
  if (mode != MC_GEMM_SIMT_FP32 && tc::stored_form_enabled(B, B, D)) {
    // tc::workspace_bytes(B, B, ...) already holds the stored-weights buffers behind the sweeps' partials
    tc::StoredLayout sl = tc::stored_layout(B, D, mode);
    l.off_w = l.off_phase + sl.off_w;
    l.off_diz = l.off_phase + sl.off_diz;
    l.off_cols = l.off_phase + sl.off_cols;
    l.cols_bytes = sl.cols_bytes;
    l.phase_bytes = sl.off_w;     // what a row strip's sweep may use
  }
  return l;
}

}  // namespace mc

using namespace mc;

extern "C" {

size_t mc_clip_loss_workspace_bytes(int b, int B, int D, int mode) {
  if (b <= 0 || B <= 0 || D <= 0) return 0;
  mode = eff_mode(mode, D);
  return mode == MC_GEMM_SIMT_FP32 ? simt::workspace_bytes(b, B, D) : tc::workspace_bytes(b, B, D, mode);
}

size_t mc_clip_planes_bytes(int B, int D, int mode) {
  if (B <= 0 || D <= 0 || eff_mode(mode, D) == MC_GEMM_SIMT_FP32) return 0;
  return tc::planes_bytes(B, D, mode);
}

int mc_clip_prepare(const float* I_loc, const float* T_loc, int b, int B, int D, int row_offset,
                    int mode, void* planes_all, void* stream) {
  MC_ARCH_GUARD();
  MC_REQUIRE(I_loc && T_loc, MC_ERR_BAD_ARG, "clip_prepare: null pointer");
  MC_REQUIRE(b > 0 && B >= b && D > 0 && row_offset >= 0 && row_offset + b <= B, MC_ERR_BAD_ARG,
             "clip_prepare: bad sizes");
  MC_REQUIRE(mode >= MC_GEMM_SIMT_FP32 && mode <= MC_GEMM_TC_F16, MC_ERR_BAD_ARG, "clip_prepare: bad mode %d", mode);
  if (eff_mode(mode, D) == MC_GEMM_SIMT_FP32) return MC_OK;
  MC_REQUIRE(planes_all, MC_ERR_BAD_ARG, "clip_prepare: planes_all is null");
  return tc::prepare(I_loc, T_loc, b, B, D, row_offset, mode, planes_all,
                     static_cast<cudaStream_t>(stream));
}

size_t mc_clip_tile_flags_bytes(int b, int B, int D, int mode) {
  if (b <= 0 || B <= 0 || D <= 0 || eff_mode(mode, D) == MC_GEMM_SIMT_FP32) return 0;
  return tc::tile_flags_bytes(b, B);
}

int mc_clip_flags_finalize(const uint8_t* flags_all, int B, int b, int row_offset, uint8_t* flags_loc, void* stream) {
  MC_ARCH_GUARD();
  MC_REQUIRE(flags_all && flags_loc && b > 0 && B >= b && row_offset >= 0 && row_offset + b <= B, MC_ERR_BAD_ARG,
             "clip_flags_finalize: bad argument");
  return tc::flags_finalize(flags_all, B, b, row_offset, flags_loc, static_cast<cudaStream_t>(stream));
}

int mc_clip_amax(const float* I_loc, const float* T_loc, int b, int D, float* I_copy, float* T_copy,
                 unsigned int* amax_bits, void* stream) {
  MC_ARCH_GUARD();
  MC_REQUIRE(I_loc && T_loc && amax_bits && b > 0 && D > 0, MC_ERR_BAD_ARG, "clip_amax: bad argument");
  return tc::amax_copy(I_loc, T_loc, b, D, I_copy, T_copy, amax_bits, static_cast<cudaStream_t>(stream));
}

int mc_clip_push_shards(const float* I_loc, const float* T_loc, int b, int D, int rank, int world,
                        float* const* I_all_dst_host, float* const* T_all_dst_host,
                        unsigned int* const* amax_slots_host, unsigned int* scratch, void* stream) {
  MC_ARCH_GUARD();
  MC_REQUIRE(I_loc && T_loc && I_all_dst_host && T_all_dst_host && amax_slots_host && scratch && b > 0 && D > 0,
             MC_ERR_BAD_ARG, "clip_push_shards: bad argument");
  return tc::push_shards(I_loc, T_loc, b, D, rank, world, I_all_dst_host, T_all_dst_host, amax_slots_host, scratch,
                         static_cast<cudaStream_t>(stream));
}

int mc_clip_prepare_peers(const float* const* I_peers_host, const float* const* T_peers_host, int world, int b,
                          int D, int mode, const unsigned int* amax_slots, void* planes_all, void* stream) {
  MC_ARCH_GUARD();
  MC_REQUIRE(I_peers_host && T_peers_host && amax_slots && planes_all && b > 0 && D > 0, MC_ERR_BAD_ARG,
             "clip_prepare_peers: bad argument");
  MC_REQUIRE(mode == MC_GEMM_TC_F16X3 || mode == MC_GEMM_TC_F16, MC_ERR_UNSUPPORTED,
             "clip_prepare_peers: peer staging feeds the tcgen05 engine only (mode %d)", mode);
  return tc::prepare_peers(I_peers_host, T_peers_host, world, b, D, mode, amax_slots, planes_all,
                           static_cast<cudaStream_t>(stream));
}

int mc_clip_stats(const float* I_all, const float* T_all, const void* planes_all, int b, int B,
                  int D, int row_offset, float tau, int mode, float* r_loc, float* c_loc,
                  float* rz_loc, float* ps_loc, uint8_t* tile_flags_out, void* ws, size_t ws_bytes, void* stream) {
  MC_ARCH_GUARD();
  int rc = check_problem("clip_stats", I_all, T_all, b, B, D, row_offset, tau, mode);
  if (rc) return rc;
  MC_REQUIRE(r_loc && c_loc && rz_loc && ps_loc && ws, MC_ERR_BAD_ARG, "clip_stats: null output/workspace");
  ClipProblem p{I_all, T_all, planes_all, b, B, D, row_offset, tau};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  mode = eff_mode(mode, D);
  if (mode == MC_GEMM_SIMT_FP32) return simt::stats(p, r_loc, c_loc, rz_loc, ps_loc, ws, ws_bytes, st);
  p.tile_flags_out = tile_flags_out;
  return tc::stats(p, mode, r_loc, c_loc, rz_loc, ps_loc, ws, ws_bytes, st);
}

size_t mc_clip_stats_colpart_workspace_bytes(int b, int B, int D, int mode) {
  if (b <= 0 || B <= 0 || D <= 0 || eff_mode(mode, D) == MC_GEMM_SIMT_FP32) return 0;
  return tc::stats_colpart_workspace_bytes(b, B, D, mode);
}

int mc_clip_stats_colpart(const void* planes_all, int b, int B, int D, int row_offset, float tau, int mode,
                          float* r_loc, float* c_part_all, float* rz_loc, float* ps_loc, uint8_t* tile_flags_out,
                          void* ws, size_t ws_bytes, void* stream) {
  MC_ARCH_GUARD();
  int rc = check_problem("clip_stats_colpart", nullptr, nullptr, b, B, D, row_offset, tau, mode);
  if (rc) return rc;
  MC_REQUIRE(eff_mode(mode, D) != MC_GEMM_SIMT_FP32, MC_ERR_UNSUPPORTED,
             "clip_stats_colpart: the column-partials form belongs to the tcgen05 engines (mode %d, D %d)", mode, D);
  MC_REQUIRE(planes_all && r_loc && c_part_all && rz_loc && ps_loc && ws, MC_ERR_BAD_ARG, "clip_stats_colpart: null pointer");
  ClipProblem p{nullptr, nullptr, planes_all, b, B, D, row_offset, tau};
  p.tile_flags_out = tile_flags_out;
  return tc::stats(p, mode, r_loc, nullptr, rz_loc, ps_loc, ws, ws_bytes, static_cast<cudaStream_t>(stream), c_part_all);
}

int mc_clip_colpart_merge(const float* parts, int n_parts, int64_t stride, int B, float* col_lse_all, void* stream) {
  MC_ARCH_GUARD();
  MC_REQUIRE(parts && col_lse_all && n_parts > 0 && B > 0 && stride >= B, MC_ERR_BAD_ARG, "clip_colpart_merge: bad argument");
  return tc::ranks_lse_merge(parts, n_parts, stride, B, col_lse_all, static_cast<cudaStream_t>(stream));
}

int mc_clip_rowloss(const float* I_all, const float* T_all, const void* planes_all, int b, int B,
                    int D, int row_offset, float tau, int mode, const float* r_all,
                    const float* c_all, const float* rz_all, const float* ps_loc, float* g_loc,
                    float* q_loc, float* loss_part, const uint8_t* tile_flags, void* ws, size_t ws_bytes,
                    void* stream) {
  MC_ARCH_GUARD();
  int rc = check_problem("clip_rowloss", I_all, T_all, b, B, D, row_offset, tau, mode);
  if (rc) return rc;
  MC_REQUIRE(r_all && c_all && rz_all && ps_loc && g_loc && q_loc && loss_part && ws, MC_ERR_BAD_ARG,
             "clip_rowloss: null pointer");
  ClipProblem p{I_all, T_all, planes_all, b, B, D, row_offset, tau};
  ClipStatsAll s{r_all, c_all, rz_all, nullptr, nullptr};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  mode = eff_mode(mode, D);
  if (mode == MC_GEMM_SIMT_FP32) return simt::rowloss(p, s, ps_loc, g_loc, q_loc, loss_part, ws, ws_bytes, st);
  p.tile_flags = tile_flags;
  return tc::rowloss(p, mode, s, ps_loc, g_loc, q_loc, loss_part, ws, ws_bytes, st);
}

int mc_clip_bwd(const float* I_all, const float* T_all, const void* planes_all, int b, int B, int D,
                int row_offset, float tau, int mode, const float* r_all, const float* c_all,
                const float* rz_all, const float* g_all, const float* q_all, const float* grad_loss,
                float* dI_loc, float* dT_loc, const uint8_t* tile_flags, void* ws, size_t ws_bytes, void* stream) {
  MC_ARCH_GUARD();
  int rc = check_problem("clip_bwd", I_all, T_all, b, B, D, row_offset, tau, mode);
  if (rc) return rc;
  MC_REQUIRE(r_all && c_all && rz_all && g_all && q_all && dI_loc && dT_loc && ws, MC_ERR_BAD_ARG,
             "clip_bwd: null pointer");
  ClipProblem p{I_all, T_all, planes_all, b, B, D, row_offset, tau};
  ClipStatsAll s{r_all, c_all, rz_all, g_all, q_all};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  mode = eff_mode(mode, D);
  if (mode == MC_GEMM_SIMT_FP32) return simt::bwd(p, s, grad_loss, dI_loc, dT_loc, ws, ws_bytes, st);
  p.tile_flags = tile_flags;
  return tc::bwd(p, mode, s, grad_loss, dI_loc, dT_loc, ws, ws_bytes, st);
}

int mc_clip_bwd_gate(const uint8_t* tile_flags, size_t n_flags, int* gate_out, void* stream) {
  MC_ARCH_GUARD();
  MC_REQUIRE(tile_flags && n_flags > 0 && gate_out, MC_ERR_BAD_ARG, "clip_bwd_gate: bad argument");
  return tc::bwd_gate(tile_flags, n_flags, gate_out, static_cast<cudaStream_t>(stream));
}

size_t mc_clip_stored_weights_bytes(int b, int B) {
  if (b <= 0 || B <= 0) return 0;
  return tc::stored_weights_bytes(b, B);
}

size_t mc_clip_bwd_cols_workspace_bytes(int n_cols, int D) {
  if (n_cols <= 0 || D <= 0) return 0;
  return tc::bwd_cols_workspace_bytes(0, n_cols, D);
}

int mc_clip_bwd_rows(const void* planes_all, int b, int B, int D, int row_offset, float tau, int mode,
                     const float* r_all, const float* c_all, const float* rz_all, const float* g_all, const float* q_all,
                     const float* grad_loss, float* dT_loc, float* dIz_loc, void* W_loc, const uint8_t* tile_flags,
                     const int* gate, float* dI_loc_ownrows, void* ws, size_t ws_bytes, void* stream) {
  MC_ARCH_GUARD();
  int rc = check_problem("clip_bwd_rows", nullptr, nullptr, b, B, D, row_offset, tau, mode);
  if (rc) return rc;
  MC_REQUIRE(eff_mode(mode, D) != MC_GEMM_SIMT_FP32, MC_ERR_UNSUPPORTED,
             "clip_bwd_rows: the stored-weights form belongs to the tcgen05 engines (mode %d, D %d)", mode, D);
  MC_REQUIRE(planes_all && r_all && c_all && rz_all && g_all && q_all && dT_loc && dIz_loc && W_loc && ws, MC_ERR_BAD_ARG,
             "clip_bwd_rows: null pointer");
  ClipProblem p{nullptr, nullptr, planes_all, b, B, D, row_offset, tau};
  p.tile_flags = tile_flags;
  p.gate = gate;
  ClipStatsAll s{r_all, c_all, rz_all, g_all, q_all};
  return tc::bwd_rows(p, mode, s, grad_loss, dT_loc, dIz_loc, W_loc, ws, ws_bytes, static_cast<cudaStream_t>(stream),
                      dI_loc_ownrows);
}

int mc_clip_bwd_cols(const void* planes_all, int B, int D, float tau, int mode, const float* r_all, const float* c_all,
                     const float* rz_all, const float* q_all, const float* grad_loss, const void* W, int w_rows,
                     int w_row_offset, int j0, int j1, const float* dIz, float* dI_out, const int* gate, void* ws,
                     size_t ws_bytes, void* stream) {
  MC_ARCH_GUARD();
  int rc = check_problem("clip_bwd_cols", nullptr, nullptr, B, B, D, 0, tau, mode);
  if (rc) return rc;
  MC_REQUIRE(eff_mode(mode, D) != MC_GEMM_SIMT_FP32, MC_ERR_UNSUPPORTED,
             "clip_bwd_cols: the stored-weights form belongs to the tcgen05 engines (mode %d, D %d)", mode, D);
  MC_REQUIRE(planes_all && r_all && c_all && rz_all && q_all && W && dI_out && ws, MC_ERR_BAD_ARG, "clip_bwd_cols: null pointer");
  MC_REQUIRE(w_rows > 0 && w_row_offset >= 0 && w_row_offset + w_rows <= B, MC_ERR_BAD_ARG,
             "clip_bwd_cols: stored strip rows %d at %d out of range", w_rows, w_row_offset);
  ClipProblem p{nullptr, nullptr, planes_all, B, B, D, 0, tau};
  p.gate = gate;
  ClipStatsAll s{r_all, c_all, rz_all, nullptr, q_all};
  return tc::bwd_cols(p, mode, s, grad_loss, W, w_rows, w_row_offset, j0, j1, dIz, dI_out, ws, ws_bytes,
                      static_cast<cudaStream_t>(stream));
}

size_t mc_clip_loss_fused_workspace_bytes(int B, int D, int mode) {
  if (B <= 0 || D <= 0) return 0;
  return fused_layout(B, D, mode).total;
}

// The fused single-GPU step.  The gradient sweep runs over `n_strips` row strips (the row-sharded form the ranks of
// a multi-GPU job use, here back to back on one device); `hook`, when given, is called on the host after the loss
// kernels (rows < 0) and after each strip's gradient kernels have been enqueued (row0, rows) - the host-buffer entry
// uses it to start the device -> host copy of a finished strip while the next one is still being swept.
struct StripHook {
  int (*fn)(void* ctx, int row0, int rows, int what);   // what: 1 = dT rows are final, 2 = dI rows, 3 = both
  void* ctx;
};
// MAE_CLIP_HOST_TRACE=1: the host-buffer entry records a timing event after every copy and phase and prints the
// timeline (ms since the call's first event) to stderr - the substitute for an nsys timeline on boxes without it.
namespace {
struct Trace {
  std::vector<std::pair<std::string, cudaEvent_t>> marks;
  void mark(const char* name, int k, cudaStream_t s) {
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, s);
    marks.emplace_back(k >= 0 ? std::string(name) + "[" + std::to_string(k) + "]" : std::string(name), e);
  }
  void dump() {
    if (marks.empty()) return;
    cudaEventSynchronize(marks.back().second);
    for (auto& m : marks) {
      cudaEventSynchronize(m.second);
      float ms = 0.f;
      cudaEventElapsedTime(&ms, marks.front().second, m.second);
      fprintf(stderr, "[mc trace] %8.3f ms  %s\n", ms, m.first.c_str());
      }
    for (auto& m : marks) cudaEventDestroy(m.second);
    marks.clear();
  }
};
thread_local Trace* g_trace = nullptr;
inline void trace_mark(const char* name, int k, cudaStream_t s) { if (g_trace) g_trace->mark(name, k, s); }
}  // namespace

// `feed`, when given: the batch is still arriving from the host in `chunks` row chunks (event k = rows of chunk k are in
// device memory); staging and the statistics sweep then run chunk by chunk behind the copy (tc::prepare_chunk,
// tc::stats_chunk) instead of waiting for the whole batch.
struct ChunkFeed {
  int chunks;
  const cudaEvent_t* arrived;
  unsigned int* words;  // {true max so far, scale slot, bad flag} in device memory
};
static int fused_run(const float* I, const float* T, int B, int D, float tau, int mode, float* loss_out, float* dI,
                     float* dT, void* ws, size_t ws_bytes, void* stream, int n_strips, const StripHook* hook,
                     const ChunkFeed* feed = nullptr, double last_frac = 0.0) {
  int rc = check_problem("clip_loss_fwd_bwd", I, T, B, B, D, 0, tau, mode);
  if (rc) return rc;
  MC_REQUIRE(loss_out && ws, MC_ERR_BAD_ARG, "clip_loss_fwd_bwd: null loss_out/workspace");
  MC_REQUIRE((dI == nullptr) == (dT == nullptr), MC_ERR_BAD_ARG,
             "clip_loss_fwd_bwd: pass both dI and dT or neither");
  FusedLayout l = fused_layout(B, D, mode);
  MC_REQUIRE(ws_bytes >= l.total, MC_ERR_WORKSPACE, "clip_loss_fwd_bwd: workspace %zu < %zu",
             ws_bytes, l.total);
  char* base = static_cast<char*>(ws);
  float* r = reinterpret_cast<float*>(base + l.off_vec + 0 * l.vec_stride);
  float* c = reinterpret_cast<float*>(base + l.off_vec + 1 * l.vec_stride);
  float* rz = reinterpret_cast<float*>(base + l.off_vec + 2 * l.vec_stride);
  float* g = reinterpret_cast<float*>(base + l.off_vec + 3 * l.vec_stride);
  float* q = reinterpret_cast<float*>(base + l.off_vec + 4 * l.vec_stride);
  float* ps = reinterpret_cast<float*>(base + l.off_vec + 5 * l.vec_stride);
  void* planes = base + l.off_planes;
  void* phase = base + l.off_phase;
  size_t phase_bytes = l.phase_bytes;
  // tile flags: the statistics sweep marks the tiles that carry soft-target mass; the later sweeps skip the rest
  // (MAE_CLIP_DENSE=1 keeps every tile: the A/B switch)
  static const bool dense = getenv("MAE_CLIP_DENSE") != nullptr && getenv("MAE_CLIP_DENSE")[0] == '1';
  uint8_t* flags_raw = (l.flags_bytes && !dense) ? reinterpret_cast<uint8_t*>(base + l.off_flags) : nullptr;
  uint8_t* flags = flags_raw ? flags_raw + l.flags_bytes : nullptr;
  if (feed) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int emode = eff_mode(mode, D), chunk_rows = B / feed->chunks;
    ClipProblem p{I, T, planes, B, B, D, 0, tau};
    p.tile_flags_out = flags_raw;
    MC_CUDA(cudaMemsetAsync(feed->words, 0, 3 * sizeof(unsigned int), st));
    if ((rc = tc::stats_begin(p, st))) return rc;
    for (int k = 0; k < feed->chunks; ++k) {
      MC_CUDA(cudaStreamWaitEvent(st, feed->arrived[k], 0));
      if ((rc = tc::prepare_chunk(I, T, B, D, k * chunk_rows, chunk_rows, planes, feed->words, st))) return rc;
      trace_mark("staged", k, st);
      if ((rc = tc::stats_chunk(p, emode, k, feed->chunks, phase, st))) return rc;
      trace_mark("stats", k, st);
    }
    if ((rc = tc::verify_scale(feed->words, st))) return rc;
    if ((rc = tc::stats_end(p, emode, feed->chunks, r, c, rz, ps, phase, st))) return rc;
    trace_mark("stats_end", -1, st);
  } else {
    if ((rc = mc_clip_prepare(I, T, B, B, D, 0, mode, planes, stream))) return rc;
    trace_mark("staged", -1, static_cast<cudaStream_t>(stream));
    if ((rc = mc_clip_stats(I, T, planes, B, B, D, 0, tau, mode, r, c, rz, ps, flags_raw, phase, phase_bytes, stream)))
      return rc;
    trace_mark("stats", -1, static_cast<cudaStream_t>(stream));
  }
  if (flags_raw && (rc = mc_clip_flags_finalize(flags_raw, B, B, 0, flags, stream))) return rc;
  if ((rc = mc_clip_rowloss(I, T, planes, B, B, D, 0, tau, mode, r, c, rz, ps, g, q, loss_out, flags, phase,
                            phase_bytes, stream)))
    return rc;
  trace_mark("rowloss", -1, static_cast<cudaStream_t>(stream));
  if (hook && (rc = hook->fn(hook->ctx, -1, 0, 0))) return rc;
  if (!dI) return MC_OK;
  // strips of whole 128-row blocks; a strip whose partial-sum workspace would not fit the step's buffer (more
  // column splits per row block) folds the sweep back into one launch.  last_frac > 0: the LAST strip takes that share
  // of the row blocks and the others split the rest evenly (the host-buffer entry: only the last strip's copy back to
  // the host is exposed, so it is the short one).
  const int n_blocks = (B + 127) / 128;
  if (n_strips > n_blocks) n_strips = n_blocks;
  if (n_strips < 1) n_strips = 1;
  int strip_first[17];
  {
    int last = (last_frac > 0.0 && n_strips > 1) ? (int)(n_blocks * last_frac + 0.5) : 0;
    if (last < 1 || last > n_blocks - (n_strips - 1)) last = 0;
    const int head = last ? n_strips - 1 : n_strips, head_blocks = n_blocks - last;
    const int per = (head_blocks + head - 1) / head;
    for (int k = 0; k < head; ++k) strip_first[k] = k * per < head_blocks ? k * per : head_blocks;
    strip_first[head] = head_blocks;
    strip_first[n_strips] = n_blocks;
  }
  for (int k = 0; k < n_strips && n_strips > 1; ++k) {
    const int rows_k = (strip_first[k + 1] - strip_first[k]) * 128;
    if (rows_k <= 0 || mc_clip_loss_workspace_bytes(rows_k, B, D, mode) > phase_bytes) n_strips = 1;
  }
  const int n_tiles = n_blocks;  // column tiles of B = row blocks of B
  int last_strip_rows = B;
  // the stored-weights form needs tile flags (its dense kernel computes the softmax part only) and a tcgen05 engine
  // (tc_f16x3 or tc_f16: rowgrad_kernel runs three passes or one); which form actually runs is decided on the device
  // from the flag density (tc::bwd_gate)
  const bool stored = l.off_w != 0 && flags != nullptr && eff_mode(mode, D) != MC_GEMM_SIMT_FP32;
  int* gate = nullptr;
  if (stored) {
    gate = reinterpret_cast<int*>(base + l.off_vec + 6 * l.vec_stride);
    if ((rc = tc::bwd_gate(flags, tc::tile_flags_bytes(B, B), gate, static_cast<cudaStream_t>(stream)))) return rc;
  }
  const int Bp = n_blocks * 128;
  for (int k = 0; k < n_strips; ++k) {
    const int row0 = n_strips == 1 ? 0 : strip_first[k] * 128;
    const int rows = n_strips == 1 ? B : (strip_first[k + 1] * 128 <= B ? strip_first[k + 1] * 128 : B) - row0;
    const uint8_t* fl = flags ? flags + (size_t)(row0 / 128) * n_tiles : nullptr;
    if (stored) {
      // row half: dT of the strip is final; the strip's weights and the soft-target part of its dI wait for the column half
      ClipProblem p{I, T, planes, rows, B, D, row0, tau};
      p.tile_flags = fl;
      p.gate = gate;
      ClipStatsAll s{r, c, rz, g, q};
      if ((rc = tc::bwd_rows(p, eff_mode(mode, D), s, nullptr, dT + (size_t)row0 * D,
                             reinterpret_cast<float*>(base + l.off_diz) + (size_t)row0 * D,
                             base + l.off_w + (size_t)row0 * Bp * 2, phase, phase_bytes,
                             static_cast<cudaStream_t>(stream), dI + (size_t)row0 * D)))
        return rc;
      last_strip_rows = rows;
      trace_mark("bwd rows strip", k, static_cast<cudaStream_t>(stream));
      if (hook && (rc = hook->fn(hook->ctx, row0, rows, 1))) return rc;
    } else {
      if ((rc = mc_clip_bwd(I, T, planes, rows, B, D, row0, tau, mode, r, c, rz, g, q, nullptr, dI + (size_t)row0 * D,
                            dT + (size_t)row0 * D, fl, phase, phase_bytes, stream)))
        return rc;
      trace_mark("bwd strip", k, static_cast<cudaStream_t>(stream));
      if (hook && (rc = hook->fn(hook->ctx, row0, rows, 3))) return rc;
    }
  }
  if (stored) {
    // column half, in as many strips of output rows as the row half had (the host entry copies a finished strip back
    // while the next is computed)
    ClipProblem p{I, T, planes, B, B, D, 0, tau};
    p.gate = gate;
    ClipStatsAll s{r, c, rz, g, q};
    for (int k = 0; k < n_strips; ++k) {
      const int j0 = n_strips == 1 ? 0 : strip_first[k] * 128;
      const int j1 = n_strips == 1 ? B : (strip_first[k + 1] * 128 <= B ? strip_first[k + 1] * 128 : B);
      if ((rc = tc::bwd_cols(p, eff_mode(mode, D), s, nullptr, base + l.off_w, B, 0, j0, j1,
                             reinterpret_cast<const float*>(base + l.off_diz) + (size_t)j0 * D, dI + (size_t)j0 * D,
                             base + l.off_cols, l.cols_bytes, static_cast<cudaStream_t>(stream),
                             tc::bwd_rows_wscale(phase, last_strip_rows, B, D))))
        return rc;
      trace_mark("bwd cols strip", k, static_cast<cudaStream_t>(stream));
      if (hook && (rc = hook->fn(hook->ctx, j0, j1 - j0, 2))) return rc;
    }
  }
  return MC_OK;
}

int mc_clip_loss_fwd_bwd(const float* I, const float* T, int B, int D, float tau, int mode,
                         float* loss_out, float* dI, float* dT, void* ws, size_t ws_bytes,
                         void* stream) {
  MC_ARCH_GUARD();
  return fused_run(I, T, B, D, tau, mode, loss_out, dI, dT, ws, ws_bytes, stream, 1, nullptr);
}

size_t mc_clip_loss_host_workspace_bytes(int B, int D, int mode) {
  if (B <= 0 || D <= 0) return 0;
  size_t emb = round_up((size_t)B * D * 4, 256);
  return 4 * emb + 256 + fused_layout(B, D, mode).total;
}

// Host-buffer form.  Gradients leave the device strip by strip: a second stream copies the rows of a finished strip
// while the next strip is being swept, so of the 2 B D 4 bytes going back only the last strip's share is exposed.
namespace {
struct HostCopyCtx {
  cudaStream_t st, copy;
  cudaEvent_t ev[16];
  int n_ev;
  const float *loss_dev, *gI, *gT;
  float *loss_host, *dI_host, *dT_host;
  int D;
  bool want_grad;
};
int host_copy_hook(void* vctx, int row0, int rows, int what) {
  HostCopyCtx* c = static_cast<HostCopyCtx*>(vctx);
  if (rows <= 0 || row0 < 0) {  // after the loss kernels
    MC_CUDA(cudaMemcpyAsync(c->loss_host, c->loss_dev, 4, cudaMemcpyDeviceToHost, c->st));
    return MC_OK;
  }
  if (!c->want_grad) return MC_OK;
  const size_t off = (size_t)row0 * c->D, bytes = (size_t)rows * c->D * 4;
  MC_REQUIRE(c->n_ev < 16, MC_ERR_BAD_ARG, "clip_loss_host: too many strips");
  cudaEvent_t ev = c->ev[c->n_ev++];
  MC_CUDA(cudaEventRecord(ev, c->st));
  MC_CUDA(cudaStreamWaitEvent(c->copy, ev, 0));
  if (what & 1) MC_CUDA(cudaMemcpyAsync(c->dT_host + off, c->gT + off, bytes, cudaMemcpyDeviceToHost, c->copy));
  if (what & 2) MC_CUDA(cudaMemcpyAsync(c->dI_host + off, c->gI + off, bytes, cudaMemcpyDeviceToHost, c->copy));
  trace_mark("d2h strip done", c->n_ev - 1, c->copy);
  return MC_OK;
}
// one copy stream per device, created on first use and kept (callers on different threads may share it: every
// copy is ordered by the caller's own events)
int copy_stream_for_current_device(cudaStream_t* out) {
  static std::mutex mu;
  static cudaStream_t streams[64] = {};
  int dev = 0;
  MC_CUDA(cudaGetDevice(&dev));
  MC_REQUIRE(dev >= 0 && dev < 64, MC_ERR_BAD_ARG, "clip_loss_host: device index %d", dev);
  std::lock_guard<std::mutex> lk(mu);
  if (!streams[dev]) MC_CUDA(cudaStreamCreateWithFlags(&streams[dev], cudaStreamNonBlocking));
  *out = streams[dev];
  return MC_OK;
}
}  // namespace

int mc_clip_loss_fwd_bwd_host(const float* I_host, const float* T_host, int B, int D, float tau,
                              int mode, float* loss_host, float* dI_host, float* dT_host, void* dws,
                              size_t dws_bytes, void* stream) {
  MC_ARCH_GUARD();
  MC_REQUIRE(I_host && T_host && loss_host && dws, MC_ERR_BAD_ARG, "clip_loss_host: null pointer");
  MC_REQUIRE(B > 0 && D > 0, MC_ERR_BAD_ARG, "clip_loss_host: bad sizes");
  MC_REQUIRE(dws_bytes >= mc_clip_loss_host_workspace_bytes(B, D, mode), MC_ERR_WORKSPACE,
             "clip_loss_host: device workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  size_t emb = round_up((size_t)B * D * 4, 256);
  char* base = static_cast<char*>(dws);
  float* dIin = reinterpret_cast<float*>(base);
  float* dTin = reinterpret_cast<float*>(base + emb);
  float* gI = reinterpret_cast<float*>(base + 2 * emb);
  float* gT = reinterpret_cast<float*>(base + 3 * emb);
  float* loss = reinterpret_cast<float*>(base + 4 * emb);
  void* ws = base + 4 * emb + 256;
  size_t ws_bytes = dws_bytes - (4 * emb + 256);
  size_t bytes = (size_t)B * D * 4;
  const bool want_grad = dI_host && dT_host;
  // two strips where a strip still fills the machine (>= 8192 rows: 64 row blocks x column splits) and the tcgen05
  // engine runs; small batches and the SIMT engine keep the single sweep.  Measured at B = 32768 (tools/e2e_strips.py,
  // profiles/r01i_e2e_strips.json): 1 strip 9.52 ms, 2: 9.20, 3: 9.81, 4: 9.31, 6: 9.21, 8: 10.5 - every strip adds a
  // partly filled last wave and its own finalize, which eats the shorter exposed copy beyond two
  int n_strips = 1;
  if (want_grad && eff_mode(mode, D) != MC_GEMM_SIMT_FP32 && B >= 16384) n_strips = 2;
  if (const char* e = getenv("MAE_CLIP_HOST_STRIPS")) {  // A/B switch (1 = the single sweep + one copy at the end)
    const int v = atoi(e);
    if (want_grad && v >= 1 && v <= 8 && eff_mode(mode, D) != MC_GEMM_SIMT_FP32) n_strips = v;
  }
  // share of the row blocks the LAST strip takes (0 = equal strips).  A short last strip shortens the exposed copy,
  // but measured at B = 32768 (tools/e2e_trace.py, profiles/r02k_e2e_trace.log) the two sweeps of an uneven split
  // lose more to their partly filled last rounds (3/4 + 1/4: 2.99 + 1.11 ms against 1.91 + 1.92) than the copy gains
  double last_frac = 0.0;
  if (const char* e = getenv("MAE_CLIP_HOST_LAST_STRIP")) {
    const double v = atof(e);
    if (v >= 0.0 && v < 1.0) last_frac = v;
  }
  // row chunks of the inbound copy (MAE_CLIP_HOST_CHUNKS, 1 = copy everything, then stage): with the batch arriving
  // in pieces, staging and the statistics sweep of the rows that have landed run behind the rest of the copy.  The
  // planes share one power-of-two scale, which the first chunk fixes with a binade of headroom; a batch whose later
  // rows exceed it is detected on the device (tc::verify_scale) and the step is redone from the resident copy.
  // Measured at B = 32768 with the current kernels (tools/e2e_strips.py, profiles/r02ag_e2e_strips.json; chunks x strips):
  // 1x1 5.73 ms, 2x2 5.28, 4x2 5.09, 4x3 5.06, 8x2 5.15, 16x2 5.51 - four chunks from 32768 rows on, two from 8192.
  int chunks = (eff_mode(mode, D) != MC_GEMM_SIMT_FP32 && B >= 8192) ? (B >= 32768 ? 4 : 2) : 1;
  if (const char* e = getenv("MAE_CLIP_HOST_CHUNKS")) {
    const int v = atoi(e);
    if (v >= 1 && v <= 16) chunks = v;
  }
  if (chunks > 1 && !(eff_mode(mode, D) != MC_GEMM_SIMT_FP32 && tc::stats_chunkable(B, D, chunks))) chunks = 1;
  unsigned int* words = reinterpret_cast<unsigned int*>(base + 4 * emb + 16);
  HostCopyCtx ctx = {};
  ctx.st = st; ctx.D = D; ctx.want_grad = want_grad;
  ctx.loss_dev = loss; ctx.gI = gI; ctx.gT = gT;
  ctx.loss_host = loss_host; ctx.dI_host = dI_host; ctx.dT_host = dT_host;
  int rc = MC_OK;
  cudaEvent_t done = nullptr, arrived[17] = {};
  int n_created = 0, n_arrived = 0;
  auto destroy_all = [&]() {
    for (int i = 0; i < n_created; ++i) cudaEventDestroy(ctx.ev[i]);
    for (int i = 0; i < n_arrived; ++i) cudaEventDestroy(arrived[i]);
    if (done) cudaEventDestroy(done);
  };
  if (want_grad || chunks > 1) {
    if ((rc = copy_stream_for_current_device(&ctx.copy))) return rc;
    bool ok = true;
    for (; ok && want_grad && n_created < 2 * n_strips; ++n_created)   // row half + column half of every strip
      if (cudaEventCreateWithFlags(&ctx.ev[n_created], cudaEventDisableTiming) != cudaSuccess) { ok = false; break; }
    const int want_arrived = chunks > 1 ? chunks + 1 : 0;  // + the "stream is free" event the copy stream waits for
    for (; ok && n_arrived < want_arrived; ++n_arrived)
      if (cudaEventCreateWithFlags(&arrived[n_arrived], cudaEventDisableTiming) != cudaSuccess) { ok = false; break; }
    if (ok && cudaEventCreateWithFlags(&done, cudaEventDisableTiming) != cudaSuccess) ok = false;
    if (!ok) {
      destroy_all();
      MC_REQUIRE(false, MC_ERR_CUDA, "clip_loss_host: cudaEventCreate failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
  }
  auto body = [&]() -> int {
    StripHook hook{host_copy_hook, &ctx};
    float* gIo = want_grad ? gI : nullptr;
    float* gTo = want_grad ? gT : nullptr;
    auto finish = [&]() -> int {
      if (want_grad) {
        MC_CUDA(cudaEventRecord(done, ctx.copy));
        MC_CUDA(cudaStreamWaitEvent(st, done, 0));
      }
      MC_CUDA(cudaStreamSynchronize(st));
      return MC_OK;
    };
    int r2;
    if (chunks > 1) {
      // the copy stream may not overwrite the inbound buffers before earlier work on the caller's stream is done
      MC_CUDA(cudaEventRecord(arrived[chunks], st));
      MC_CUDA(cudaStreamWaitEvent(ctx.copy, arrived[chunks], 0));
      const size_t crow = (size_t)(B / chunks) * D;
      for (int k = 0; k < chunks; ++k) {
        MC_CUDA(cudaMemcpyAsync(dTin + k * crow, T_host + k * crow, crow * 4, cudaMemcpyHostToDevice, ctx.copy));
        MC_CUDA(cudaMemcpyAsync(dIin + k * crow, I_host + k * crow, crow * 4, cudaMemcpyHostToDevice, ctx.copy));
        MC_CUDA(cudaEventRecord(arrived[k], ctx.copy));
        trace_mark("h2d chunk arrived", k, ctx.copy);
      }
      ChunkFeed feed{chunks, arrived, words};
      if ((r2 = fused_run(dIin, dTin, B, D, tau, mode, loss, gIo, gTo, ws, ws_bytes, stream, n_strips, &hook, &feed, last_frac)))
        return r2;
      if ((r2 = finish())) return r2;
      unsigned int bad = 0;
      MC_CUDA(cudaMemcpy(&bad, words + 2, sizeof(bad), cudaMemcpyDeviceToHost));
      if (!bad) return MC_OK;
      ctx.n_ev = 0;  // rare: a later chunk outgrew the first chunk's scale - redo from the resident fp32 copy
    } else {
      MC_CUDA(cudaMemcpyAsync(dTin, T_host, bytes, cudaMemcpyHostToDevice, st));
      MC_CUDA(cudaMemcpyAsync(dIin, I_host, bytes, cudaMemcpyHostToDevice, st));
      trace_mark("h2d arrived", -1, st);
    }
    if ((r2 = fused_run(dIin, dTin, B, D, tau, mode, loss, gIo, gTo, ws, ws_bytes, stream, n_strips, &hook, nullptr, last_frac)))
      return r2;
    return finish();
  };
  Trace trace;
  const bool tracing = getenv("MAE_CLIP_HOST_TRACE") != nullptr && getenv("MAE_CLIP_HOST_TRACE")[0] == '1';
  if (tracing) { g_trace = &trace; trace.mark("call", -1, st); }
  rc = body();
  if (tracing) { trace.mark("end", -1, st); trace.dump(); g_trace = nullptr; }
  if (rc && ctx.copy) cudaStreamSynchronize(ctx.copy);  // nothing of this call may still be in flight
  destroy_all();
  return rc;
}

}  // extern "C"

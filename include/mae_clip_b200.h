/*
 * mae_clip_b200 - C ABI of the B200-native training-loss hot path.
 *
 * The reference (ykojima4020/mae_clip) is pure Python and has no FFI of its
 * own; its boundary is the Python API (CLIPModel.forward / ProjectionHead /
 * cross_entropy).  This header is the NEW C boundary that sits directly
 * underneath that API: each entry point names the reference lines whose
 * arithmetic it replaces.  INTEGRATION.md shows the ctypes stub a maintainer
 * of the reference would add.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *  - tensors are dense row-major unless strides are passed explicitly;
 *  - `stream` is a cudaStream_t passed as void* (0 = default stream);
 *  - no entry point on the step path allocates device memory: scratch comes
 *    in through `ws`/`ws_bytes`, sized by the matching `*_workspace_bytes`
 *    query (the one exception is the set-up call mc_peer_alloc, which creates
 *    the exchange region other processes map);
 *  - every entry point returns an mc_status (0 = ok) and never throws;
 *    mc_last_error_string() describes the last failure on the calling thread;
 *  - entry points are re-entrant; the library keeps no mutable global state
 *    except cached TMA descriptors keyed by (pointer, shape).
 *  - the library refuses to run on anything but compute capability 10.x
 *    (MC_ERR_ARCH); there is no fallback path.
 */
#ifndef MAE_CLIP_B200_H_
#define MAE_CLIP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  MC_OK = 0,
  MC_ERR_BAD_ARG = 1,     /* null pointer, non-positive size, unsupported shape */
  MC_ERR_ALIGN = 2,       /* pointer not aligned for the vector width used      */
  MC_ERR_ARCH = 3,        /* device is not sm_100                               */
  MC_ERR_CUDA = 4,        /* a CUDA runtime / driver call failed                */
  MC_ERR_WORKSPACE = 5,   /* ws_bytes smaller than *_workspace_bytes()          */
  MC_ERR_UNSUPPORTED = 6  /* valid request this build does not implement        */
} mc_status;

/* precision / engine of the contrastive-loss and projection GEMMs */
typedef enum {
  MC_GEMM_SIMT_FP32 = 0, /* plain fp32 FMA tiles (bring-up / cross-check path)            */
  MC_GEMM_TC_F16X3 = 1, /* tcgen05 kind::f16, operands split into fp16 hi + lo planes, 3 passes
                            (hi*hi + hi*lo + lo*hi): ~2^-22 relative operand error, fp32 accumulate:
                            meets the fp32 tolerance                                       */
  MC_GEMM_TC_F16 = 2    /* tcgen05 kind::f16, single fp16 pass (looser, stated tolerance)  */
} mc_gemm_mode;

int mc_version(void);                       /* major*10000 + minor*100 + patch */
const char* mc_last_error_string(void);
int mc_device_supported(int device);        /* 1 when `device` is compute capability 10.x */
/* kernels launched by this library since load (process-wide, monotonic): callers difference it
 * around a region to count launches */
unsigned long long mc_kernel_launch_count(void);

/* ---------------------------------------------------------------------------
 * L5  cross_entropy(preds, targets, reduction)            CLIP.py:46-52
 * loss_rows[r] = -sum_c targets[r,c] * log_softmax(preds[r,:])[c]
 * Strides are in elements so the transposed views of CLIP.py:41 are accepted
 * without a copy.  row_lse / row_tsum (rows floats each) are kept for backward.
 * ------------------------------------------------------------------------- */
/* ws: optional scratch of mc_soft_ce_workspace_bytes(rows, cols) (0 for small problems); with it the
 * transposed-view forward splits the columns over more blocks (NULL / too small: single-kernel form). */
size_t mc_soft_ce_workspace_bytes(int rows, int cols);
int mc_soft_ce_fwd(const float* preds, int64_t p_row_stride, int64_t p_col_stride,
                   const float* targets, int64_t t_row_stride, int64_t t_col_stride,
                   int rows, int cols, float* loss_rows, float* row_lse, float* row_tsum,
                   void* ws, size_t ws_bytes, void* stream);
/* dpreds / dtargets (either may be NULL) are written through their own element strides, so the
 * caller can give them the layout of the (possibly transposed) inputs and keep stores coalesced. */
int mc_soft_ce_bwd(const float* preds, int64_t p_row_stride, int64_t p_col_stride,
                   const float* targets, int64_t t_row_stride, int64_t t_col_stride,
                   int rows, int cols, const float* row_lse, const float* row_tsum,
                   const float* grad_rows, float* dpreds, int64_t dp_row_stride,
                   int64_t dp_col_stride, float* dtargets, int64_t dt_row_stride,
                   int64_t dt_col_stride, void* stream);

/* ---------------------------------------------------------------------------
 * L3-L6  contrastive soft-target loss on embeddings        CLIP.py:34-43 (+ autograd, main.py:58)
 *
 * Rows are partitioned: this rank owns `b` rows of the global batch `B`
 * starting at `row_offset`; *_loc pointers have b rows/entries, *_all have B.
 * On one GPU b == B, row_offset == 0 and loc == all.  Three phases, each one
 * sweep over the (b x B) strip; the caller all-gathers the small statistic
 * vectors between phases when B > b (mae_clip_b200/dist.py).
 *
 *   stats  : row_lse_s[i] = LSE_j S_ij,  col_lse_s[i] = LSE_j S_ji,
 *            row_lse_z[i] = LSE_j Z_ij            (S = T I^T / tau, Z = (I I^T + T T^T) tau/2)
 *            row_ps[i]    = sum_j P_ij S_ij       (accumulated online; lets the next sweep skip S)
 *   rowloss: row_g[i] = sum_j P_ij G_ij, col_sum_p[i] = sum_k P_ki, loss_part = sum_i row_g[i]
 *            (P = softmax_row(Z), G = -(2S - r_i - c_j)/(2B); loss = sum over ranks of loss_part)
 *   bwd    : dI_loc, dT_loc = grad_loss * d loss / d (I_loc, T_loc), every term of the owned rows
 *            (the strip of dS, the transposed strip of dS and dZ + dZ^T), so no gradient
 *            exchange is needed afterwards.
 * ------------------------------------------------------------------------- */
size_t mc_clip_loss_workspace_bytes(int b, int B, int D, int mode);

/* prepare(): mode-specific operand staging (fp16 hi/lo planes for the tcgen05 modes; no-op for
 * SIMT).  `planes_all` receives the staged copy of the *local* rows at row_offset; when B > b the
 * caller all-gathers the planes instead of the fp32 embeddings.  planes layout: see DESIGN.md. */
size_t mc_clip_planes_bytes(int B, int D, int mode);
int mc_clip_prepare(const float* I_loc, const float* T_loc, int b, int B, int D, int row_offset,
                    int mode, void* planes_all, void* stream);

/* Peer-memory staging for the row-sharded loss (one process per GPU; tcgen05 modes only): the
 * embedding all-gather is fused into prepare.  mc_clip_amax() reduces this rank's shards to the
 * bit pattern of their largest magnitude (and optionally copies them into the exchange region);
 * after every rank's value has been published into `amax_slots` (world words, see
 * mc_peer_publish / mc_peer_barrier) mc_clip_prepare_peers() pulls each global row from its
 * owner - I_peers_host[q] / T_peers_host[q] are HOST arrays of `world` device pointers to rank
 * q's (b, D) fp32 shards, mapped on this device - and writes the local planes of all world*b rows.
 * I_all / T_all of the three phases below may then be NULL.
 * mc_clip_push_shards() is the push form of the same exchange: this rank's shards are stored into
 * rows [rank*b, (rank+1)*b) of EVERY rank's (world*b, D) fp32 image (I_all_dst_host[q] /
 * T_all_dst_host[q]: HOST arrays of the images' base pointers) with posted NVLink stores while the
 * local amax is reduced; the last block publishes it into amax_slots_host[q][rank].  `scratch`:
 * two zero-initialised device words private to this rank (re-armed by the kernel).  After a
 * barrier, mc_clip_prepare_peers() is called with every I_peers_host[q] pointing into the LOCAL
 * image. */
int mc_clip_push_shards(const float* I_loc, const float* T_loc, int b, int D, int rank, int world,
                        float* const* I_all_dst_host, float* const* T_all_dst_host,
                        unsigned int* const* amax_slots_host, unsigned int* scratch, void* stream);
int mc_clip_amax(const float* I_loc, const float* T_loc, int b, int D, float* I_copy, float* T_copy,
                 unsigned int* amax_bits, void* stream);
int mc_clip_prepare_peers(const float* const* I_peers_host, const float* const* T_peers_host, int world,
                          int b, int D, int mode, const unsigned int* amax_slots, void* planes_all,
                          void* stream);

/* Tile flags (tcgen05 engines; optional).  The soft targets P = softmax_row(Z) are usually concentrated (for
 * LayerNorm-ed embeddings Z_ii = 256 tau/2 towers over the off-diagonal entries), so most 128 x 128 tiles hold no
 * P_ij above 2^-44.  When mc_clip_stats is given a flag array it runs as a PROBE (S, S^T at full precision, Z from
 * the hi planes only) that records, per (row block of 128, column tile of 128), whether the tile's largest Z_ij
 * comes within 44 binades (plus the probe's worst-case rounding bound) of Z_ii <= rz_i - a rigorous superset of "some
 * P_ij >= 2^-44" - and then computes the exact Z statistics on the flagged tiles only.  mc_clip_flags_finalize ORs that with the transposed relation (P_ji, by the symmetry of Z) from
 * the flags of ALL row blocks (the caller gathers them over ranks: [B/128][B/128] bytes).  mc_clip_rowloss then
 * visits flagged tiles only and mc_clip_bwd skips the Z recompute and the dZ GEMMs elsewhere; the dropped terms
 * sum to < B 2^-44 per row.  NULL pointers = dense (every tile).  mc_clip_tile_flags_bytes: size of the
 * per-rank array (0 when the engine is the fp32 FMA one). */
size_t mc_clip_tile_flags_bytes(int b, int B, int D, int mode);
int mc_clip_flags_finalize(const uint8_t* flags_all, int B, int b, int row_offset, uint8_t* flags_loc,
                           void* stream);

int mc_clip_stats(const float* I_all, const float* T_all, const void* planes_all, int b, int B,
                  int D, int row_offset, float tau, int mode, float* row_lse_s_loc,
                  float* col_lse_s_loc, float* row_lse_z_loc, float* row_ps_loc,
                  uint8_t* tile_flags_loc_out, void* ws, size_t ws_bytes, void* stream);
/* Column-partials form of the statistics sweep (tcgen05 engines).  mc_clip_stats obtains the column LSE of S for the
 * owned indices from a second, transposed strip of logits (3 more tensor-core passes per tile).  Here the transposed
 * strip is not computed: every epilogue warp reduces its 32 x 32 block of S along the rows in registers (exact:
 * exponentials against each column's own maximum) and the sweep returns, for EVERY column j of the global batch,
 *     col_lse_part_all[j] = log sum_{i in the owned rows} exp(S_ij)            (B floats).
 * The ranks exchange these vectors and mc_clip_colpart_merge folds them: col_lse_all[j] = log sum_q exp(parts[q][j])
 * (parts: n_parts vectors, `stride` floats apart).  With b == B mc_clip_stats uses this form by itself
 * (MAE_CLIP_COLPART=0 restores the transposed strip). */
size_t mc_clip_stats_colpart_workspace_bytes(int b, int B, int D, int mode);
int mc_clip_stats_colpart(const void* planes_all, int b, int B, int D, int row_offset, float tau, int mode,
                          float* row_lse_s_loc, float* col_lse_part_all, float* row_lse_z_loc,
                          float* row_ps_loc, uint8_t* tile_flags_loc_out, void* ws, size_t ws_bytes,
                          void* stream);
int mc_clip_colpart_merge(const float* parts, int n_parts, int64_t stride, int B, float* col_lse_all,
                          void* stream);

int mc_clip_rowloss(const float* I_all, const float* T_all, const void* planes_all, int b, int B,
                    int D, int row_offset, float tau, int mode, const float* row_lse_s_all,
                    const float* col_lse_s_all, const float* row_lse_z_all, const float* row_ps_loc,
                    float* row_g_loc, float* col_sum_p_loc, float* loss_part,
                    const uint8_t* tile_flags_loc, void* ws, size_t ws_bytes, void* stream);
int mc_clip_bwd(const float* I_all, const float* T_all, const void* planes_all, int b, int B, int D,
                int row_offset, float tau, int mode, const float* row_lse_s_all,
                const float* col_lse_s_all, const float* row_lse_z_all, const float* row_g_all,
                const float* col_sum_p_all, const float* grad_loss /* device scalar or NULL = 1 */,
                float* dI_loc, float* dT_loc, const uint8_t* tile_flags_loc, void* ws, size_t ws_bytes,
                void* stream);

/* Stored-weights form of the gradient (tcgen05 engines).  mc_clip_bwd keeps every gradient term of the owned rows
 * local by recomputing the transposed strip of logits (8 GEMM units per tile pair).  The stored form computes S once:
 *   mc_clip_bwd_rows  S = T_i I_j^T over the owned strip -> dT_loc (final), the fp16 weight strip W (b x B:
 *                     w_ij = 2B dS_ij x a power-of-two scale) and dIz_loc, the un-scaled soft-target (dZ) part of dI
 *                     of the owned rows;
 *   mc_clip_bwd_cols  dI_j = scale (dIz_j + sum_i w_ij T_i) for the rows j0 .. j1 of the GLOBAL batch from a stored
 *                     strip (w_rows rows starting at global row w_row_offset) - W is read transposed by the tensor
 *                     cores (MN-major operand), nothing is transposed in memory.  dIz NULL = W part only.
 * 5 GEMM units per tile pair instead of 8, at the price of b x B fp16 of HBM and, under row sharding, a reduce of the
 * ranks' (B x D) partial dI (dist.PeerStep does it over peer memory).  A call that owns every row (b == B) takes this
 * form inside mc_clip_bwd already (its workspace size includes the buffers); MAE_CLIP_BWD_FORM=ownrows switches it off.
 * Sizes: W = mc_clip_stored_weights_bytes(b, B); mc_clip_bwd_rows needs the workspace of mc_clip_loss_workspace_bytes
 * for a strip (b < B) and W 256-byte aligned; mc_clip_bwd_cols needs mc_clip_bwd_cols_workspace_bytes(j1 - j0, D). */
size_t mc_clip_stored_weights_bytes(int b, int B);
size_t mc_clip_bwd_cols_workspace_bytes(int n_cols, int D);
/* The stored form pays while the soft targets are concentrated (few flagged tiles); with many flagged tiles the
 * own-rows sweep is cheaper.  mc_clip_bwd_gate writes the choice into a device word from the flags of ALL row blocks
 * (1 = stored, 0 = own rows; break-even at 15% flagged tiles, MAE_CLIP_BWD_GATE overrides); given that word, the calls
 * below enqueue the kernels of BOTH forms and the ones of the other form return at once - no host synchronisation.
 * gate NULL = the stored form unconditionally.  A gated mc_clip_bwd_rows needs tile flags and
 * dI_loc_ownrows (where the own-rows form writes this strip's dI); mc_peer_reduce takes the same word. */
int mc_clip_bwd_gate(const uint8_t* tile_flags_all, size_t n_flags, int* gate_out, void* stream);
int mc_clip_bwd_rows(const void* planes_all, int b, int B, int D, int row_offset, float tau, int mode,
                     const float* row_lse_s_all, const float* col_lse_s_all, const float* row_lse_z_all,
                     const float* row_g_all, const float* col_sum_p_all, const float* grad_loss, float* dT_loc,
                     float* dIz_loc, void* W_loc, const uint8_t* tile_flags_loc, const int* gate,
                     float* dI_loc_ownrows, void* ws, size_t ws_bytes, void* stream);
int mc_clip_bwd_cols(const void* planes_all, int B, int D, float tau, int mode, const float* row_lse_s_all,
                     const float* col_lse_s_all, const float* row_lse_z_all, const float* col_sum_p_all,
                     const float* grad_loss, const void* W, int w_rows, int w_row_offset, int j0, int j1,
                     const float* dIz, float* dI_out, const int* gate, void* ws, size_t ws_bytes, void* stream);

/* Single-GPU convenience: prepare + three phases, forward and backward in one call
 * (loss_out: device scalar; dI/dT may both be NULL for forward only). */
size_t mc_clip_loss_fused_workspace_bytes(int B, int D, int mode);
int mc_clip_loss_fwd_bwd(const float* I, const float* T, int B, int D, float tau, int mode,
                         float* loss_out, float* dI, float* dT, void* ws, size_t ws_bytes,
                         void* stream);
/* Same through HOST buffers (pinned or pageable): copies in, computes, copies loss/grads out
 * and synchronises the stream.  `dws`/`dws_bytes` is DEVICE scratch of at least
 * mc_clip_loss_host_workspace_bytes().  From B = 16384 (tcgen05 engines) the gradient sweep runs
 * as two row strips and a per-device copy stream returns a finished strip while the next one is
 * swept (environment MAE_CLIP_HOST_STRIPS=1..8 overrides the strip count; 1 = single sweep);
 * when the call returns nothing of it is in flight on either stream. */
size_t mc_clip_loss_host_workspace_bytes(int B, int D, int mode);
int mc_clip_loss_fwd_bwd_host(const float* I_host, const float* T_host, int B, int D, float tau,
                              int mode, float* loss_host, float* dI_host, float* dT_host,
                              void* dws, size_t dws_bytes, void* stream);

/* ---------------------------------------------------------------------------
 * Peer memory (SURVEY.md section 8 e; the reference is single-process).  Each rank allocates one
 * exchange region, ships its 64-byte CUDA IPC handle to the other local ranks (any transport;
 * mae_clip_b200/dist.py uses torch.distributed) and maps theirs.  The kernels then load / store
 * peer memory directly over NVLink / NVSwitch:
 *   mc_peer_barrier  all ranks: epoch = ++epoch_counter[0] (epoch_counter: TWO private device
 *                    words {epoch, error}, zero at creation; every rank issues the same
 *                    sequence of barriers, so no launch argument depends on the step and the
 *                    step can be graph-captured); flag[rank] := epoch in every peer's flag
 *                    array (MC_PEER_MAX_WORLD zero-initialised words at flag_ptrs_host[q]),
 *                    then wait until every peer wrote the same epoch here.  A peer that does
 *                    not arrive within timeout_s (<= 0: 600 s, the order of a process-group
 *                    timeout) makes the kernel record 1 + that peer's rank in epoch_counter[1]
 *                    and return: the context stays usable (no trap), the data of the step is
 *                    invalid, and the host decides (mae_clip_b200/peer.py: PeerExchange.check()).
 *   mc_peer_publish  dst[q][dst_offset + kk*dst_stride + i] = src[kk*src_stride + i] (32-bit
 *                    words, kk < k, i < n) for every peer q < world.
 * mc_peer_alloc zero-fills the region and synchronises the device (set-up time, not the hot path).
 * ------------------------------------------------------------------------- */
#define MC_PEER_HANDLE_BYTES 64
#define MC_PEER_MAX_WORLD 16
int mc_peer_alloc(size_t bytes, void** dev_ptr_out, void* ipc_handle_out /* MC_PEER_HANDLE_BYTES */);
int mc_peer_open(const void* ipc_handle, void** dev_ptr_out);
int mc_peer_close(void* dev_ptr);
int mc_peer_free(void* dev_ptr);
int mc_peer_barrier(void* const* flag_ptrs_host, int rank, int world, unsigned int* epoch_counter,
                    double timeout_s, void* stream);
int mc_peer_publish(const void* src, int k, int n, int64_t src_stride, void* const* dst_ptrs_host,
                    int64_t dst_stride, int64_t dst_offset, int world, void* stream);
/* out[i] = sum over ranks q of src_ptrs_host[q][i], i < n_floats (a multiple of 4; 16-byte aligned pointers, usually
 * peer-mapped): the reduce-scatter step of the stored-weights gradient, each rank pulling its own rows. */
int mc_peer_reduce(void* const* src_ptrs_host, int world, size_t n_floats, float* out, const int* gate /* NULL or a device
                   word: the kernel returns unless it is 1 */, void* stream);

/* ---------------------------------------------------------------------------
 * L1-L2  ProjectionHead                                    modules.py:55-76
 *   projected = x Wp^T + bp; hidden = gelu(projected); y = hidden Wf^T + bf;
 *   z = keep*y/(1-p) + projected; out = LayerNorm(z) * gamma + beta
 * keep_mask: (B, P) bytes of 0/1 or NULL (eval mode).  projected / hidden / z /
 * mean / rstd are written for backward (all (B,P) or (B)); pass NULL for
 * hidden/z/mean/rstd under no_grad to skip the stores.  fwd_amax: optional EIGHT
 * device words the forward fills ([0], [1]: bit patterns of max|x|, max|hidden|; [2], [3]:
 * internal; [4], [5]: max|Wp|, max|Wf|) and the backward reads, so it need not reduce them again (NULL on either side:
 * recomputed).  prev_amax: optional, the fwd_amax words of an EARLIER forward of the same
 * head.  The fp16 operand planes take a power-of-two scale from max|x|; with prev_amax the
 * scale comes from the earlier call, the true maximum is reduced while x streams through
 * the GEMM, and a second, gated launch redoes the GEMM only if the old scale was outside
 * the safe fp16 window - the 268 MB activation is then read once, not twice.  Results do
 * not depend on prev_amax (a power-of-two scale changes nothing inside that window).
 * ------------------------------------------------------------------------- */
size_t mc_proj_head_workspace_bytes(int B, int E, int P, int mode);
int mc_proj_head_fwd(const float* x, int B, int E, int P, const float* w_proj, const float* b_proj,
                     const float* w_fc, const float* b_fc, const float* gamma, const float* beta,
                     const uint8_t* keep_mask, float p_drop, float eps, int mode, float* projected,
                     float* hidden, float* z, float* mean, float* rstd, float* out, float* fwd_amax,
                     const float* prev_amax, void* ws, size_t ws_bytes, void* stream);
/* dx may be NULL (frozen tower below the head: modules.py:35 / CLIP.py:18). */
int mc_proj_head_bwd(const float* grad_out, const float* x, int B, int E, int P,
                     const float* w_proj, const float* w_fc, const float* gamma,
                     const uint8_t* keep_mask, float p_drop, int mode, const float* projected,
                     const float* hidden, const float* z, const float* mean, const float* rstd,
                     float* dx, float* dw_proj, float* db_proj, float* dw_fc, float* db_fc,
                     float* dgamma, float* dbeta, const float* fwd_amax, void* ws, size_t ws_bytes,
                     void* stream);

/* fp32-class tensor-core GEMM the heads are built from (exposed for tests and reuse):
 * C[M,N] = A[M,K] . B[N,K]^T (+ bias[n]); A, B, C dense row-major fp32; gelu_out (optional) =
 * gelu(C), exact erf form.  Operands are staged as fp16 hi/lo planes inside `ws`. */
size_t mc_tc_gemm_workspace_bytes(int M, int N, int K);
int mc_tc_gemm(const float* A, const float* B, int M, int N, int K, const float* bias, float* C,
               float* gelu_out, void* ws, size_t ws_bytes, void* stream);

/* The pair kernels the heads run on from round 2 (csrc/head_tc.cu), exposed for tests: the activation
 * operand is read as fp32 and split into fp16 hi / lo inside the kernel (converter warps -> tensor
 * memory), the weights are staged as planes inside `ws`.  passes: 3 (fp32-class) or 1.
 *   kind 0  C(M, 256) = A(M, K) . B(256, K)^T (+ bias; gelu_out = gelu(C) when given)
 *   kind 1  C(M, N)   = A(M, K) . B(N, K)^T, K <= 256 (A stays resident in tensor memory)
 *   kind 2  C(256, N) = A(K, 256)^T . B(K, N) (both operands transposed in the kernel; split-K) */
size_t mc_head_gemm_workspace_bytes(int kind, int M, int N, int K);
int mc_head_gemm(int kind, const float* A, const float* B, int M, int N, int K, const float* bias,
                 float* C, float* gelu_out, int passes, void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------
 * M1  MAE per-sample random masking        (NOT in the reference: north_star; oracle/mae_ref.py)
 * noise (N,L) fp32; stable ascending argsort (ties -> lower index).  Outputs:
 * ids_restore (N,L) int64, mask (N,L) fp32 (0 keep / 1 removed), ids_keep
 * (N,len_keep) int64, x_masked (N,len_keep,Dm) gathered rows of x (N,L,Dm).
 * elem_size 2 (bf16/fp16) or 4 (fp32).  x / x_masked may be NULL (indices only).
 * ------------------------------------------------------------------------- */
int mc_random_masking(const void* x, int elem_size, const float* noise, int N, int L, int Dm,
                      int len_keep, void* x_masked, float* mask, int64_t* ids_restore,
                      int64_t* ids_keep, void* stream);
/* backward of the gather: grad_x (N,L,Dm) = scatter(grad_x_masked) with zeros elsewhere */
int mc_random_masking_bwd(const void* grad_x_masked, int elem_size, const float* mask,
                          const int64_t* ids_restore, int N, int L, int Dm, int len_keep,
                          void* grad_x, void* stream);

/* ---------------------------------------------------------------------------
 * M2-M3  patchify + normalised-pixel target + masked MSE   (NOT in the reference)
 * pred (N,L,p*p*3) in pred_elem_size (2 = bf16, 4 = fp32); imgs (N,3,H,W) fp32;
 * mask (N,L) fp32.  loss = sum(mask * mean_e (pred-target)^2) / sum(mask).
 * The target is never materialised.  `ws` needs mc_masked_mse_workspace_bytes().
 * ------------------------------------------------------------------------- */
size_t mc_masked_mse_workspace_bytes(int N, int L);
int mc_masked_mse_fwd(const void* pred, int pred_elem_size, const float* imgs, const float* mask,
                      int N, int H, int W, int p, int norm_pix, float* loss_out,
                      float* mask_sum_out, void* ws, size_t ws_bytes, void* stream);
int mc_masked_mse_bwd(const void* pred, int pred_elem_size, const float* imgs, const float* mask,
                      int N, int H, int W, int p, int norm_pix, const float* mask_sum,
                      const float* grad_loss /* device scalar or NULL = 1 */, void* dpred,
                      void* stream);

/* "next" rows (SURVEY.md section 8 f, rank 2): standalone patchify and decoder-side un-shuffle */
int mc_patchify(const float* imgs, int N, int H, int W, int p, int norm_pix, float* out,
                void* stream);
int mc_restore_tokens(const void* x_kept, int elem_size, const void* mask_token,
                      const int64_t* ids_restore, int N, int L, int Dm, int len_keep, void* out,
                      void* stream);

/* backward of mc_restore_tokens: grad_out (N,L,Dm) -> d x_kept (N,len_keep,Dm) (rows whose
 * ids_restore < len_keep) and d mask_token (Dm) = column sum of the other rows (fp32 accumulate,
 * written in the element type; is_bf16 selects bf16 vs fp16 when elem_size == 2).  Rows must be
 * 16-byte multiples of at most 16 KB. */
size_t mc_restore_tokens_bwd_workspace_bytes(int N, int L, int Dm);
int mc_restore_tokens_bwd(const void* grad_out, int elem_size, int is_bf16,
                          const int64_t* ids_restore, int N, int L, int Dm, int len_keep,
                          void* dx_kept, void* dmask_token, void* ws, size_t ws_bytes, void* stream);

/* "next" row 3: inference-side retrieval                       inference.py:42-46 (find_matches)
 *   scores[q][n] = <text[q] / max(|text[q]|, 1e-12), image[n] / max(|image[n]|, 1e-12)>   (F.normalize + matmul)
 *   out_vals / out_idx (Q, k): the k largest scores of every query, descending, ties -> lower index
 *   (torch.topk leaves tie order unspecified).  The image bank (N, D) fp32 is streamed once.
 *   scores_out: optional (Q, N) fp32 buffer that receives the full similarity matrix (NULL: it
 *   lives in `ws`).  k = 0 computes the scores only.  k <= 1024, k <= N. */
size_t mc_similarity_topk_workspace_bytes(int Q, long long N, int D);
int mc_similarity_topk(const float* text, int Q, const float* image, long long N, int D, int k,
                       float* out_vals, int64_t* out_idx, float* scores_out, void* ws,
                       size_t ws_bytes, void* stream);

/* Retrieval evaluation   (NOT in the reference: the standard evaluation of a CLIP model, recall@K in
 * both directions; oracle/retrieval_ref.py)
 *   s[q][n] = <text[q] / max(|text[q]|, 1e-12), image[n] / max(|image[n]|, 1e-12)>, text (Q, D) and
 *   image (N, D) fp32.  g(q) = text_to_image[q], the image of caption q (NULL: Q == N, g(q) = q).
 *   t2i_rank[q] = #{ n != g(q) : s[q][n] > s[q][g(q)] }                    (0: own image first)
 *   i2t_rank[n] = #{ q : g(q) != n, s[q][n] > u_n },  u_n = max over q with g(q) == n of s[q][n]
 *                 (rank of the best-ranked caption); -1 for an image without a caption.
 * Strict comparisons: exact ties count for the positive.  The counts are exact integers and identical
 * run to run, but they compare the engine's scores (mode MC_GEMM_TC_F16X3 or MC_GEMM_TC_F16;
 * MC_GEMM_SIMT_FP32 -> MC_ERR_UNSUPPORTED): a candidate within ~3e-5 (tc_f16x3) or ~2e-3 (tc_f16)
 * of the threshold may land on either side.  D <= 256 and D % 4 == 0, else MC_ERR_UNSUPPORTED.
 * text_to_image entries must lie in [0, N) (not checked here).  The score matrix is never stored;
 * the call allocates nothing and does not synchronise. */
size_t mc_retrieval_ranks_workspace_bytes(int Q, int N, int D, int mode);
int mc_retrieval_ranks(const float* text, int Q, const float* image, int N, int D,
                       const int64_t* text_to_image, int mode, int32_t* t2i_rank,
                       int32_t* i2t_rank, void* ws, size_t ws_bytes, void* stream);

/* Retrieval top-k for query batches   (NOT in the reference)
 *   out_vals / out_idx (Q, k): the exact top-k of s[q][n] (as mc_retrieval_ranks defines it, the same
 *   score bits) for every query q: descending, exact ties -> lower index, bit-identical run to run.
 *   out_vals holds the engine's fp32 scores (mode MC_GEMM_TC_F16X3 or MC_GEMM_TC_F16; within ~3e-5 /
 *   ~2e-3 of the true cosine), out_idx the image indices.  Image-to-text top-k: swap the arguments.
 * Limits: 1 <= k <= N (else MC_ERR_BAD_ARG); k <= 1024, D <= 256 and D % 4 == 0, tensor-core modes
 * only (else MC_ERR_UNSUPPORTED).  The call allocates nothing and does not synchronise.
 * The (Q, N) matrix is never stored: the bank is swept in chunks of C entries and a query keeps at
 * most C survivors per chunk.  C = min(max(floor(2^28 / (8 Q)) rounded down to u, u), 65536,
 * N rounded up to u), u = 128 when Q >= N and 256 otherwise.  The workspace is
 *   4 Q D + 4 N D + 4 min(Q, N) D' + 8 Q k + 8 Q + 8 Q C  bytes (+ 256-byte padding per piece),
 * D' = D rounded up to 8 (the fp16 hi + lo planes of the smaller side): O((Q + N) D + Q (k + C)). */
size_t mc_retrieval_topk_workspace_bytes(int Q, int N, int D, int k, int mode);
int mc_retrieval_topk(const float* text, int Q, const float* image, int N, int D, int k, int mode,
                      float* out_vals, int64_t* out_idx, void* ws, size_t ws_bytes, void* stream);

/* Token side of the data feed (dataset.py:19-31): the reference tokenises all captions once, padded to one length L, and
 * builds torch.tensor(values[idx]) per sample for input_ids / attention_mask (stacked by the default collate).  Here the
 * (N, L) int64 tables stay resident in HBM and a batch is a gather of rows by the sampler's n indices (negative indices
 * wrap like python's).  An index outside [-N, N) sets *bad_index_flag (device int, cleared by the caller) and yields a
 * row of zeros - the reference raises IndexError; mae_clip_b200/data.py turns the flag into one. */
int mc_gather_token_rows(const int64_t* ids_all, const int64_t* mask_all, int64_t N, int L,
                         const int64_t* idx, int n, int64_t* ids_out, int64_t* mask_out,
                         int* bad_index_flag, void* stream);

/* "next" row 4: image side of the data feed        dataset.py:33-34,49 (A.Normalize + permute + float)
 * hwc: (N, H, W, 3) uint8 DEVICE pixels (after the reference's cv2 resize, which stays on the host);
 * out_nchw: (N, 3, H, W) fp32 = (pixel - mean*max_pixel_value) * (1 / (std*max_pixel_value)).
 * mean3_host / std3_host: HOST arrays of three floats (albumentations defaults: ImageNet statistics). */
int mc_normalize_images(const uint8_t* hwc, int N, int H, int W, const float* mean3_host,
                        const float* std3_host, float max_pixel_value, float* out_nchw, void* stream);

/* "next" row 1: the optimiser step of the training driver      main.py:103-105, main.py:59
 * (torch.optim.AdamW, decoupled weight decay, no amsgrad).  params / grads / exp_avg /
 * exp_avg_sq: HOST arrays of `ntensors` device pointers (dense fp32), numel: HOST array of
 * element counts.  `step` counts from 1 (bias correction).  grad_scale: optional device scalar
 * multiplied into every gradient (NULL = 1).  One launch per 48 tensors. */
int mc_adamw_step(int ntensors, float* const* params, const float* const* grads,
                  float* const* exp_avg, float* const* exp_avg_sq, const int64_t* numel, double lr,
                  double beta1, double beta2, double eps, double weight_decay, int step,
                  const float* grad_scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MAE_CLIP_B200_H_ */

/* thinkdiff_b200.h -- C ABI of the B200-native ThinkDiff aligner hot path (libthinkdiff_b200.so).
 *
 * The reference (avi22bhattacharya/ThinkDiff-mlre) is 100 % Python and has no FFI of its own: the hot path is the
 * `mm_projector` nn.Module built by `build_vision_projector` and the ops either side of it. Each entry point below
 * names the reference code it replaces (paths relative to the reference root). The host side that binds these
 * symbols is thinkdiff_mlre_b200/_lib.py (ctypes); INTEGRATION.md shows the binding a maintainer adds.
 *
 * Conventions: plain pointers and sizes only; every pointer is a DEVICE pointer unless marked [host]; the caller owns
 * all buffers (outputs, saved activations, workspaces); every call is asynchronous on `stream` (a cudaStream_t);
 * return value 0 = ok, negative = error, text via td_last_error() (thread-local). No exceptions cross the ABI.
 * bf16 tensors are row-major, 16-byte aligned, with feature dimensions that are multiples of 64.
 * There is no CPU fallback: a device that is not sm_100 makes every call fail with TD_ERR_UNSUPPORTED.
 */
#ifndef THINKDIFF_B200_H
#define THINKDIFF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* td_stream_t; /* cudaStream_t */

enum { TD_DTYPE_F32 = 0, TD_DTYPE_BF16 = 1 };
enum { TD_OK_ = 0, TD_ERR_ARG_ = -1, TD_ERR_UNSUPPORTED_ = -2, TD_ERR_DRIVER_ = -3 };
/* td_aligner_bwd phases (bit mask): the split lets the caller start the all-reduce of the Linear2 gradients
 * while the Linear1 gradients are still being computed (DDP bucket overlap, thinkdiff/runners/runner_base.py:88-92). */
enum { TD_BWD_PHASE_NORM_W2 = 1, TD_BWD_PHASE_GELU_W1 = 2, TD_BWD_PHASE_ALL = 3,
       /* td_aligner_bwd_dh2 only: the two halves of NORM_W2, so the small vectors' all-reduce can start before the dW2 GEMM */
       TD_BWD_PHASE_SMALL2_ONLY = 4, TD_BWD_PHASE_W2_ONLY = 8,
       /* the two halves of GELU_W1: the dh0 GEMM + db1 (dh0 stays in the workspace), and the dW1 GEMM from that dh0 */
       TD_BWD_PHASE_GELU_ONLY = 16, TD_BWD_PHASE_W1_ONLY = 32 };
/* td_aligner_mse_fwd stages (bit mask) */
enum { TD_FWD_STAGE_LINEAR1 = 1, TD_FWD_STAGE_REST = 2, TD_FWD_STAGE_ALL = 3,
       /* leave the loss un-finished: td_aligner_bwd_dh2(loss_out = ...) sums the per-CTA partials in its own finisher launch */
       TD_FWD_STAGE_DEFER_LOSS = 4 };

const char* td_last_error(void);
int32_t td_version(void);
/* 0 when the current CUDA device can run this library (compute capability 10.x), else TD_ERR_UNSUPPORTED. */
int32_t td_device_check(void);

/* Per-launch device timing for benchmarks: while enabled, every kernel launch of the library is bracketed by CUDA
 * events on its stream. td_profile_report fills `buf` [host] with "tag,launches,total_ms,total_work\n" lines, where
 * work = algorithmic FLOPs for gemm_* tags and for the attention kernels attn_fwd / attn_bwd_dkdv / attn_bwd_dq (visible
 * (query, key) pairs only, see td_t5_attention_fwd), and algorithmic bytes for the row kernels. Enabling clears old records. */
int32_t td_profile_enable(int32_t on);
int32_t td_profile_report(char* buf /*[host]*/, int32_t buflen);
/* One "tag,stream,start_ms,end_ms\n" line per recorded launch, relative to the first record: a per-stream device timeline. */
int32_t td_profile_timeline(char* buf /*[host]*/, int32_t buflen);

/* ---- (1) ragged pack / pad / mask ------------------------------------------------------------------------
 * Replaces the collater's pad/stack/mask loop, thinkdiff/datasets/datasets/llava_instruct_dataset_mllama_embed_2.py
 * :101-131 (random split), :132-162 (fixed max), :78-99 (input embeds), and the padded H2D copy of
 * thinkdiff/datasets/data_utils.py:83-96. Source = all samples' full embeddings back to back, `row_bytes` per row;
 * sample i keeps rows [src_row_start[i], src_row_start[i] + len_i). Outputs are bit-exact copies. */
int32_t td_cu_seqlens(const int32_t* lens, int32_t B, int32_t* cu_seqlens /*[B+1]*/, td_stream_t stream);
int32_t td_pack_varlen(const void* src, const int64_t* src_row_start /*[B]*/, const int32_t* cu_seqlens /*[B+1]*/,
                       int32_t B, int64_t total_rows /* = cu_seqlens[B], known to the host */, int64_t row_bytes,
                       void* dst_packed /*[total_rows, row_bytes]*/, td_stream_t stream);
/* Same, and also writes src_row_out[r] (int64, may be NULL) = the source row that packed row r came from, so that a sibling
 * tensor in the same ragged source layout (e.g. the T5 targets) can be read in place instead of being packed too. */
int32_t td_pack_varlen_indexed(const void* src, const int64_t* src_row_start, const int32_t* cu_seqlens, int32_t B,
                               int64_t total_rows, int64_t row_bytes, void* dst_packed, int64_t* src_row_out,
                               td_stream_t stream);
/* Gather from TWO sources with one launch: segment i with src_row_start[i] >= 0 reads rows of `src`, with src_row_start[i] =
 * -(s + 1) rows s.. of `src2`. The ragged `[img1 | img2 | text]` composition of the reference's two-image demo
 * (scripts/test/test_blip_vision_t5_decoder_flux_text.py:184-208: torch.cat([...], dim=1) per sample) without first concatenating
 * the aligner output and the text embeddings into one buffer. */
int32_t td_pack_varlen2(const void* src, const void* src2, const int64_t* src_row_start, const int32_t* cu_seqlens, int32_t B,
                        int64_t total_rows, int64_t row_bytes, void* dst_packed, td_stream_t stream);
/* Reference layout: zero-padded [B, L_max, row_bytes] + int64 mask [B, L_max] (mask may be NULL). With
 * src = a packed buffer and src_row_start[i] = cu_seqlens[i] this is the inverse of td_pack_varlen. */
int32_t td_pack_padded(const void* src, const int64_t* src_row_start, const int32_t* cu_seqlens, int32_t B, int32_t L_max,
                       int64_t row_bytes, void* dst_padded, int64_t* mask, td_stream_t stream);

/* ---- parameters: fp32 master -> bf16 compute copy (what autocast does per call, base_task.py:237) ---------- */
int32_t td_cast_f32_to_bf16(const float* src, void* dst_bf16, int64_t n, td_stream_t stream);

/* ---- (2) aligner = Linear -> GELU(erf) -> Linear -> T5LayerNorm ---------------------------------------------
 * Replaces `self.mm_projector(x)` (thinkdiff/models/mllama_vllm_t5_embed_decoder_2.py:585, :761, :998, :1115;
 * thinkdiff/models/blip_vision_t5_decoder.py:414, :641) for the module built at ...embed_decoder_2.py:58-63.
 *   x [M, Din] bf16 (rows = tokens; pass the packed buffer), W1 [D, Din], b1 [D], W2 [D, D], b2 [D] bf16, g [D] fp32.
 *   Saved for backward (may be NULL for inference, except h2): h0 = Linear1 out, h1 = GELU out, h2 = Linear2 out
 *   (all bf16 [M, D]), rstd fp32 [M].  y [M, D]: fp32 (training rule) or bf16 (pure-bf16 inference rule). */
int64_t td_aligner_fwd_workspace_bytes(int64_t M, int32_t Din, int32_t D);
int32_t td_aligner_fwd(const void* x, int64_t M, int32_t Din, int32_t D, const void* W1, const void* b1, const void* W2,
                       const void* b2, const float* g, float eps, void* h0, void* h1, void* h2, float* rstd, void* y,
                       int32_t y_dtype, void* workspace, int64_t workspace_bytes, td_stream_t stream);
/* Backward of the above for an upstream gradient dy [M, D] (fp32 or bf16). Replaces autograd through the Sequential
 * (triggered at thinkdiff/tasks/base_task.py:241-244). Writes (not accumulates) fp32 gradients scaled by grad_scale:
 * dW1 [D, Din], db1 [D], dW2 [D, D], db2 [D], dg [D]. No dx (the features do not require grad). */
int64_t td_aligner_bwd_workspace_bytes(int64_t M, int32_t Din, int32_t D);
int32_t td_aligner_bwd(const void* dy, int32_t dy_dtype, const void* x, const void* h0, const void* h1, const void* h2,
                       const float* rstd, const void* W2, const float* g, int64_t M, int32_t Din, int32_t D,
                       float grad_scale, float* dW1, float* db1, float* dW2, float* db2, float* dg, void* workspace,
                       int64_t workspace_bytes, int32_t phases, td_stream_t stream);

/* Fused training path against T5 targets (masked MSE over all M packed rows): forward GEMMs, then ONE pass that forms
 * y = T5LayerNorm(h2) in registers, accumulates sum (y - target)^2 and writes the norm backward of dy = 2 (y - target) / (M D)
 * -- y and dy never touch HBM. Outputs for a UNIT upstream gradient: dh2 bf16 [M, D], the per-CTA partial column sums for
 * dg / db2 (`norm_partials`, td_aligner_norm_partials_bytes bytes, caller-owned until the backward) and the loss (fp32 device
 * scalar). `target` rows are read at target_row_index[r] (int64 [M]) when given, else at r -- targets in the un-packed
 * source layout need no pack pass. td_aligner_bwd_dh2 finishes the backward, multiplying by grad_scale * (*grad_scale_ptr)
 * (grad_scale_ptr: optional DEVICE scalar = the upstream gradient of the loss, e.g. GradScaler's scale; no host sync).
 * Same gradients as td_aligner_fwd -> td_masked_mse_fwd_bwd -> td_aligner_bwd (base_task.py:237-244 with an MSE loss).
 * `stages` lets the caller run Linear1 and the rest as two calls (same buffers), e.g. to apply the Linear2 parameter update
 * of the previous step in between while that bucket's all-reduce was still in flight.
 * td_aligner_bwd_dh2 extras: loss_out (optional) finishes a loss deferred with TD_FWD_STAGE_DEFER_LOSS; stats (optional, fp32
 * [2], zeroed by the caller once per optimizer step) counts non-finite gradient values in stats[0] -- GradScaler's inf check,
 * thinkdiff/tasks/base_task.py:241-258; accumulate != 0 adds into the gradient buffers instead of overwriting them
 * (accum_grad_iters > 1, base_task.py:247). Launch order inside one call: dh0 GEMM, ONE finisher launch (db1 | dg, db2 | loss),
 * dW1 GEMM, dW2 GEMM. */
int64_t td_aligner_mse_fwd_workspace_bytes(int64_t M, int32_t Din, int32_t D);
int64_t td_aligner_norm_partials_bytes(int64_t M, int32_t D);
int32_t td_aligner_mse_fwd(const void* x, int64_t M, int32_t Din, int32_t D, const void* W1, const void* b1, const void* W2,
                           const void* b2, const float* g, float eps, const void* target, int32_t target_dtype,
                           const int64_t* target_row_index, void* h0, void* h1, void* dh2, void* norm_partials, float* loss,
                           void* workspace, int64_t workspace_bytes,
                           int32_t stages /* TD_FWD_STAGE_* */, td_stream_t stream);
int32_t td_aligner_bwd_dh2(const void* dh2, const void* x, const void* h0, const void* h1, const void* W2,
                           const void* norm_partials, int64_t M, int32_t Din, int32_t D, float grad_scale,
                           const float* grad_scale_ptr, float* dW1, float* db1, float* dW2, float* db2, float* dg,
                           float* loss_out, float* stats, int32_t accumulate, void* workspace, int64_t workspace_bytes,
                           int32_t phases, td_stream_t stream);

/* Standalone T5LayerNorm forward / backward (transformers modeling_t5.py T5LayerNorm, imported at
 * ...embed_decoder_2.py:24). x bf16 [M, D]; y fp32 or bf16; dW/db are fp32 [D]; db = column sums of dx (may be NULL). */
int32_t td_rmsnorm_fwd(const void* x, const float* g, float eps, int64_t M, int32_t D, void* y, int32_t y_dtype,
                       float* rstd, td_stream_t stream);
int64_t td_rmsnorm_bwd_workspace_bytes(int64_t M, int32_t D);
int32_t td_rmsnorm_bwd(const void* dy, int32_t dy_dtype, const void* x, const float* rstd, const float* g, int64_t M,
                       int32_t D, void* dx_bf16, float* dg, float* dxsum, void* workspace, int64_t workspace_bytes,
                       td_stream_t stream);

/* Workspace of one GEMM launch for its stream-K tail (the output tiles left over after the last full wave of CTA pairs are
 * cut along K; partial accumulators meet here). The td_aligner_* workspaces include it; the two entries below take it as an
 * optional argument (NULL: the leftover tiles run as a last, partially filled wave). */
int64_t td_gemm_workspace_bytes(void);
/* Plain bf16 linear  out[M, N] = x[M, K] . W[N, K]^T (+ bias)  -- nn.Linear under autocast (F.linear). */
int32_t td_linear_bf16(const void* x, int64_t M, int32_t K, const void* W, int32_t N, const void* bias, void* out,
                       void* workspace, int64_t workspace_bytes, td_stream_t stream);
/* Input gradient of td_linear_bf16 for a FROZEN weight:  dx[M, K] (bf16) = dy[M, N] (bf16) . W[N, K]  -- W is contracted over
 * its row index and read where it lies (MN-major operand), no transposed copy. Needs N % 8 == 0, K % 64 == 0. */
int32_t td_linear_bf16_dx(const void* dy, int64_t M, int32_t N, const void* W, int32_t K, void* dx, void* workspace,
                          int64_t workspace_bytes, td_stream_t stream);
/* Generic entry to the tcgen05 GEMM for tests: D[M,N] (fp32) (+)= alpha * A.B^T with either operand K-major
 * ([rows, K]) or MN-major ([K, rows]); cta_pair selects cta_group::2; accumulate != 0 adds into D. */
int32_t td_gemm_bf16_f32out(const void* A, int64_t lda, int32_t a_mn_major, const void* B, int64_t ldb,
                            int32_t b_mn_major, int64_t M, int32_t N, int64_t K, float alpha, float* out,
                            int32_t cta_pair, int32_t accumulate, void* workspace, int64_t workspace_bytes,
                            td_stream_t stream);

/* ---- optimizer (SURVEY section 8 f-3): torch.optim.AdamW semantics (thinkdiff/runners/runner_base.py:122-127), one pass
 * that reads the (all-reduced) gradient, updates p / exp_avg / exp_avg_sq in place and writes the bf16 compute copy of p.
 * Arrays below are HOST arrays of `num_tensors` (1..3) entries holding device pointers / sizes; params_bf16 (or its
 * entries) may be NULL. `step` counts from 1; gradients are multiplied by grad_scale (1 / loss scale) first.
 * step_ctl (optional, DEVICE, td_step_ctl_bytes): the device-resident control block of the step -- when given, the bias
 * corrections, the unscale / clip factor and the skip decision are read from it (no host sync), `step` is ignored. */
int32_t td_adamw_step(int32_t num_tensors, float* const* params /*[host]*/, const float* const* grads /*[host]*/,
                      float* const* exp_avg /*[host]*/, float* const* exp_avg_sq /*[host]*/,
                      void* const* params_bf16 /*[host]*/, const int64_t* numel /*[host]*/,
                      const float* weight_decay /*[host]*/, float lr, float beta1, float beta2, float eps, int64_t step,
                      float grad_scale, const void* step_ctl, td_stream_t stream);
/* Device-side GradScaler + step bookkeeping (torch.amp.GradScaler as installed at thinkdiff/runners/runner_base.py:131-139 and
 * driven at thinkdiff/tasks/base_task.py:241-258, plus clip_grad_norm_): the control block holds {skip, gradient multiplier,
 * bias corrections, applied-step count, loss scale, growth tracker, gradient norm}. td_step_ctl_update folds the step's
 * statistics (stats[0] = non-finite count, stats[1] = sum of squares of the scaled gradients, both summed over ranks by the
 * caller) into it: non-finite -> skip + scale *= backoff; else step += 1, new bias corrections, clip coefficient
 * min(1, max_grad_norm / (norm + 1e-6)) when max_grad_norm > 0, and scale *= growth every growth_interval clean steps.
 * The loss scale for the next backward is the float at byte offset TD_STEP_CTL_SCALE_OFFSET (pass it as grad_scale_ptr). */
enum { TD_STEP_CTL_SCALE_OFFSET = 20 };
int64_t td_step_ctl_bytes(void);
int32_t td_step_ctl_init(void* step_ctl, float init_scale, int64_t applied_steps, td_stream_t stream);
int32_t td_step_ctl_update(void* step_ctl, const float* stats, int32_t use_scaler, float growth_factor, float backoff_factor,
                           int32_t growth_interval, float beta1, float beta2, float max_grad_norm, td_stream_t stream);
/* stats[0] += number of non-finite values, stats[1] += sum of squares of grad[0..numel) (what unscale_ + clip_grad_norm_ read). */
int32_t td_grad_stats(const float* grad, int64_t numel, float* stats, td_stream_t stream);

/* ---- (e) data parallel over NVLink peer memory ----------------------------------------------------------------------------
 * Replaces DDP's NCCL all-reduce of the aligner gradients + the replicated optimizer step
 * (thinkdiff/runners/runner_base.py:88-92, :98-127; thinkdiff/tasks/base_task.py:247-258) with a reduce-scatter fused into
 * the weight-gradient GEMM epilogues: rank o owns rows [o D/world, (o+1) D/world) of W1 and W2; every rank's GEMM stores
 * those rows of its (1/world-scaled) gradient straight into "slot[this rank]" of rank o's exchange buffer; rank o sums the
 * slots in rank order inside its AdamW pass and stores the updated bf16 rows into every rank's compute copy. Ordering is by
 * monotonically increasing counters in the destination's memory (td_peer_signal / td_peer_wait), no collectives.
 * Buffers come from td_peer_alloc (cudaMalloc + CUDA IPC handle, zero-filled); the other processes map them with td_peer_open.
 * All pointer arrays are HOST arrays of `n` / `world` device pointers (<= TD_MAX_PEERS), entry o = the address in rank o. */
enum { TD_MAX_PEERS = 8, TD_IPC_HANDLE_BYTES = 64 };
int32_t td_peer_alloc(int64_t bytes, void** ptr /*[host] out*/, uint8_t* handle /*[host] out, TD_IPC_HANDLE_BYTES*/);
int32_t td_peer_free(void* ptr);
int32_t td_peer_open(const uint8_t* handle /*[host]*/, void** ptr /*[host] out*/);
int32_t td_peer_close(void* ptr);
/* flag_arrays[i][slot] += 1 at every rank i (remote atomic add, release at system scope), ordered after all earlier work on
 * `stream`: a counter reaches t * world when every rank has signalled step t. */
int32_t td_peer_signal(void* const* flag_arrays /*[host]*/, int32_t n, int32_t slot, td_stream_t stream);
/* Blocks `stream` until flags[0..n) >= value (local int32 flags written by the peers). Implemented with stream memory operations
 * (cuStreamWaitValue32: no kernel occupies an SM while waiting; a peer that never signals blocks the stream, as a lost NCCL rank
 * would); with TD_PEER_WAIT=kernel a polling kernel is used instead, which traps after timeout_s (<= 0: 600 s). */
int32_t td_peer_wait(const int32_t* flags, int32_t n, int32_t value, float timeout_s, td_stream_t stream);
/* dst[i][0..numel) = src[0..numel) for every rank i (the three small gradient vectors: every rank gets every rank's copy). */
int32_t td_peer_post(const float* src, void* const* dst /*[host]*/, int32_t n, int64_t numel, td_stream_t stream);
/* out = slots[0] + slots[1] + ... + slots[n_slots - 1] (slot s at slots + s * slot_stride), always in that order. */
int32_t td_sum_slots(const float* slots, int64_t slot_stride, int32_t n_slots, float* out, int64_t numel, td_stream_t stream);
/* td_adamw_step for one row block whose gradient is the sum of n_slots slots; the bf16 rows go to params_bf16[0..n_dst). */
int32_t td_adamw_slots_step(float* param, const float* grad_slots, int64_t slot_stride, int32_t n_slots, float* exp_avg,
                            float* exp_avg_sq, void* const* params_bf16 /*[host]*/, int32_t n_dst, int64_t numel,
                            float weight_decay, float lr, float beta1, float beta2, float eps, int64_t step,
                            float grad_scale, const void* step_ctl, td_stream_t stream);
/* td_aligner_bwd_dh2 with the two weight gradients row-scattered: dW?_dst[o] = [D / world, cols] fp32 block for the rows
 * rank o owns. Every output element is stored exactly once (bit-reproducible) with coalesced 128-byte stores. */
/* Optional extras of td_aligner_bwd_dh2_scatter: the exchange protocol's tiny launches folded into the kernels of the call.
 *   signal_flags / signal_slot : the LAST weight-gradient GEMM of the call, once ALL of its stores have completed, adds 1 to int32
 *                                element `signal_slot` of every rank's flag array (what td_peer_signal after the call would do);
 *   small_dst / small_base / small_numel : the finisher launch stores every output that lies in [small_base, small_base +
 *                                small_numel) -- this rank's [db2 | dg | db1] bucket -- at the same offset into small_dst[o], this
 *                                rank's slot at every rank (what td_peer_post after the call would do). */
typedef struct td_peer_fold {
  void* const* signal_flags; /* [host] world device pointers, or NULL */
  int32_t signal_slot;
  void* const* small_dst;    /* [host] world device pointers, or NULL */
  const float* small_base;
  int64_t small_numel;
} td_peer_fold;
int32_t td_aligner_bwd_dh2_scatter(const void* dh2, const void* x, const void* h0, const void* h1, const void* W2,
                                   const void* norm_partials, int64_t M, int32_t Din, int32_t D, float grad_scale,
                                   const float* grad_scale_ptr, float* const* dW1_dst /*[host]*/, float* db1,
                                   float* const* dW2_dst /*[host]*/, float* db2, float* dg, float* loss_out, float* stats,
                                   int32_t world, int32_t rank /* of the caller; < 0: no traffic shaping */,
                                   const td_peer_fold* fold /*[host] or NULL*/, void* workspace, int64_t workspace_bytes,
                                   int32_t phases, td_stream_t stream);
/* Host arithmetic only (needs no GPU): the work schedule of one M x N x K GEMM launch on `workers` CTA pairs -- the whole-tile
 * waves and, with stream_k != 0, the tail whose tiles are cut along K -- as the list of segments the kernel's workers claim, in
 * claim order: out[8 i ..] = {unit, tile, first k-block, end k-block, kind (0 whole tile or unshared, 1 owner of a shared tile,
 * 2 contributor), first contributor range, number of contributor ranges, tail range index}. Returns the number of segments (which
 * may exceed max_segments: only that many are written), -1 on bad arguments. For tests of the scheduler's coverage properties. */
int32_t td_gemm_schedule(int64_t M, int32_t N, int64_t K, int32_t workers, int32_t stream_k, int32_t* out /*[host]*/,
                         int32_t max_segments);
/* Host arithmetic only (needs no GPU): the rank that owns the rows of output tile number `tile` (256 x 256 tiles, in the order
 * the kernel claims them) of a row-scattered M x N weight-gradient GEMM run by `rank` of `world`; the tile's block coordinates
 * go to m_blk / n_blk when those are non-NULL. Documents (and lets a CPU test check) the traffic shaping: for any `tile`, the
 * owners over rank = 0..world-1 are all different. Returns -1 on arguments the scattered GEMM would reject. */
int32_t td_scatter_tile_owner(int32_t tile, int32_t M, int32_t N, int32_t world, int32_t rank, int32_t* m_blk /*[host]*/,
                              int32_t* n_blk /*[host]*/);
/* Test entry for the scatter epilogue: out[M, N] = alpha * A^T.B with A [K, M], B [K, N] (both MN-major, the weight-gradient
 * shape), rows [o M/world, (o+1) M/world) written to dst[o] ([M / world, N] fp32). `rank` >= 0 (and an owner's rows being whole
 * 256-row tiles) selects the owner-grouped tile order rotated by rank that the data-parallel step uses, so that the N ranks'
 * GEMMs store to N different owners at any moment; rank < 0 keeps the tile order -- and the bits -- of the local-output GEMM. */
int32_t td_gemm_tn_scatter(const void* A, int64_t lda, const void* B, int64_t ldb, int64_t M, int32_t N, int64_t K,
                           float alpha, float* const* dst /*[host]*/, int32_t world, int32_t rank, void* workspace,
                           int64_t workspace_bytes, td_stream_t stream);

/* ---- (3) masked losses, forward + gradient in one pass -----------------------------------------------------
 * Cross entropy replaces `CrossEntropyLoss(ignore_index=-100)(lm_logits.view(-1, V), labels.view(-1))`
 * (thinkdiff/models/mllama_vllm_t5_embed_decoder_2.py:241-246; blip_vision_t5_decoder.py:222-227).
 * Masked MSE is the north-star's added loss (absent from the reference): mean over valid rows x D of (y - t)^2.
 * loss: fp32 scalar on the device. Gradients are multiplied by grad_scale (GradScaler, base_task.py:241). */
int64_t td_loss_workspace_bytes(int64_t rows);
int32_t td_masked_mse_fwd_bwd(const void* y, int32_t y_dtype, const void* target, int32_t target_dtype,
                              const int64_t* row_mask /* NULL = all rows valid; else != 0 is valid */, int64_t M,
                              int32_t D, float grad_scale, float* loss, void* dy /* y_dtype, may be NULL */,
                              void* workspace, int64_t workspace_bytes, td_stream_t stream);
int32_t td_masked_ce_fwd_bwd(const void* logits, int32_t logits_dtype, const int64_t* labels /* -100 = ignore */,
                             int64_t R, int32_t V, float grad_scale, float* loss,
                             void* dlogits /* logits_dtype, may be NULL */, void* workspace, int64_t workspace_bytes,
                             td_stream_t stream);


/* ---- SURVEY section 8 f-1, first slice: the frozen T5 decoder's output head with its loss --------------------------
 * Replaces `lm_logits = self.lm_head(sequence_output)` + `CrossEntropyLoss(ignore_index=-100)(lm_logits.view(-1, V),
 * labels.view(-1))` of T5ForDecoder.forward (thinkdiff/models/mllama_vllm_t5_embed_decoder_2.py:236-246) under the bf16
 * autocast of tasks/base_task.py:237, and the backward of both down to the decoder output:
 *   logits[R, V]  = bf16(seq[R, K] . W_lm[V, K]^T)                     tcgen05 GEMM (lm_head has no bias, T5Config)
 *   loss          = mean over rows with label != -100 of logsumexp(logits) - logits[label]   (fp32; row staged in smem, one read)
 *   dlogits[R, V] = bf16((softmax - onehot) * grad_scale / n_valid)   same pass; may alias `logits` (in place) to save R*V*2 bytes
 *   dseq[R, K]    = bf16(dlogits . W_lm)                               tcgen05 GEMM, W_lm read in place (frozen: no dW)
 * `dlogits` and `dseq` may both be NULL (evaluation: loss only). `tie_word_embeddings` checkpoints scale seq by K^-0.5 first
 * (:231-234); google/flan-t5-xxl -- the checkpoint every shipped config names -- is untied, so no scale is applied here.
 * Needs K % 64 == 0, V % 32 == 0. */
int64_t td_lm_head_ce_workspace_bytes(int64_t R);
int32_t td_lm_head_ce_fwd_bwd(const void* seq, int64_t R, int32_t K, const void* W_lm, int32_t V, const int64_t* labels,
                              float grad_scale, float* loss, void* logits /* [R, V] bf16 */,
                              void* dlogits /* [R, V] bf16, may be == logits, may be NULL */,
                              void* dseq /* [R, K] bf16, may be NULL */, void* workspace, int64_t workspace_bytes,
                              td_stream_t stream);

/* ---- SURVEY section 8 f-1: the frozen T5 decoder's attention core on PACKED rows -----------------------------------------
 * Replaces the score / softmax / value product of transformers' T5Attention.forward (models/t5/modeling_t5.py, transformers==4.46.1
 * as pinned by requirements.txt:14) for both of a decoder block's uses, called from T5ForDecoder.forward
 * (thinkdiff/models/mllama_vllm_t5_embed_decoder_2.py:211-224) under the bf16 autocast of tasks/base_task.py:237:
 *   cross (self_attention = 0): decoder rows cu_q[b]..cu_q[b+1] attend to aligner rows cu_k[b]..cu_k[b+1]   s = q.k
 *   self  (self_attention = 1): decoder rows attend to the same rows (cu_k must be NULL or cu_q), causal    s = q.k + bias
 * with T5's rules: no 1/sqrt(d_kv) scaling, fp32 softmax, d_kv = 64. The relative position bias arrives as a per-distance table
 * bias_by_distance [H, n_dist] (fp32; row h = head h), entry min(i - j, n_dist - 1) for query position i >= key position j, both
 * counted from the sample's first row (n_dist = max_distance = 128 is exact for T5's 32 buckets: every distance >= 113 is in the
 * last bucket). Cross-attention takes no table.
 *   Q [Mq, >= inner], K / V [Mk, >= inner], O [Mq, >= inner] bf16 with row pitches ld* (elements, multiples of 8; Q/K/V may be column
 *   slices of one fused projection output), inner = 64 H columns per row, head h = columns [64 h, 64 h + 64).
 *   lse [H, Mq] fp32 (natural-log softmax normaliser per row and head; NULL = inference). A sample with no keys gets O = 0 and
 *   lse = -inf. max_len_q / max_len_k bound every sample's length (host-known, like flash-attn's max_seqlen): the grid is
 *   (ceil(max_len / 128), H, B); cu_* stay on the device and nothing synchronises. Rows outside every sample are not written.
 * The backward writes dQ [Mq], dK, dV [Mk] (bf16, pitches lddq / lddk / lddv: dK and dV may be the two halves of one [Mk, 2 inner]
 * buffer, the input gradient of a fused [Wk; Wv] projection) in three launches: Delta = rowsum(dO * O) into the workspace, dK / dV
 * (one CTA per key tile), dQ (one CTA per query tile). Deterministic: every output element is written once, no atomics. Keys of a
 * sample that no query sees get zero dK / dV. The bias table is frozen: it has no gradient.
 * Profiling tags: attn_fwd, attn_bwd_delta (bytes), attn_bwd_dkdv, attn_bwd_dq (FLOPs of the products each kernel runs, over the
 * VISIBLE (query, key) pairs only: 4, 8 and 6 x 64 H per pair). While profiling is enabled a call copies cu_* to the host to count
 * the pairs (a synchronisation of `stream`). */
int64_t td_t5_attention_workspace_bytes(int64_t Mq, int32_t H);
int32_t td_t5_attention_fwd(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                            const int32_t* cu_q, const int32_t* cu_k, int32_t B, int32_t H, int32_t inner, int32_t max_len_q,
                            int32_t max_len_k, int64_t Mq, int32_t self_attention, const float* bias_by_distance /* [H, n_dist] or NULL */,
                            int32_t n_dist, void* o, int64_t ldo, float* lse /* [H, Mq] or NULL */, td_stream_t stream);
int32_t td_t5_attention_bwd(const void* dout, int64_t lddo, const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v,
                            int64_t ldv, const int32_t* cu_q, const int32_t* cu_k, int32_t B, int32_t H, int32_t inner,
                            int32_t max_len_q, int32_t max_len_k, int64_t Mq, int32_t self_attention, const float* bias_by_distance,
                            int32_t n_dist, const void* o, int64_t ldo, const float* lse, void* dq, int64_t lddq, void* dk,
                            int64_t lddk, void* dv, int64_t lddv, void* workspace, int64_t workspace_bytes, td_stream_t stream);

/* ---- SURVEY section 8 f-1: the frozen T5 decoder's feed-forward sublayer on PACKED rows ------------------------------------
 * transformers' T5LayerFF with T5DenseGatedActDense (feed_forward_proj = "gated-gelu", Flan-T5), the model cast to bf16 and run
 * under bf16 autocast with dropout off, rounded where HF materialises a bf16 tensor and accumulated in fp32:
 *   rstd = rsqrt(mean(x^2) + eps)            xn = bf16(bf16(ln_w) * bf16(x * rstd))      (td_rmsnorm_fwd's bf16 rule)
 *   a = bf16(xn . wi_0^T)   b = bf16(xn . wi_1^T)   g = bf16(bf16(gelu_new(a)) * b)   out = bf16(x + bf16(g . wo^T))
 * gelu_new (tanh form) is evaluated once in fp32 from a. The backward gives the gradient to x only (the weights are frozen):
 *   t = bf16(dy . wo)   d_b = bf16(t * bf16(gelu_new(a)))   d_a = bf16(bf16(t * b) * gelu_new'(a))   dxn = bf16([d_a|d_b] . [wi_0; wi_1])
 *   dx = bf16(dy + rstd * ln_w * dxn - x * rstd^3 * mean(x * ln_w * dxn))
 * x, out, dy, dx [M, d] bf16; ln_w [d] fp32; rstd [M] fp32 (written by the forward); wo [d, d_ff] bf16 (nn.Linear layout);
 * wi [2 d_ff, d] bf16 holds wi_0 and wi_1 INTERLEAVED in blocks of 32 rows: rows [64k, 64k + 32) = wi_0 rows [32k, 32k + 32),
 * rows [64k + 32, 64k + 64) = wi_1 rows [32k, 32k + 32). ab / d_ab [M, 2 d_ff] bf16 carry a / b (their gradients) in the same
 * column order; gated [M, d_ff] bf16 is g. ab = NULL (inference) skips writing it; gated = NULL and d_ab = NULL keep them in the
 * workspace. Every buffer is contiguous and 16-byte aligned. Needs d % 64 == 0, d <= 4096, d_ff % 32 == 0; M == 0 does nothing.
 * Forward: 3 launches (norm, [wi_0; wi_1] GEMM with the gate in its epilogue, wo GEMM with the residual add in its epilogue);
 * backward: 3 launches (dy . wo GEMM with the gate's backward in its epilogue, d_ab . wi GEMM, norm backward with the residual).
 * Profiling tags: ffn_norm, gemm_ffn_gate, gemm_ffn_out, gemm_ffn_dgate, gemm_ffn_dx (2 M N K FLOPs each), ffn_norm_bwd (bytes). */
int64_t td_t5_ffn_workspace_bytes(int64_t M, int32_t d, int32_t d_ff);
int32_t td_t5_ffn_fwd(const void* x, int64_t M, int32_t d, int32_t d_ff, const float* ln_w, float eps, const void* wi, const void* wo,
                      void* out, float* rstd, void* ab /* [M, 2 d_ff] or NULL */, void* gated /* [M, d_ff] or NULL */, void* workspace,
                      int64_t workspace_bytes, td_stream_t stream);
int32_t td_t5_ffn_bwd(const void* dy, const void* x, const float* rstd, const float* ln_w, const void* ab, const void* wi, const void* wo,
                      int64_t M, int32_t d, int32_t d_ff, void* dx, void* d_ab /* [M, 2 d_ff] or NULL */, void* workspace,
                      int64_t workspace_bytes, td_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* THINKDIFF_B200_H */

/*
 * aa_b200.h -- C ABI of libaa_b200.so: the B200 (sm_100a) implementation of
 * align-anything's RLHF loss hot path.
 *
 * The reference (PKU-Alignment/align-anything) has NO FFI layer for this path:
 * the boundary is plain Python (module-level helpers in align_anything/utils/tools.py
 * and methods on the trainer classes).  Each entry point below names the reference
 * function(s) whose arithmetic it replaces (file:line relative to the reference's
 * align_anything/ directory); the Python mirror in align_anything_b200/ keeps the
 * reference's names and signatures and calls these through ctypes (INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - the caller owns every buffer (inputs, outputs, scratch); the library allocates
 *     nothing and keeps no state besides a thread-local error string;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no entry
 *     point synchronises the host;
 *   - return value: 0 on success, AA_ERR_* (<0) for argument errors, or a positive
 *     cudaError_t from the launch.  aa_last_error() gives the text;
 *   - offsets / strides are in ELEMENTS of the tensor they index;
 *   - `mode`: AA_MODE_FAITHFUL reproduces the reference's rounding points when the
 *     tensors are bf16/f16 (fp32 arithmetic, round-to-nearest-even to the tensor dtype
 *     where the reference's eager ops round); AA_MODE_F32 keeps fp32 throughout;
 *     AA_MODE_CE (K6 / K6b only) rounds the logits to bf16 like nn.Linear's output and keeps the
 *     log-softmax in fp32: the rounding of transformers' ForCausalLMLoss, which upcasts the logits.
 */
#ifndef AA_B200_H_
#define AA_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AA_B200_ABI_VERSION 3

enum { AA_BF16 = 0, AA_F16 = 1, AA_F32 = 2 };
enum { AA_MODE_FAITHFUL = 0, AA_MODE_F32 = 1, AA_MODE_CE = 2 };
enum { AA_MASK_U8 = 0, AA_MASK_I64 = 1 };

enum {
  AA_OK = 0,
  AA_ERR_DTYPE = -1,
  AA_ERR_ARG = -2,
  AA_ERR_ALIGN = -3,
  AA_ERR_UNSUPPORTED = -4
};

/* bits OR-ed into the device status word by kernels (never cleared by the library) */
enum {
  AA_STATUS_LABEL_OOB = 1,      /* a label outside [0, V): torch.gather would raise           */
  AA_STATUS_SHORT_SEQUENCE = 2, /* fewer non-pad tokens than response_len (dpo.py:135-137)   */
  AA_STATUS_EMPTY_MASK = 4,     /* a mask row with no True: m.nonzero()[-1] would raise       */
  AA_STATUS_DIVERGE_RANGE = 8   /* simpo.py:72-73 `assert 0 <= diverge_index <= end_index` fails */
};

/* Descriptor of the one-shot NVLink all-reduce fused into the metric-producing kernels (multi-GPU only).
 * peer_bufs: DEVICE array [world] of peer-mapped pointers to each rank's symmetric buffer of
 * 2 * world * 16 floats + world uint32 flags, zero-initialised once (torch.distributed._symmetric_memory
 * gives such pointers).  epoch: 1, 2, 3, ... incremented by the caller on every use, identically on every
 * rank.  max_lanes: bit t set -> lane t is MAX-reduced, otherwise averaged (utils/multi_process.py:74-89). */
typedef struct aa_coll {
  void *const *peer_bufs;
  int32_t rank;
  int32_t world;
  uint32_t epoch;
  uint32_t max_lanes;
} aa_coll;

int aa_abi_version(void);
const char *aa_last_error(void);
/* Number of SMs / max dynamic smem of the current device (for host-side grid sizing). */
int aa_device_info(int *sm_count, int *max_smem_optin);
/* Tuning / diagnostic knobs (process-wide).  variant = kernel digit + 10 * shape code.
 *   forward  kernel digit: 0 = vectorised LDG (default), 1 = cp.async.bulk staged through shared memory;
 *            shape: 0 = default (128 threads x 8 vectors x 16 CTAs/SM), 1 = 256x8, 2 = 512x4, 3 = 128x8, 4 = 256x2, 5 = 512x2.
 *   backward kernel digit: 0 / 1 = TMA-staged (cp.async.bulk loads AND stores through a shared-memory ring;
 *            the default whenever row_scratch is given), 2 = experimental address-ordered chunked sweep,
 *            3 = one-CTA-per-row LDG/STG kernel (also used when row_scratch == NULL);
 *            shape (TMA): 0 = 4 stages x 8 KB, lag 3, 3 CTAs/SM (default); see logprob.cu for the others.
 * ctas_per_sm <= 0 keeps the default persistent-grid size. */
int aa_logprob_set_tuning(int variant, int ctas_per_sm);
/* Same, for K1b only (variant -1: follow aa_logprob_set_tuning). */
int aa_logprob_set_tuning_bwd(int variant, int ctas_per_sm);

/* ---------------------------------------------------------------------------------------
 * K1  per-token log-prob: row log-softmax over V fused with the label gather.
 * Replaces utils/tools.py:402-413 gather_log_probabilities and the per-sample slicing loop
 * around it (trainers/text_to_text/dpo.py:133-142, text_image_to_text/ppo.py:229-239).
 *
 * A "segment" is one run of consecutive logits rows scored against consecutive labels
 * (one sample's response tail, or one whole sample).  Segment s covers flat rows
 * [seg_cum[s], seg_cum[s+1]); its j-th row reads logits[seg_logit_off[s] + j*row_stride + 0..V),
 * label labels[seg_label_off[s] + j], and writes out[seg_out_off[s] + j].
 *
 *   out         : out_dtype (the logits dtype in FAITHFUL mode -> same rounding as
 *                 F.log_softmax's output; AA_F32 otherwise)
 *   stat_max, stat_logsum : optional fp32 [n_rows] (flat row order) saved for K1b.
 *   status      : optional device int32 word, see AA_STATUS_*.
 *   use_ignore  : != 0 -> rows whose label == ignore_index are skipped (out = 0, no traffic; K1b
 *                 zero-fills them): the cross-entropy `ignore_index` of the SFT / PTX loss.
 * Algorithmic HBM traffic: V * sizeof(logit) bytes per row, read once.
 * ------------------------------------------------------------------------------------- */
int aa_logprob_fwd(const void *logits, int logits_dtype, int64_t row_stride, int32_t V,
                   const int64_t *labels, int64_t ignore_index, int32_t use_ignore,
                   int32_t n_segments, int64_t n_rows,
                   const int64_t *seg_logit_off, const int64_t *seg_label_off,
                   const int64_t *seg_out_off, const int64_t *seg_cum,
                   void *out, int out_dtype, float *stat_max, float *stat_logsum,
                   int32_t *status, void *stream);

/* ---------------------------------------------------------------------------------------
 * K1b  d(log-prob)/d(logits): autograd of the two ops above (ATen _log_softmax_backward_data
 * + gather backward) in ONE pass: grad[j] = g * ([j == label] - softmax_j), written in the
 * logits dtype.  g for flat row r of segment s is
 *     (grad_rows ? grad_rows[seg_out_off[s] + j] : 1) * (grad_seg ? grad_seg[s] : 1)
 *                                                   * (grad_scale ? *grad_scale : 1)
 * (grad_scale: one device scalar of dtype grad_scale_dtype -- the upstream d loss of a fused loss node, read as it is).
 * The gradient tile is `n_tile_rows` rows of `grad_row_stride` elements; segment s owns tile
 * rows [seg_tile_row[s], seg_tile_row[s] + n_s) (ascending, non-overlapping); every other
 * tile row is ZERO-FILLED by the same kernel (the reference's autograd materialises those
 * zeros through the slice / pad backward).  n_tile_rows == 0: only scored rows are written,
 * at grad_logits + seg_tile_row[s]*grad_row_stride, followed by the `n_extra_zero_rows` tile rows
 * listed in `extra_zero_rows` (device, int64), which are zero-filled.  A caller that knows the row
 * layout on the host uses this form together with aa_zero_rows: long zero spans go to the copy
 * engine (cudaMemsetAsync: 7.4 TB/s on B200 vs 6.45 TB/s for stores issued by a kernel), isolated
 * zero rows are listed, and the kernel's static row stride sees equally expensive rows first.
 * FAITHFUL mode recomputes softmax_j as exp(round_dtype((x_j - max) - logsum)), which is what
 * the reference's backward sees (it re-reads the ROUNDED log-softmax output).
 * row_scratch: 16-byte aligned device scratch of 32 bytes per work row (n_tile_rows, or
 * n_rows + n_extra_zero_rows when n_tile_rows == 0).  With it the backward is TMA-staged: a tiny prep kernel resolves every row into a
 * 32-byte record, then a persistent kernel moves the tile with cp.async.bulk in both directions through
 * a shared-memory ring (6.48 TB/s sustained at V = 128257 vs 5.8 TB/s for the LDG/STG kernel that runs
 * when row_scratch == NULL).
 * Algorithmic HBM traffic: 2 * V * sizeof(logit) per scored row (+ V * sizeof per zero row).
 * ------------------------------------------------------------------------------------- */
int aa_logprob_bwd(const void *logits, int logits_dtype, int64_t row_stride, int32_t V,
                   const int64_t *labels, int64_t ignore_index, int32_t use_ignore,
                   int32_t n_segments, int64_t n_rows,
                   const int64_t *seg_logit_off, const int64_t *seg_label_off,
                   const int64_t *seg_out_off, const int64_t *seg_cum,
                   const int64_t *seg_tile_row,
                   const float *stat_max, const float *stat_logsum,
                   const void *grad_rows, int grad_rows_dtype, const float *grad_seg,
                   const void *grad_scale, int grad_scale_dtype,
                   void *grad_logits, int64_t grad_row_stride, int64_t n_tile_rows,
                   const int64_t *extra_zero_rows, int64_t n_extra_zero_rows,
                   void *row_scratch, int mode, void *stream);

/* Zero-fill row spans of an (n_tile_rows, V) tile with the copy engine.  spans_host: n_spans pairs
 * (first_row, n_rows) in HOST memory (read during the call); rows are row_stride elements apart.
 * Used for the prompt / padding rows of the gradient tile, BEFORE aa_logprob_bwd on the same stream:
 * for a contiguous tile (row_stride == V) each span is widened to 256-byte boundaries inside the tile
 * (an unaligned memset runs far below the copy engine's rate and rows of an odd V start 2-byte
 * aligned), i.e. up to 255 bytes of the neighbouring rows are cleared too -- aa_logprob_bwd rewrites
 * those rows in full afterwards.  Pitched tiles (row_stride > V) are cleared exactly. */
int aa_zero_rows(void *tile, int dtype, int64_t row_stride, int32_t V, int64_t n_tile_rows,
                 const int64_t *spans_host, int32_t n_spans, void *stream);

/* ---------------------------------------------------------------------------------------
 * Label extraction for DPO: labels of sample i = strip_pad(input_ids[i])[-R_i:]
 * (trainers/text_to_text/dpo.py:52-54, :135-137): the last R_i tokens that are != pad,
 * wherever the pads sit.  strip == 0 reproduces text_audio_to_text/dpo.py:100 (plain tail).
 * Writes labels_out[i*out_stride + k], k in [0, R_i) (bit-exact int64 copy).
 * ------------------------------------------------------------------------------------- */
int aa_strip_pad_tail(const int64_t *input_ids, int32_t n_samples, int32_t L, int64_t ids_row_stride,
                      int64_t pad_id, int strip, const int32_t *response_lens,
                      int64_t *labels_out, int64_t out_stride, int32_t *status, void *stream);

/* ---------------------------------------------------------------------------------------
 * K2  DPO pairwise loss + metrics.  Replaces trainers/text_to_text/dpo.py:166-203 (loss) and
 * :215-221 (local means); text_audio_to_text/dpo.py:134-139 when `input_ids` != NULL (pairs
 * whose chosen / rejected id rows are identical are dropped).
 *   policy_lp, ref_lp : (2*n_pairs, width), rows 0..n_pairs-1 chosen, rest rejected, zero padded.
 *   per_pair : fp32 [5][n_pairs] = loss_i, better_reward_i, worse_reward_i,
 *              g_i (= d mean-loss / d chosen-logp-sum_i ; rejected gets -g_i), valid_i (0/1).
 *   grad_seg : optional fp32 [2*n_pairs] = (+g_i ..., -g_i ...) ready for aa_logprob_bwd.
 *   stats    : fp32 [8] = loss, reward, better_sample_reward, worse_sample_reward,
 *              reward_accuracy, reward_margin (all means over valid pairs), n_valid, status.
 *   status   : optional device status word (AA_STATUS_* bits set by K1 / the label kernels earlier on the
 *              stream); its value is copied into stats[7] so that the caller's ONE host read of the metrics
 *              also tells it whether the reference would have raised (lane 7 is MAX-reduced across ranks).
 *   counter  : device uint32 scratch, zero before first use (the kernel re-zeroes it).
 *   coll / stats_global : optional (NULL on one GPU).  With them the last block of K2 also performs the
 *              step's packed all-reduce (trainers/text_to_text/dpo.py:222-227) over NVLink peer memory and
 *              writes the reduced vector to stats_global[8]; `stats` always holds the LOCAL values (the
 *              loss that is back-propagated is the local mean, as in the reference).
 * ------------------------------------------------------------------------------------- */
int aa_dpo_loss(const void *policy_lp, const void *ref_lp, int lp_dtype, int32_t n_pairs,
                int32_t width, int64_t lp_row_stride, float scale_coeff, int mode,
                const int64_t *input_ids, int32_t L, int64_t ids_row_stride,
                float *per_pair, float *grad_seg, float *stats, uint32_t *counter,
                const aa_coll *coll, float *stats_global, const int32_t *status, void *stream);

/* ---------------------------------------------------------------------------------------
 * Pair bookkeeping and slice sums of SimPO / ORPO / KTO (SURVEY.md 8f row 2).
 * aa_pair_slices: trainers/text_to_text/simpo.py:61-77 (orpo.py:61-77, kto.py:111-125): identical-pair test, last
 *   attended index of both rows, first index where the id rows differ -> out int32 [4][n_pairs] =
 *   valid, diverge_index, end_better, end_worse (bit-exact; 4 host syncs per pair in the reference).
 * aa_slice_sums: sums[r] = sum(lp[r, diverge : end + 1]) (simpo.py:78-79; Python slice semantics on the (2B, W)
 *   zero-padded log-prob rows), fp32 accumulate, rounded to the lp dtype in FAITHFUL mode; fp32 [2 * n_pairs] out.
 * The O(B) scalar formulas on top (log-ratio, log-sigmoid, odds ratio ...) are elementwise ATen ops on B-vectors in
 * the Python mirror -- bit-identical to the reference by construction; every O(rows * V) byte still goes through K1.
 * ------------------------------------------------------------------------------------- */
int aa_pair_slices(const int64_t *input_ids, int64_t ids_row_stride, const void *attention_mask, int mask_kind,
                   int64_t mask_row_stride, int32_t n_pairs, int32_t L, int32_t *out, int32_t *status, void *stream);
int aa_slice_sums(const void *lp, int lp_dtype, int64_t lp_row_stride, int32_t n_pairs, int32_t width,
                  const int32_t *slices, int mode, float *sums, void *stream);

/* ---------------------------------------------------------------------------------------
 * Reward-model pairwise loss (sibling of K2; SURVEY.md 8f row 2).  Replaces the loss tail of
 * trainers/text_to_text/rm.py:97-132: end_scores fp32 [2*n_pairs] (higher first, lower second) ->
 *   out[0] = mean(-logsigmoid(higher - lower)) + regularization * mean(square(all 2B scores)),
 *   out[1] = accuracy = mean(higher > lower);  grad_end_scores (optional) = d out[0] / d end_scores.
 * ------------------------------------------------------------------------------------- */
int aa_rm_pair_loss(const float *end_scores, int32_t n_pairs, float regularization, float *out,
                    float *grad_end_scores, void *stream);

/* ---------------------------------------------------------------------------------------
 * K3  scalar score head of the reward / critic models: scores[r] = <hidden[r,:], w>.
 * Replaces `self.score_head(last_hidden_state)` (models/llama.py:62-63, opt.py, llava.py:62-63,
 * qwen2_vl.py:59-60, qwen2_audio.py:77-78).  FAITHFUL: fp32 dot rounded to the hidden dtype
 * (what nn.Linear returns) and then widened if out_dtype is AA_F32 (`.float()`).
 * A GEMV (N = 1): HBM-bound on reading hidden, H * sizeof per row.
 * ------------------------------------------------------------------------------------- */
int aa_score_head_fwd(const void *hidden, int dtype, int64_t n_rows, int32_t H, int64_t row_stride,
                      const void *weight, void *scores, int out_dtype, int mode, void *stream);

/* end_index = last nonzero of each attention-mask row (models/llama.py:71 `m.nonzero()[-1]`),
 * or L-1 when mask == NULL (llava.py:64-66 / qwen2_vl.py:62-64 take position -1);
 * end_scores[b] = scores[b, end_index[b]] (fp32); optional end_hidden (B, H) gather. */
int aa_score_end(const void *scores, int scores_dtype, int64_t scores_row_stride,
                 const void *mask, int mask_kind, int64_t mask_row_stride, int32_t B, int32_t L,
                 int64_t *end_index, float *end_scores,
                 const void *hidden, int hidden_dtype, int64_t hidden_batch_stride,
                 int64_t hidden_row_stride, int32_t H, void *end_hidden,
                 int32_t *status, void *stream);

/* Backward of the head: grad_hidden[r,:] = g[r] * w  (dtype of hidden), and
 * grad_weight[:] = sum_r g[r] * hidden[r,:] (fp32, deterministic two-stage reduction through
 * `partial` = fp32 [n_partials][H] scratch; n_partials = value returned in *n_partials_needed
 * when partial == NULL). */
int aa_score_head_bwd(const void *hidden, int dtype, int64_t n_rows, int32_t H, int64_t row_stride,
                      const void *weight, const void *grad_scores, int grad_dtype,
                      void *grad_hidden, int64_t grad_row_stride, float *grad_weight,
                      float *partial, int32_t *n_partials_needed, int mode, void *stream);

/* ---------------------------------------------------------------------------------------
 * K4  PPO preparation, one launch: KL-shaped rewards, GAE reverse scan, returns.
 * Replaces trainers/text_to_text/ppo.py:528-547 (add_kl_divergence_regularization) and
 * :487-508 (get_advantages_and_returns) -- a Python loop over t in the reference -- plus the
 * row sums behind the kl_divergence / reward_with_kl_penalty / generated-length metrics
 * (:361-369).  All 2-D inputs are (B, W) with their own row strides; mask is torch.bool.
 *   old_rewards : (B, W) lp dtype (FAITHFUL) or fp32
 *   advantages, returns : (B, W - start), `adv_dtype` (torch promotion of values x rewards)
 *   row_stats : fp32 [B][8] = kl_sum, reward_kl_sum, mask_count(start..), adv_row_mean,
 *               ret_row_mean, end_index, 0, 0
 * log_probs == ref_log_probs == reward == NULL: GAE only -- `old_rewards` is then an INPUT holding
 * precomputed per-token rewards (PPOTrainer.get_advantages_and_returns called on its own).
 * The scan is a warp-shuffle affine scan (A_t = d_t + gamma*lambda*A_{t+1}) in fp32; when
 * adv_dtype is 16-bit in FAITHFUL mode the recurrence is evaluated sequentially with the
 * reference's per-op rounding so that results are reproducible bit for bit.
 * ------------------------------------------------------------------------------------- */
int aa_ppo_prep(const void *log_probs, const void *ref_log_probs, int lp_dtype, int64_t lp_row_stride,
                const float *reward, const void *values, int val_dtype, int64_t val_row_stride,
                const uint8_t *mask, int64_t mask_row_stride, int32_t B, int32_t W, int32_t start,
                float kl_coeff, float clip_range_score, float gamma, float gae_lambda, int mode,
                void *old_rewards, int rew_dtype, void *advantages, void *returns, int adv_dtype,
                float *row_stats, int32_t *status, void *stream);

/* ---------------------------------------------------------------------------------------
 * K5  PPO losses, forward AND backward in one launch each (the backward is elementwise).
 * actor : trainers/text_to_text/ppo.py:291-307  (+ utils/tools.py:460-467 masked_mean)
 * critic: trainers/text_to_text/ppo.py:510-526
 * Inputs are (B, Wm) views (caller passes pointers already offset to column `start`).
 *   loss      : fp32 [2]: [0] = the loss; when the promoted dtype of the inputs is 16-bit, the first two bytes of [1]
 *               hold the same value in that dtype (the caller views it as the 0-dim bf16 / f16 tensor the reference's
 *               loss is: no conversion launch)
 *   grad      : (B, Wm) d loss / d new_log_probs (resp. new values), input dtype, or NULL
 *   value_tail_lens / value_src_width (critic, optional): `values` is then the RAW (B, value_src_width) tensor
 *               `scores.squeeze(-1)[:, :-1]` and the kernel reads values[b, t] = t < R_b ? raw[b, value_src_width - R_b + t] : 0
 *               (the pad_sequence of per-sample tails of text_image_to_text/ppo.py:318-330 folded into the load);
 *               aa_tail_scatter_scaled is its adjoint.
 *   row_mean  : optional fp32 [B], masked row mean of `new` values (critic: reward_value metric)
 *   counter   : device uint32 scratch (zero before first use; self-cleaning)
 * ------------------------------------------------------------------------------------- */
int aa_ppo_actor_loss(const void *log_probs, int64_t lp_stride, const void *old_log_probs,
                      int64_t old_stride, int lp_dtype, const void *advantages, int64_t adv_stride,
                      int adv_dtype, const uint8_t *mask, int64_t mask_stride, int32_t B, int32_t Wm,
                      float clip_range_ratio, int mode, float *loss, void *grad, int64_t grad_stride,
                      float *row_scratch, uint32_t *counter, void *stream);

int aa_ppo_critic_loss(const void *values, int64_t val_stride, const void *old_values,
                       int64_t old_stride, int val_dtype, const void *returns, int64_t ret_stride,
                       int ret_dtype, const uint8_t *mask, int64_t mask_stride, int32_t B, int32_t Wm,
                       float clip_range_value, int mode, float *loss, void *grad, int64_t grad_stride,
                       float *row_mean, float *row_scratch, uint32_t *counter, const int32_t *value_tail_lens,
                       int32_t value_src_width, void *stream);

/* Adjoint of the tail gather above times an upstream scalar, one launch for the whole (B, out_width) tile (zeros
 * included): out[b, t] = src_width - R_b <= t < src_width ? scale * grad[b, t - (src_width - R_b)] : 0.  grad (B, W) and out
 * share `dtype`; scale: optional device scalar of scale_dtype (fp32 product, rounded once).  Replaces the autograd of
 * `scores.squeeze(-1)[:, :-1]` + per-sample slicing + pad_sequence (SliceBackward / CatBackward / a zero-filled tile). */
int aa_tail_scatter_scaled(const void *grad, int dtype, int64_t grad_row_stride, const int32_t *lens, int32_t B, int32_t W,
                           int32_t src_width, const void *scale, int scale_dtype, void *out, int64_t out_row_stride,
                           int32_t out_width, void *stream);

/* ---------------------------------------------------------------------------------------
 * K1f  The actor half of a PPO rl_step in ONE pass over the logits tile: log-probs of the response tails
 * (K1), d actor_loss / d log-prob per token (K5's arithmetic) and the gradient tile (K1b) -- the clipped-ratio
 * objective is a masked mean of per-token terms, so a row's gradient only needs that row's own log-prob plus values
 * known before the forward.  Each scored row is streamed twice by the same CTA (the second pass is served by the
 * 126 MB L2), so HBM sees V*e read + V*e written per scored row instead of 2*V*e + V*e.
 * Replaces trainers/text_image_to_text/ppo.py:296-316 (text: trainers/text_to_text/ppo.py:336-349):
 * actor forward logits -> gather_log_probabilities -> actor_loss_fn -> backward up to d logits.
 *   row plan    : as aa_logprob_bwd in tile mode (segments = samples, n_tile_rows / n_segments tile rows each;
 *                 host RowPlan or aa_tail_plan_build table)
 *   log_probs   : (n_segments, W) lp_dtype, zero-initialised by the caller (pad columns stay 0)
 *   stat_*      : optional fp32 [n scored rows] (max, logsum) as aa_logprob_fwd
 *   old_log_probs (lp_dtype) / advantages / mask : (n_segments, W) with element row strides
 *   grad_logits : every tile row is written (scored rows: d loss / d logits for an upstream gradient of 1; others 0)
 *   row_scratch : device scratch, 48 bytes per tile row, 16-byte aligned
 * The loss VALUE is aa_ppo_actor_loss on `log_probs`; aa_scale_tile applies an upstream scalar != 1. */
int aa_logprob_actor_fused(const void *logits, int logits_dtype, int64_t row_stride, int32_t V,
                           const int64_t *labels, int32_t n_segments, const int64_t *seg_logit_off,
                           const int64_t *seg_label_off, const int64_t *seg_out_off, const int64_t *seg_cum,
                           const int64_t *seg_tile_row, int64_t n_tile_rows, void *log_probs, int lp_dtype,
                           float *stat_max, float *stat_logsum, const void *old_log_probs, int64_t old_stride,
                           const void *advantages, int64_t adv_stride, int adv_dtype, const uint8_t *mask,
                           int64_t mask_stride, int32_t W, float clip_range_ratio, int mode, void *grad_logits,
                           int64_t grad_row_stride, void *row_scratch, int32_t *status, void *stream);

/* The same single pass for the mean cross-entropy behind `outputs.loss` (trainers/text_to_text/sft.py:95-98
 * `SupervisedTrainer.loss`, ppo.py:400-408 `ptx_step`; transformers' ForCausalLMLoss): every row whose label !=
 * ignore_index has the upstream gradient -loss_scale / n_valid, known before the row is read, so the fp32 log-probs
 * AND d (loss_scale * loss) / d logits come out of one pass over the valid rows (HBM: V*e read + V*e written per valid
 * row; aa_logprob_fwd + aa_logprob_bwd: 2*V*e + V*e).  Ignored rows cost no reads (log-prob 0, zero gradient row).
 *   labels      : the SHIFTED labels the row plan addresses; n_labels = how many of them to count for n_valid
 *   log_probs   : fp32, zero-initialised by the caller; the loss value is aa_nll_mean over it
 *   row_scratch : 48 bytes per tile row (16-byte aligned); coeff_scratch: one device float */
int aa_logprob_ce_fused(const void *logits, int logits_dtype, int64_t row_stride, int32_t V, const int64_t *labels,
                        int64_t n_labels, int64_t ignore_index, int32_t n_segments, const int64_t *seg_logit_off,
                        const int64_t *seg_label_off, const int64_t *seg_out_off, const int64_t *seg_cum,
                        const int64_t *seg_tile_row, int64_t n_tile_rows, float *log_probs, float loss_scale,
                        void *grad_logits, int64_t grad_row_stride, void *row_scratch, float *coeff_scratch,
                        int32_t *status, void *stream);

/* ... and for the GRPO loss (trainers/text_to_text/grpo.py:290-312): per-token loss -(exp(lp - lp.detach()) * A - beta * KL)
 * with the k3 KL against the reference log-probs, counted up to and including the first eos of each completion, token
 * mean.  d loss / d lp of a token needs its own log-prob, the reference model's log-prob (scored BEFORE this call) and
 * the sequence's group advantage.  Segments = sequences; log_probs (n_segments, K) lp_dtype zero-initialised by the
 * caller; ref_log_probs (n_segments, K) lp_dtype; advantages fp32 [n_segments]; completion_tokens (n_segments, K).
 * row_end (int32 [n_segments]) and total (fp32 [1]) are outputs of the mask pass; the loss VALUE is aa_grpo_loss on
 * `log_probs`.  counter: device uint32 scratch (zero before first use; self-cleaning). */
int aa_logprob_grpo_fused(const void *logits, int logits_dtype, int64_t row_stride, int32_t V, const int64_t *labels,
                          int32_t n_segments, const int64_t *seg_logit_off, const int64_t *seg_label_off,
                          const int64_t *seg_out_off, const int64_t *seg_cum, const int64_t *seg_tile_row,
                          int64_t n_tile_rows, void *log_probs, int lp_dtype, const void *ref_log_probs, int64_t ref_stride,
                          const float *advantages, const int64_t *completion_tokens, int64_t tok_stride, int64_t eos_id,
                          int32_t K, float beta, int mode, void *grad_logits, int64_t grad_row_stride, void *row_scratch,
                          int32_t *row_end, float *total, uint32_t *counter, int32_t *status, void *stream);

/* tile[0..n) *= *scale unless *scale == 1 (checked on the device: the usual `loss.backward()` costs one empty launch).
 * Contiguous tile; scale: device scalar of scale_dtype.  The autograd backward of the K1f node. */
int aa_scale_tile(void *tile, int dtype, int64_t n, const void *scale, int scale_dtype, void *stream);

/* ---------------------------------------------------------------------------------------
 * Mean negative log-likelihood over the rows whose label != ignore_index: the epilogue that turns
 * K1's per-token log-probs into the causal-LM cross-entropy behind `outputs.loss`
 * (trainers/text_to_text/sft.py:95-98 `SupervisedTrainer.loss`, ppo.py:400-408 `ptx_step`;
 * transformers' ForCausalLMLoss: fp32 log-softmax, mean over non-ignored tokens).
 *   loss[0] = -sum(logp[valid]) / n_valid ; neg_inv_count[0] = -1 / n_valid (the per-row upstream
 *   gradient that aa_logprob_bwd takes as grad_scale).  partial: fp32 [2 * 256] scratch.
 * ------------------------------------------------------------------------------------- */
int aa_nll_mean(const void *logp, int dtype, const int64_t *labels, int64_t n, int64_t ignore_index,
                float *loss, float *neg_inv_count, float *partial, uint32_t *counter, void *stream);

/* ---------------------------------------------------------------------------------------
 * GRPO (sibling of K5; SURVEY.md 8f row 2).  trainers/text_to_text/grpo.py:268-318.
 * aa_group_advantages: rewards fp32 [n_groups][group_size] -> (r - mean) / (std_unbiased + 1e-4)   (:268-274)
 * aa_grpo_loss: per-token KL exp(ref - lp) - (ref - lp) - 1, per-token loss -(A - beta * KL), completion mask up to
 *   and including the first eos of `completion_tokens` (B, K), loss = sum(masked) / sum(mask)      (:290-312),
 *   forward AND d loss / d log_probs (lp dtype; NULL to skip) in two launches.
 *   row_end: int32 [B] scratch (out: counted tokens per row); scratch: fp32 [1 + B]; counter: uint32 [2], zeroed once.
 * ------------------------------------------------------------------------------------- */
int aa_group_advantages(const float *rewards, int32_t n_groups, int32_t group_size, float *advantages, void *stream);
int aa_grpo_loss(const void *log_probs, int64_t lp_stride, const void *ref_log_probs, int64_t ref_stride, int lp_dtype,
                 const float *advantages, const int64_t *completion_tokens, int64_t tok_stride, int64_t eos_id,
                 int32_t B, int32_t K, float beta, int mode, float *loss, void *grad, int64_t grad_stride,
                 int32_t *row_end, float *scratch, uint32_t *counter, void *stream);

/* masked_mean (utils/tools.py:460-467): mean over rows of masked row means -> out[0];
 * mask == NULL: plain mean. */
int aa_masked_mean(const void *x, int dtype, int64_t x_stride, const uint8_t *mask, int64_t mask_stride,
                   int32_t B, int32_t W, float *out, float *row_scratch, uint32_t *counter, void *stream);

/* Pack the local PPO metrics (trainers/text_to_text/ppo.py:360-381) from the row statistics:
 * stats fp32 [12] = actor_loss, reward_critic_loss, reward, reward_with_kl_penalty,
 * reward_advantage, reward_return, reward_value, kl_divergence, mean_generated_length,
 * max_generated_length, status, 0 (status: the optional device status word, as in aa_dpo_loss; MAX lane).
 * Entries 0..8 are all-reduced with AVG, entries 9 and 10 with MAX; with `coll` the
 * kernel does that reduction itself over NVLink peer memory (the reference: 10 NCCL launches + a barrier). */
int aa_ppo_pack_metrics(const float *row_stats, const float *reward, const float *value_row_mean,
                        const float *actor_loss, const float *critic_loss, int32_t B, float *stats,
                        const aa_coll *coll, const int32_t *status, void *stream);

/* The same one-shot NVLink all-reduce on its own: dst[0..n) = reduce over ranks of src[0..n), n <= 16 floats, src may
 * equal dst.  The DPO trainer launches it on a side stream right after K2, so that the wait for the slowest rank
 * overlaps K1b instead of sitting between K2 and K1b on the critical path. */
int aa_allreduce_packed(const float *src, float *dst, int32_t n, const aa_coll *coll, void *stream);

/* ---------------------------------------------------------------------------------------
 * K6  lm_head x log-prob in one kernel (SURVEY.md 8f rank 1; rows that carry no gradient):
 *   out[r] = log_softmax(hidden[r, :] @ weight^T)[labels[r]]
 * = gather_log_probabilities(lm_head(hidden), labels) (utils/tools.py:402-413 on the output of the model's
 * nn.Linear lm_head; callers trainers/text_to_text/dpo.py:128 (reference model), ppo.py:266-267 (rollout))
 * without the (n_rows, V) logits tile.  hidden (n_rows, H) and weight (V, H) are bf16, K-major, rows
 * 16-byte aligned (strides in elements, multiples of 8), H a multiple of 64; V is arbitrary (128257 works:
 * the odd leading dimension only exists in the tile that is never written).  tcgen05.mma (M128 N256 K16,
 * fp32 accumulators in TMEM), operands staged by TMA into a 4-stage 128-byte-swizzled ring, epilogue =
 * online (max, sum-exp) + label pick straight out of TMEM.  FAITHFUL: each logit is rounded to bf16 before
 * the softmax (the rounding point of nn.Linear) and the result is rounded to bf16.  stat_max / stat_logsum
 * (optional, n_rows fp32 each) receive the row statistics.  `partial` (optional, `partial_floats` fp32 of
 * device scratch; 3 * 148 * 128 always suffices): with fewer 128-row tiles than SMs the vocabulary is also
 * split across CTAs and the per-split (max, sum, label logit) are merged by a second tiny launch.  Needs a driver that exports
 * cuTensorMapEncodeTiled (resolved at run time; the library does not link libcuda).
 * Work: 2 * n_rows * H * V flops; HBM: weight + hidden read ~once (the weight sweep stays in L2).
 * ------------------------------------------------------------------------------------- */
int aa_linear_logprob_fwd(const void *hidden, int64_t n_rows, int32_t H, int64_t hidden_row_stride,
                          const void *weight, int32_t V, int64_t weight_row_stride, const int64_t *labels,
                          void *out, int out_dtype, float *stat_max, float *stat_logsum, float *partial,
                          int64_t partial_floats, int mode, int32_t *status, void *stream);

/* K6b: K6's pipeline with a store epilogue -- the first of the three backward kernels of the fused lm_head x
 * log-prob path.  Recomputes the logits tile on the tensor cores and writes
 *   dlogits[r, j] = g[r] * ([j == labels[r]] - softmax_j)      (bf16; FAITHFUL: softmax from the rounded log-softmax)
 * into a (n_rows, ld) buffer, ld >= ceil(V / 256) * 256 and a multiple of 8 (columns >= V are written as 0), from the
 * (max, logsum) K6 saved -- the "recompute + K1b" step of the lm_head backward in one kernel; d(hidden) and d(weight)
 * are aa_linear_dhidden / aa_linear_dweight on that buffer. */
int aa_linear_dlogits(const void *hidden, int64_t n_rows, int32_t H, int64_t hidden_row_stride,
                      const void *weight, int32_t V, int64_t weight_row_stride, const int64_t *labels,
                      const float *stat_max, const float *stat_logsum, const void *grad_rows,
                      int grad_rows_dtype, void *dlogits, int64_t ld, int mode, void *stream);

/* The two GEMMs that finish that backward: the autograd of the model's nn.Linear lm_head (callers
 * trainers/text_to_text/dpo.py:128, ppo.py:338) given the d(logits) buffer of aa_linear_dlogits.  Same tcgen05 / TMEM / TMA
 * pipeline as K6 (M128 N256 K16, fp32 accumulation), persistent grid, operands read in place:
 *   aa_linear_dhidden:  d_hidden (n_rows, H) bf16 = dlogits (n_rows, ld) . weight (V, H)       [columns >= V of dlogits
 *                       must be zero; the weight is consumed MN-major, vocabulary rows >= V are zero-filled by TMA]
 *   aa_linear_dweight:  (V, H) result = [acc_f32 if accumulate] + dlogits^T . hidden (n_rows, H), both operands MN-major.
 *                       Written to acc_f32 (fp32, row stride acc_row_stride) when d_weight == NULL, else rounded to bf16
 *                       into d_weight.  Row chunks: first chunk accumulate = 0, d_weight = NULL; middle chunks
 *                       accumulate = 1, d_weight = NULL; last chunk accumulate = 1, d_weight given -- one rounding at the
 *                       end, like a single GEMM over all rows.  A single chunk needs no fp32 buffer at all.
 * ld: multiple of 64, >= V; H: multiple of 64; all bases 16-byte aligned. */
int aa_linear_dhidden(const void *dlogits, int64_t n_rows, int64_t ld, const void *weight, int32_t V, int32_t H,
                      int64_t weight_row_stride, void *d_hidden, int64_t d_hidden_row_stride, void *stream);
int aa_linear_dweight(const void *dlogits, int64_t n_rows, int64_t ld, const void *hidden, int32_t H,
                      int64_t hidden_row_stride, int32_t V, float *acc_f32, int64_t acc_row_stride, int32_t accumulate,
                      void *d_weight, int64_t d_weight_row_stride, void *stream);

/* ---------------------------------------------------------------------------------------
 * Integer layout kernels (bit-exact).
 * move_padding_left : trainers/text_image_to_text/ppo.py:56-87 (utils/tools.py:615-639)
 * count_nonpad      : the host `.tolist()` bookkeeping at text_image_to_text/ppo.py:190-203
 *                     (response_len = nonpad(sequence) - nonpad(prompt))
 * ------------------------------------------------------------------------------------- */
int aa_move_padding_left(const int64_t *ids, int32_t B, int32_t L, int64_t row_stride, int64_t pad_id,
                         int64_t *out, void *stream);
int aa_count_nonpad(const int64_t *ids, int32_t B, int32_t L, int64_t row_stride, int64_t pad_id,
                    int32_t *counts, void *stream);

/* Everything trainers/text_image_to_text/ppo.py:185-203 does after `generate`, in one launch and without the host:
 * moved = move_padding_left(sequences) (B, L) int64; attention_mask = moved != pad (B, L) bytes (torch.bool);
 * response_lens[b] = max(nonpad(sequences[b]) - nonpad(prompt_ids[b]), 0) int32 (the reference: two `.tolist()` and a
 * Python list filter per sample). */
int aa_ppo_rollout_layout(const int64_t *prompt_ids, int32_t P, int64_t prompt_row_stride, const int64_t *sequences,
                          int32_t L, int64_t seq_row_stride, int32_t B, int64_t pad_id, int64_t *moved,
                          uint8_t *attention_mask, int32_t *response_lens, void *stream);

/* The K1 / K1b row plan of per-sample response tails built from DEVICE response lengths (the reference slices each
 * sample on the host, text_image_to_text/ppo.py:229-239).  table: int64 [5][B + 1] = seg_logit_off, seg_label_off,
 * seg_out_off, seg_cum, seg_tile_row as aa_logprob_fwd / aa_logprob_bwd take them (pass n_rows = B * width, the kernels
 * read the exact total from seg_cum[B]; the backward runs in tile mode, n_tile_rows = B * seq).  Sample b scores
 * n_b = clamp(lens[b] - label_shift, 0, width) rows from tile position seq - lens[b] + row_shift on, against
 * labels[b * label_row_stride + (label_tail_len > 0 ? label_tail_len - lens[b] : 0) + label_shift + j], results at
 * out[b * width + j].  Lengths that do not fit set AA_STATUS_SHORT_SEQUENCE and are clamped.
 * copies > 1 (table: [5][copies * B + 1]): the plan repeated for `copies` identically shaped logits tensors lying
 * copy_logit_delta ELEMENTS apart (their base pointers differ by that much), results copy_out_delta apart -- the actor
 * and the reference model of a rollout are then scored by ONE aa_logprob_fwd launch (forward only). */
int aa_tail_plan_build(const int32_t *response_lens, int32_t B, int32_t seq, int64_t sample_stride, int64_t row_stride,
                       int64_t label_row_stride, int32_t label_tail_len, int32_t label_shift, int32_t row_shift,
                       int32_t width, int32_t copies, int64_t copy_logit_delta, int64_t copy_out_delta, int64_t *table,
                       int32_t *status, void *stream);

/* The rows a causal-LM cross-entropy scores (transformers ForCausalLMLoss; trainers/text_to_text/sft.py:95-98, ppo.py:400-408),
 * for the lm_head path that never builds the logits tile: position (b, t) of a (B, L) batch is scored against the SHIFTED
 * label labels[b, t + 1] (the last position is ignored).  One launch writes, in ascending row order (which fixes the fp32
 * summation order of the loss), the flat indices b * L + t of the rows whose shifted label != ignore_index into
 * row_index_out, their labels into labels_out (both int64 [B * L] capacity) and their number into count_out[0] (int64).
 * A label that is neither ignore_index nor in [0, V) sets AA_STATUS_LABEL_OOB (ATen's cross_entropy would raise); the row
 * stays in the list.  Strides in elements. */
int aa_ce_rows(const int64_t *labels, int32_t B, int32_t L, int64_t label_batch_stride, int64_t label_row_stride,
               int64_t ignore_index, int32_t V, int64_t *row_index_out, int64_t *labels_out, int64_t *count_out,
               int32_t *status, void *stream);

/* pad_sequence([x[b][-R_b:] for b], batch_first=True) -- trainers/text_image_to_text/ppo.py:233-249 (rollout) and
 * :318-330 (rl_step: critic values), a Python loop + pad_sequence in the reference -- and its adjoint.
 *   adjoint = 0:  src (B, W), out (B, Rmax):  out[b, k] = k < R_b ? src[b, W - R_b + k] : 0
 *   adjoint = 1:  src (B, Rmax), out (B, W):  out[b, j] = j >= W - R_b ? src[b, j - (W - R_b)] : 0   (gradient)
 * src / out hold `dtype` elements (bit copies); lens (B,) int32 on the device, 0 <= R_b <= Rmax <= W. */
int aa_tail_rows(const void *src, int dtype, int64_t src_row_stride, const int32_t *lens, int32_t B, int32_t W,
                 int32_t Rmax, void *out, int64_t out_row_stride, int32_t adjoint, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* AA_B200_H_ */

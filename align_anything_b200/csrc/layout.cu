// layout.cu -- bit-exact integer kernels for the batch-layout steps that sit on the PPO path.
//
// aa_move_padding_left : trainers/text_image_to_text/ppo.py:56-87 (dup utils/tools.py:615-639);
//                        six ATen kernels in the reference.
// aa_count_nonpad      : the per-sample `.tolist()` + remove_pad_tokens bookkeeping at
//                        trainers/text_image_to_text/ppo.py:190-203 (a host round-trip per sample).
// aa_ce_rows           : the valid rows of a causal-LM cross-entropy (shifted labels != ignore_index), compacted in
//                        row order for the lm_head path that never builds the logits tile.
#include "common.cuh"

namespace aa {

template <int THREADS>
__global__ void __launch_bounds__(THREADS)
    move_padding_left_kernel(const int64_t *__restrict__ ids, int L, int64_t row_stride, int64_t pad,
                             int64_t *__restrict__ out) {
  __shared__ int sh_kept[THREADS / kWarp], sh_first[THREADS / kWarp];
  __shared__ int kept_all, first_all;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int64_t *row = ids + static_cast<int64_t>(b) * row_stride;
  int kept = 0, first = L;  // first = index of the first non-pad token = number of leading pads
  for (int c = tid; c < L; c += THREADS) {
    if (row[c] != pad) {
      ++kept;
      first = min(first, c);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    kept += __shfl_xor_sync(0xffffffffu, kept, o);
    first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
  }
  if (lane == 0) {
    sh_kept[wid] = kept;
    sh_first[wid] = first;
  }
  __syncthreads();
  if (tid == 0) {
    int k = 0, f = L;
    for (int w = 0; w < THREADS / kWarp; ++w) {
      k += sh_kept[w];
      f = min(f, sh_first[w]);
    }
    kept_all = k;
    first_all = f;
  }
  __syncthreads();
  // shift = L - kept - leading (>= 0): the pads that are not already leading; rows rotate right by it
  const int shift = L - kept_all - first_all;
  int64_t *dst = out + static_cast<int64_t>(b) * L;
  for (int c = tid; c < L; c += THREADS) {
    int src = c - shift;
    if (src < 0) src += L;
    dst[c] = row[src];
  }
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS)
    count_nonpad_kernel(const int64_t *__restrict__ ids, int L, int64_t row_stride, int64_t pad,
                        int32_t *__restrict__ counts) {
  __shared__ int sh[THREADS / kWarp];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int64_t *row = ids + static_cast<int64_t>(b) * row_stride;
  int kept = 0;
  for (int c = tid; c < L; c += THREADS) kept += (row[c] != pad) ? 1 : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) kept += __shfl_xor_sync(0xffffffffu, kept, o);
  if ((tid & 31) == 0) sh[tid >> 5] = kept;
  __syncthreads();
  if (tid == 0) {
    int k = 0;
    for (int w = 0; w < THREADS / kWarp; ++w) k += sh[w];
    counts[b] = k;
  }
}

// pad_sequence of per-sample tails (adjoint = 0):  out[b, k] = k < R_b ? src[b, W - R_b + k] : 0,  out (B, Rmax)
// its adjoint, the gradient scatter (adjoint = 1):  out[b, j] = j >= W - R_b ? src[b, j - (W - R_b)] : 0,  out (B, W)
template <typename U>
__global__ void __launch_bounds__(256)
    tail_rows_kernel(const U *__restrict__ src, int64_t src_stride, const int32_t *__restrict__ lens, int W, int Rmax,
                     U *__restrict__ out, int64_t out_stride, int adjoint) {
  const int b = blockIdx.y;
  const int c = blockIdx.x * 256 + threadIdx.x;
  const int R = lens[b];
  const int off = W - R;
  if (!adjoint) {
    if (c < Rmax) out[b * out_stride + c] = (c < R) ? src[b * src_stride + off + c] : U(0);
  } else {
    if (c < W) out[b * out_stride + c] = (c >= off) ? src[b * src_stride + (c - off)] : U(0);
  }
}

// Everything trainers/text_image_to_text/ppo.py:185-203 does after `generate`, one CTA per sample, nothing on the host:
//   moved[b]  = move_padding_left(sequences[b])              (:185, bit-exact rotation as above)
//   mask[b]   = moved[b] != pad                              (:186)
//   lens[b]   = max(nonpad(sequences[b]) - nonpad(prompt[b]), 0)   (:190-203: len(remove_pad(seq)[len(remove_pad(prompt)):]))
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
    rollout_layout_kernel(const int64_t *__restrict__ prompt, int P, int64_t prompt_stride, const int64_t *__restrict__ seq,
                          int L, int64_t seq_stride, int64_t pad, int64_t *__restrict__ moved, uint8_t *__restrict__ mask,
                          int32_t *__restrict__ lens) {
  __shared__ int sh[3][THREADS / kWarp];
  __shared__ int tot[3];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int64_t *row = seq + static_cast<int64_t>(b) * seq_stride;
  const int64_t *prow = prompt + static_cast<int64_t>(b) * prompt_stride;
  int kept = 0, first = L, pkept = 0;
  for (int c = tid; c < L; c += THREADS) {
    if (row[c] != pad) {
      ++kept;
      first = min(first, c);
    }
  }
  for (int c = tid; c < P; c += THREADS) pkept += (prow[c] != pad) ? 1 : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    kept += __shfl_xor_sync(0xffffffffu, kept, o);
    pkept += __shfl_xor_sync(0xffffffffu, pkept, o);
    first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
  }
  if (lane == 0) {
    sh[0][wid] = kept;
    sh[1][wid] = first;
    sh[2][wid] = pkept;
  }
  __syncthreads();
  if (tid == 0) {
    int k = 0, f = L, pk = 0;
    for (int w = 0; w < THREADS / kWarp; ++w) {
      k += sh[0][w];
      f = min(f, sh[1][w]);
      pk += sh[2][w];
    }
    tot[0] = k;
    tot[1] = f;
    tot[2] = pk;
    lens[b] = max(k - pk, 0);
  }
  __syncthreads();
  const int shift = L - tot[0] - tot[1];
  int64_t *dst = moved + static_cast<int64_t>(b) * L;
  uint8_t *mdst = mask + static_cast<int64_t>(b) * L;
  for (int c = tid; c < L; c += THREADS) {
    int src = c - shift;
    if (src < 0) src += L;
    const int64_t v = row[src];
    dst[c] = v;
    mdst[c] = (v != pad) ? 1 : 0;
  }
}

// The row plan of per-sample response tails (the table ops.RowPlan holds), built from DEVICE response lengths so that
// they never visit the host (trainers/text_image_to_text/ppo.py:229-239 slices per sample on the host):
//   sample b scores n_b = clamp(lens[b] - lab_shift, 0, width) rows starting at tile position first_b = seq - lens[b] +
//   row_shift of its (seq, V) tile, against labels  labels[b * lab_stride + (lab_tail_len > 0 ? lab_tail_len - lens[b] : 0)
//   + lab_shift + j];  results go to out[b * width + j].
// table: int64 [5][B + 1] = logit_off, label_off, out_off, cum (prefix row counts; cum[B] = total), tile_row.
// A length outside [0, min(seq + row_shift, lab_tail_len or inf)] sets AA_STATUS_SHORT_SEQUENCE and is clamped.
// copies > 1: the plan is repeated for `copies` logits tensors of identical shape that live copy_logit_delta elements
// apart (segment c * B + b reads tensor c, writes out[c * copy_out_delta + b * width + j]): actor and reference model are
// scored by ONE K1 launch in the rollout (no gradient: tile rows of the copies are not meaningful).
__global__ void __launch_bounds__(256)
    tail_plan_kernel(const int32_t *__restrict__ lens, int B, int seq, int64_t sb, int64_t sl, int64_t lab_stride,
                     int lab_tail_len, int lab_shift, int row_shift, int width, int copies, int64_t copy_logit_delta,
                     int64_t copy_out_delta, int64_t *__restrict__ table, int32_t *status) {
  __shared__ int64_t carry;
  __shared__ int64_t warp_tot[8];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int S = B * copies;
  int64_t *logit_off = table, *label_off = table + (S + 1), *out_off = table + 2 * (S + 1), *cum = table + 3 * (S + 1),
          *tile_row = table + 4 * (S + 1);
  if (tid == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < S; base += 256) {
    const int seg = base + tid;
    const int b = seg % B, c = seg / B;
    int64_t n = 0;
    if (seg < S) {
      int r = lens[b];
      int hi = seq + row_shift;  // first_b = seq - r + row_shift >= 0
      if (lab_tail_len > 0) hi = min(hi, lab_tail_len);
      if (r < 0 || r > hi) {
        if (status) atomicOr(status, AA_STATUS_SHORT_SEQUENCE);
        r = max(0, min(r, hi));
      }
      const int first = seq - r + row_shift;
      n = max(min(r - lab_shift, width), 0);
      logit_off[seg] = static_cast<int64_t>(b) * sb + static_cast<int64_t>(first) * sl + c * copy_logit_delta;
      label_off[seg] = static_cast<int64_t>(b) * lab_stride + (lab_tail_len > 0 ? lab_tail_len - r : 0) + lab_shift;
      out_off[seg] = static_cast<int64_t>(b) * width + c * copy_out_delta;
      tile_row[seg] = (static_cast<int64_t>(c) * B + b) * seq + first;
    }
    // block-wide exclusive scan of n
    int64_t x = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_tot[wid] = x;
    __syncthreads();
    int64_t before = carry;
    for (int w = 0; w < wid; ++w) before += warp_tot[w];
    if (seg < S) cum[seg] = before + x - n;
    __syncthreads();
    if (tid == 255) carry = before + x;
    __syncthreads();
  }
  if (tid == 0) {
    cum[S] = carry;
    logit_off[S] = label_off[S] = out_off[S] = tile_row[S] = 0;
  }
}

// Stream compaction of the causal-LM cross-entropy rows in ONE block (B * L is a few ten thousand positions: a handful of
// tiles): thread i of a tile owns ITEMS consecutive positions, a block-wide exclusive scan of the per-thread counts gives
// each valid row its output slot, so rows come out in ascending order whatever the thread timing.
template <int THREADS, int ITEMS>
__global__ void __launch_bounds__(THREADS)
    ce_rows_kernel(const int64_t *__restrict__ labels, int B, int L, int64_t sb, int64_t sl, int64_t ignore_index, int V,
                   int64_t *__restrict__ row_index, int64_t *__restrict__ labels_out, int64_t *__restrict__ count,
                   int32_t *status) {
  constexpr int WARPS = THREADS / kWarp;
  static_assert(WARPS <= kWarp, "one warp scans the warp totals");
  __shared__ int warp_tot[WARPS];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int64_t n = static_cast<int64_t>(B) * L;
  int64_t carry = 0;
  bool oob = false;
  for (int64_t base = 0; base < n; base += static_cast<int64_t>(THREADS) * ITEMS) {
    const int64_t p0 = base + static_cast<int64_t>(tid) * ITEMS;
    int64_t lab[ITEMS];
    int c = 0;
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
      const int64_t p = p0 + i;
      lab[i] = ignore_index;
      if (p < n) {
        const int64_t b = p / L;
        const int t = static_cast<int>(p - b * L);
        if (t + 1 < L) lab[i] = labels[b * sb + static_cast<int64_t>(t + 1) * sl];  // shifted: row t predicts token t + 1
      }
      if (lab[i] != ignore_index) {
        ++c;
        oob |= (lab[i] < 0 || lab[i] >= V);
      }
    }
    int x = c;  // inclusive scan inside the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_tot[wid] = x;
    __syncthreads();
    if (wid == 0) {  // inclusive scan of the warp totals
      int w = lane < WARPS ? warp_tot[lane] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += y;
      }
      if (lane < WARPS) warp_tot[lane] = w;
    }
    __syncthreads();
    int64_t slot = carry + (wid > 0 ? warp_tot[wid - 1] : 0) + (x - c);
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
      if (lab[i] != ignore_index) {
        row_index[slot] = p0 + i;
        labels_out[slot] = lab[i];
        ++slot;
      }
    }
    carry += warp_tot[WARPS - 1];
    __syncthreads();  // every thread has read warp_tot before the next tile overwrites it
  }
  if (oob && status) atomicOr(status, AA_STATUS_LABEL_OOB);
  if (tid == 0) *count = carry;
}

}  // namespace aa

using namespace aa;

extern "C" int aa_ppo_rollout_layout(const int64_t *prompt_ids, int32_t P, int64_t prompt_row_stride,
                                     const int64_t *sequences, int32_t L, int64_t seq_row_stride, int32_t B, int64_t pad_id,
                                     int64_t *moved, uint8_t *attention_mask, int32_t *response_lens, void *stream) {
  AA_REQUIRE(B >= 0 && L > 0 && P > 0, AA_ERR_ARG, "aa_ppo_rollout_layout: bad sizes");
  if (B == 0) return AA_OK;
  AA_REQUIRE(prompt_ids && sequences && moved && attention_mask && response_lens && sequences != moved, AA_ERR_ARG,
             "aa_ppo_rollout_layout: null or aliased pointers");
  rollout_layout_kernel<256><<<B, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      prompt_ids, P, prompt_row_stride, sequences, L, seq_row_stride, pad_id, moved, attention_mask, response_lens);
  return check_launch("aa_ppo_rollout_layout");
}

extern "C" int aa_tail_plan_build(const int32_t *response_lens, int32_t B, int32_t seq, int64_t sample_stride,
                                  int64_t row_stride, int64_t label_row_stride, int32_t label_tail_len, int32_t label_shift,
                                  int32_t row_shift, int32_t width, int32_t copies, int64_t copy_logit_delta,
                                  int64_t copy_out_delta, int64_t *table, int32_t *status, void *stream) {
  AA_REQUIRE(B > 0 && seq > 0 && width > 0 && copies >= 1, AA_ERR_ARG, "aa_tail_plan_build: bad sizes");
  AA_REQUIRE(response_lens && table, AA_ERR_ARG, "aa_tail_plan_build: null pointer");
  tail_plan_kernel<<<1, 256, 0, static_cast<cudaStream_t>(stream)>>>(response_lens, B, seq, sample_stride, row_stride,
                                                                     label_row_stride, label_tail_len, label_shift, row_shift,
                                                                     width, copies, copy_logit_delta, copy_out_delta, table,
                                                                     status);
  return check_launch("aa_tail_plan_build");
}

extern "C" int aa_tail_rows(const void *src, int dtype, int64_t src_row_stride, const int32_t *lens, int32_t B,
                            int32_t W, int32_t Rmax, void *out, int64_t out_row_stride, int32_t adjoint,
                            void *stream) {
  AA_REQUIRE(B >= 0 && W > 0 && Rmax > 0 && Rmax <= W, AA_ERR_ARG, "aa_tail_rows: bad sizes (W=%d Rmax=%d)", W, Rmax);
  if (B == 0) return AA_OK;
  AA_REQUIRE(src && lens && out && src != out, AA_ERR_ARG, "aa_tail_rows: null or aliased pointers");
  AA_REQUIRE(dtype == AA_BF16 || dtype == AA_F16 || dtype == AA_F32, AA_ERR_DTYPE, "aa_tail_rows: bad dtype");
  const int width = adjoint ? W : Rmax;
  const dim3 grid((width + 255) / 256, B);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == AA_F32)
    tail_rows_kernel<uint32_t><<<grid, 256, 0, st>>>(reinterpret_cast<const uint32_t *>(src), src_row_stride, lens, W, Rmax,
                                                     reinterpret_cast<uint32_t *>(out), out_row_stride, adjoint);
  else
    tail_rows_kernel<uint16_t><<<grid, 256, 0, st>>>(reinterpret_cast<const uint16_t *>(src), src_row_stride, lens, W, Rmax,
                                                     reinterpret_cast<uint16_t *>(out), out_row_stride, adjoint);
  return check_launch("aa_tail_rows");
}

extern "C" int aa_move_padding_left(const int64_t *ids, int32_t B, int32_t L, int64_t row_stride,
                                    int64_t pad_id, int64_t *out, void *stream) {
  AA_REQUIRE(B >= 0 && L > 0, AA_ERR_ARG, "aa_move_padding_left: bad sizes");
  if (B == 0) return AA_OK;
  AA_REQUIRE(ids && out && ids != out, AA_ERR_ARG, "aa_move_padding_left: null or aliased pointers");
  move_padding_left_kernel<256><<<B, 256, 0, static_cast<cudaStream_t>(stream)>>>(ids, L, row_stride, pad_id, out);
  return check_launch("aa_move_padding_left");
}

extern "C" int aa_count_nonpad(const int64_t *ids, int32_t B, int32_t L, int64_t row_stride, int64_t pad_id,
                               int32_t *counts, void *stream) {
  AA_REQUIRE(B >= 0 && L > 0, AA_ERR_ARG, "aa_count_nonpad: bad sizes");
  if (B == 0) return AA_OK;
  AA_REQUIRE(ids && counts, AA_ERR_ARG, "aa_count_nonpad: null pointer");
  count_nonpad_kernel<256><<<B, 256, 0, static_cast<cudaStream_t>(stream)>>>(ids, L, row_stride, pad_id, counts);
  return check_launch("aa_count_nonpad");
}

extern "C" int aa_ce_rows(const int64_t *labels, int32_t B, int32_t L, int64_t label_batch_stride, int64_t label_row_stride,
                          int64_t ignore_index, int32_t V, int64_t *row_index_out, int64_t *labels_out, int64_t *count_out,
                          int32_t *status, void *stream) {
  AA_REQUIRE(B > 0 && L > 0 && V > 0, AA_ERR_ARG, "aa_ce_rows: bad sizes (B=%d L=%d V=%d)", B, L, V);
  AA_REQUIRE(labels && row_index_out && labels_out && count_out, AA_ERR_ARG, "aa_ce_rows: null pointer");
  AA_REQUIRE(row_index_out != labels_out && labels != labels_out && labels != row_index_out, AA_ERR_ARG,
             "aa_ce_rows: aliased outputs");
  ce_rows_kernel<1024, 4><<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(
      labels, B, L, label_batch_stride, label_row_stride, ignore_index, V, row_index_out, labels_out, count_out, status);
  return check_launch("aa_ce_rows");
}

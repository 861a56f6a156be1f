// logprob.cu -- K1 / K1b: per-token log-prob (row log-softmax over V fused with the label
// gather) and its backward, for ragged row lists over non-contiguous logits views.
//
// Replaces utils/tools.py:402-413 (gather_log_probabilities) + autograd of F.log_softmax /
// torch.gather, and the per-sample slicing loops around them (trainers/text_to_text/dpo.py:133-142,
// trainers/text_image_to_text/ppo.py:229-239).  The (rows, V) log-prob tile is never written.
//
// HBM-bound streaming reduction: one CTA owns one row at a time (persistent, grid-strided);
// 128-bit streaming loads over the 16-byte-aligned body of the row, scalar peel for the
// (<8 element) head / tail when the row start is only 2-byte aligned (odd V such as 128257);
// per-thread online softmax in the exp2 domain, warp-shuffle + shared-memory merge of the
// (max, sum) partials.
#include <atomic>

#include "common.cuh"
#include "logprob_math.cuh"

namespace aa {

struct FwdParams {
  const void *logits;
  int64_t row_stride;
  int V;
  const int64_t *labels;
  int64_t ignore_index;  // rows whose label equals this are skipped (out = 0) when use_ignore != 0
  int use_ignore;
  RowMap map;
  int64_t n_rows;
  void *out;
  int out_dtype;
  float *stat_max;
  float *stat_logsum;
  int32_t *status;
  float log2e;  // = kLog2e, passed at run time so that ptxas keeps the packed FMUL2 (no immediate form)
};

struct BwdParams {
  const void *logits;
  int64_t row_stride;
  int V;
  const int64_t *labels;
  int64_t ignore_index;
  int use_ignore;
  RowMap map;
  int64_t n_rows;
  const int64_t *seg_tile_row;
  const float *stat_max;
  const float *stat_logsum;
  const void *grad_rows;
  int grad_rows_dtype;
  const float *grad_seg;
  const void *grad_scale;  // optional device scalar (dtype grad_scale_dtype): the upstream d loss of a fused loss node
  int grad_scale_dtype;
  void *grad_logits;
  int64_t grad_row_stride;
  int64_t n_tile_rows;
  float zero;  // +0.0f supplied at run time (see f2_round_bf16 in common.cuh)
  const int64_t *extra_zero_rows;  // n_tile_rows == 0 only: tile rows to zero-fill after the scored rows
  int64_t n_extra;
};
__host__ __device__ __forceinline__ int64_t bwd_work_rows(const BwdParams &p) {
  return p.n_tile_rows > 0 ? p.n_tile_rows : p.n_rows + p.n_extra;
}

// ---- K1 forward, variant 0: direct vectorised LDG ---------------------------------------
template <typename T, int THREADS, int UNROLL>
__global__ void __launch_bounds__(THREADS) logprob_fwd_kernel(const FwdParams p) {
  constexpr int E = Traits<T>::kVec;
  __shared__ float sh_m[32], sh_s[32];
  const int tid = threadIdx.x;
  const T *__restrict__ logits = reinterpret_cast<const T *>(p.logits);
  const int V = p.V;
  const f32x2 L2 = f2_splat(p.log2e);

  // p.n_rows is an upper bound when the plan was built on the device (aa_tail_plan_build: the response lengths never
  // visit the host); the table's last prefix entry is the exact count
  const int64_t n_rows = min(p.n_rows, __ldg(p.map.seg_cum + p.map.n_seg));
  for (int64_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
    const int seg = upper_segment(p.map.seg_cum, p.map.n_seg, row);
    const int64_t j = row - __ldg(p.map.seg_cum + seg);
    const T *x = logits + __ldg(p.map.seg_logit_off + seg) + j * p.row_stride;

    const int64_t y = __ldg(p.labels + __ldg(p.map.seg_label_off + seg) + j);  // same address in every thread
    if (p.use_ignore && y == p.ignore_index) {  // ignored position (cross-entropy ignore_index): no traffic
      if (tid == 0) {
        store_from_float(p.out, __ldg(p.map.seg_out_off + seg) + j, p.out_dtype, 0.f);
        if (p.stat_max) {
          p.stat_max[row] = 0.f;
          p.stat_logsum[row] = 0.f;
        }
      }
      continue;
    }
    float xy = 0.f;
    bool y_ok = true;
    if (tid == 0) {  // label column: one 2/4-byte load, issued before the streaming loop
      y_ok = (y >= 0) && (y < V);
      xy = y_ok ? Traits<T>::to_float(x[y]) : NAN;
    }

    const int mis = static_cast<int>((reinterpret_cast<uintptr_t>(x) & 15) / sizeof(T));
    const int head = mis ? min(E - mis, V) : 0;
    const int nvec = (V - head) / E;
    const int tail0 = head + nvec * E;
    const uint4 *body = reinterpret_cast<const uint4 *>(x + head);

    float m = -INFINITY, s = 0.f;
    if (tid < head) lse_push(m, s, Traits<T>::to_float(x[tid]));
    if (tid < V - tail0) lse_push(m, s, Traits<T>::to_float(x[tail0 + tid]));

    int k = tid;
    for (; k + (UNROLL - 1) * THREADS < nvec; k += UNROLL * THREADS) {
      uint4 v[UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) v[u] = ldg_stream(body + k + u * THREADS);
      fold_batch<T, UNROLL>(v, m, s, L2);
    }
    if (k < nvec) {  // last, partial batch: missing vectors are replaced by -inf (exp -> 0), one fold instead of
                     // up to UNROLL-1 single-vector folds (each of which pays its own max / rescale)
      uint4 v[UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u)
        v[u] = (k + u * THREADS < nvec) ? ldg_stream(body + k + u * THREADS) : bulk::neg_inf_vec<T>();
      fold_batch<T, UNROLL>(v, m, s, L2);
    }

    block_lse<THREADS>(m, s, sh_m, sh_s);
    if (tid == 0) {
      const float logsum = logf(s);
      float lp = (xy - m) - logsum;  // same association as ATen's `x - max - log(sum)`
      if (!y_ok) {
        lp = NAN;
        if (p.status) atomicOr(p.status, AA_STATUS_LABEL_OOB);
      }
      store_from_float(p.out, __ldg(p.map.seg_out_off + seg) + j, p.out_dtype, lp);
      if (p.stat_max) {
        p.stat_max[row] = m;
        p.stat_logsum[row] = logsum;
      }
    }
    __syncthreads();  // sh_m / sh_s reuse
  }
}

// ---- K1 forward, variant 1: TMA engine (cp.async.bulk, 1-D) staged through shared memory ------------
// One producer lane streams the 16-byte-aligned body of each row into a ring of shared-memory stages
// with cp.async.bulk (SASS: UBLKCP), completion signalled on mbarriers; eight consumer warps read
// the stages with conflict-free LDS.128 and run the same online softmax.  The ring runs across row
// boundaries, so the copy engine is already fetching the next row while the consumers reduce the
// current one.  Tensor maps are not needed (and could not describe V = 128257 anyway: a TMA tensor map
// wants 16-byte row strides); the 1-D bulk copy only needs the 16-byte-aligned body that the head /
// tail peel already isolates.

template <typename T, int CONSUMERS, int STAGES, int UNROLL>
__global__ void __launch_bounds__(CONSUMERS + 32) logprob_fwd_bulk_kernel(const FwdParams p) {
  constexpr int E = Traits<T>::kVec;
  constexpr int STAGE_VECS = CONSUMERS * UNROLL;
  extern __shared__ __align__(128) uint8_t smem_raw[];
  uint4 *ring = reinterpret_cast<uint4 *>(smem_raw);
  uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + static_cast<size_t>(STAGES) * STAGE_VECS * 16);
  uint64_t *empty = full + STAGES;
  __shared__ float sh_m[32], sh_s[32];
  const int tid = threadIdx.x;
  const T *__restrict__ logits = reinterpret_cast<const T *>(p.logits);
  const int V = p.V;
  const f32x2 L2 = f2_splat(p.log2e);
  if (tid == 0) {
    for (int i = 0; i < STAGES; ++i) {
      bulk::mbar_init(full + i, 1);
      bulk::mbar_init(empty + i, CONSUMERS / kWarp);
    }
    bulk::fence_barrier_init();
  }
  __syncthreads();
  int stage = 0;
  uint32_t phase = 0;
  const int64_t n_rows = min(p.n_rows, __ldg(p.map.seg_cum + p.map.n_seg));  // device-built plans: see the LDG kernel

  if (tid >= CONSUMERS) {
    // ---------------- producer warp: one elected lane drives the copy engine ----------------
    if (tid == CONSUMERS) {
      for (int64_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
        const int seg = upper_segment(p.map.seg_cum, p.map.n_seg, row);
        const int64_t j = row - __ldg(p.map.seg_cum + seg);
        const T *x = logits + __ldg(p.map.seg_logit_off + seg) + j * p.row_stride;
        if (p.use_ignore && __ldg(p.labels + __ldg(p.map.seg_label_off + seg) + j) == p.ignore_index) continue;
        const int mis = static_cast<int>((reinterpret_cast<uintptr_t>(x) & 15) / sizeof(T));
        const int head = mis ? min(E - mis, V) : 0;
        const int nvec = (V - head) / E;
        const uint4 *body = reinterpret_cast<const uint4 *>(x + head);
        for (int v0 = 0; v0 < nvec; v0 += STAGE_VECS) {
          const int n = min(STAGE_VECS, nvec - v0);
          bulk::mbar_wait(empty + stage, phase ^ 1u);
          bulk::mbar_expect_tx(full + stage, static_cast<uint32_t>(n) * 16u);
          bulk::bulk_g2s(ring + static_cast<size_t>(stage) * STAGE_VECS, body + v0, static_cast<uint32_t>(n) * 16u,
                         full + stage);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
    return;
  }

  // ---------------- consumer warps ----------------
  for (int64_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
    const int seg = upper_segment(p.map.seg_cum, p.map.n_seg, row);
    const int64_t j = row - __ldg(p.map.seg_cum + seg);
    const T *x = logits + __ldg(p.map.seg_logit_off + seg) + j * p.row_stride;
    const int64_t y = __ldg(p.labels + __ldg(p.map.seg_label_off + seg) + j);
    if (p.use_ignore && y == p.ignore_index) {
      if (tid == 0) {
        store_from_float(p.out, __ldg(p.map.seg_out_off + seg) + j, p.out_dtype, 0.f);
        if (p.stat_max) {
          p.stat_max[row] = 0.f;
          p.stat_logsum[row] = 0.f;
        }
      }
      continue;
    }
    float xy = 0.f;
    bool y_ok = true;
    if (tid == 0) {
      y_ok = (y >= 0) && (y < V);
      xy = y_ok ? Traits<T>::to_float(x[y]) : NAN;
    }
    const int mis = static_cast<int>((reinterpret_cast<uintptr_t>(x) & 15) / sizeof(T));
    const int head = mis ? min(E - mis, V) : 0;
    const int nvec = (V - head) / E;
    const int tail0 = head + nvec * E;
    float m = -INFINITY, s = 0.f;
    if (tid < head) lse_push(m, s, Traits<T>::to_float(x[tid]));
    if (tid < V - tail0) lse_push(m, s, Traits<T>::to_float(x[tail0 + tid]));

    for (int v0 = 0; v0 < nvec; v0 += STAGE_VECS) {
      const int n = min(STAGE_VECS, nvec - v0);
      bulk::mbar_wait(full + stage, phase);
      const uint4 *buf = ring + static_cast<size_t>(stage) * STAGE_VECS;
      uint4 v[UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        const int k = tid + u * CONSUMERS;
        v[u] = (k < n) ? buf[k] : bulk::neg_inf_vec<T>();
      }
      // order this warp's generic-proxy reads of the stage before the copy engine's next write to it
      // (compute-sanitizer racecheck reports the WAR pair without the proxy fence)
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if ((tid & 31) == 0) bulk::mbar_arrive(empty + stage);  // this warp's reads of the stage are done
      fold_batch<T, UNROLL>(v, m, s, L2);
      if (++stage == STAGES) {
        stage = 0;
        phase ^= 1u;
      }
    }

    // merge the partials of the CONSUMERS threads (named barrier 1: the producer warp is not part of it)
    {
      constexpr int NW = CONSUMERS / kWarp;
      const int lane = tid & 31, wid = tid >> 5;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        float m2 = __shfl_xor_sync(0xffffffffu, m, o);
        float s2 = __shfl_xor_sync(0xffffffffu, s, o);
        lse_merge(m, s, m2, s2);
      }
      if (lane == 0) {
        sh_m[wid] = m;
        sh_s[wid] = s;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(CONSUMERS) : "memory");
      if (wid == 0) {
        m = lane < NW ? sh_m[lane] : -INFINITY;
        s = lane < NW ? sh_s[lane] : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          float m2 = __shfl_xor_sync(0xffffffffu, m, o);
          float s2 = __shfl_xor_sync(0xffffffffu, s, o);
          lse_merge(m, s, m2, s2);
        }
      }
    }
    if (tid == 0) {
      const float logsum = logf(s);
      float lp = (xy - m) - logsum;
      if (!y_ok) {
        lp = NAN;
        if (p.status) atomicOr(p.status, AA_STATUS_LABEL_OOB);
      }
      store_from_float(p.out, __ldg(p.map.seg_out_off + seg) + j, p.out_dtype, lp);
      if (p.stat_max) {
        p.stat_max[row] = m;
        p.stat_logsum[row] = logsum;
      }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(CONSUMERS) : "memory");  // sh_m / sh_s reuse
  }
}

// ---- K1b backward -------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void zero_row(T *g, int V) {
  constexpr int E = Traits<T>::kVec;
  const int mis = static_cast<int>((reinterpret_cast<uintptr_t>(g) & 15) / sizeof(T));
  const int head = mis ? min(E - mis, V) : 0;
  const int nvec = (V - head) / E;
  const int tail0 = head + nvec * E;
  const int tid = threadIdx.x;
  if (tid < head) g[tid] = Traits<T>::from_float(0.f);
  if (tid < V - tail0) g[tail0 + tid] = Traits<T>::from_float(0.f);
  uint4 *body = reinterpret_cast<uint4 *>(g + head);
  const uint4 z = make_uint4(0, 0, 0, 0);
  for (int k = tid; k < nvec; k += blockDim.x) stg_stream(body + k, z);
}

template <typename T, int THREADS, int UNROLL, bool FAITHFUL>
__global__ void __launch_bounds__(THREADS) logprob_bwd_kernel(const BwdParams p) {
  constexpr int E = Traits<T>::kVec;
  const int tid = threadIdx.x;
  const int V = p.V;
  const T *__restrict__ logits = reinterpret_cast<const T *>(p.logits);
  T *__restrict__ grad = reinterpret_cast<T *>(p.grad_logits);
  const bool tile_mode = p.n_tile_rows > 0;
  const int64_t n_work = bwd_work_rows(p);

  for (int64_t work = blockIdx.x; work < n_work; work += gridDim.x) {
    int seg;
    int64_t j;
    T *g_out;
    if (!tile_mode && work >= p.n_rows) {  // listed zero rows
      zero_row<T>(grad + __ldg(p.extra_zero_rows + (work - p.n_rows)) * p.grad_row_stride, V);
      continue;
    }
    if (tile_mode) {
      g_out = grad + work * p.grad_row_stride;
      bool scored = false;
      seg = 0;
      j = 0;
      if (p.map.n_seg > 0 && work >= __ldg(p.seg_tile_row)) {
        seg = upper_segment(p.seg_tile_row, p.map.n_seg, work);
        j = work - __ldg(p.seg_tile_row + seg);
        scored = j < (__ldg(p.map.seg_cum + seg + 1) - __ldg(p.map.seg_cum + seg));
      }
      if (!scored) {
        zero_row<T>(g_out, V);
        continue;
      }
    } else {
      seg = upper_segment(p.map.seg_cum, p.map.n_seg, work);
      j = work - __ldg(p.map.seg_cum + seg);
      g_out = grad + (__ldg(p.seg_tile_row + seg) + j) * p.grad_row_stride;
    }
    const int64_t flat = __ldg(p.map.seg_cum + seg) + j;
    const T *x = logits + __ldg(p.map.seg_logit_off + seg) + j * p.row_stride;

    float g = 1.f;
    if (p.grad_rows) g *= load_as_float(p.grad_rows, __ldg(p.map.seg_out_off + seg) + j, p.grad_rows_dtype);
    if (p.grad_seg) g *= __ldg(p.grad_seg + seg);
    if (p.grad_scale) g *= load_as_float(p.grad_scale, 0, p.grad_scale_dtype);
    if (p.use_ignore && __ldg(p.labels + __ldg(p.map.seg_label_off + seg) + j) == p.ignore_index) g = 0.f;
    if (g == 0.f) {  // masked / prompt / ignored rows: 0 * softmax, no need to read the row
      zero_row<T>(g_out, V);
      continue;
    }
    const float m = __ldg(p.stat_max + flat);
    const float logsum = __ldg(p.stat_logsum + flat);
    const float lse = m + logsum;
    const float c_f32 = -lse * kLog2e;
    // F32 mode: p_j = 2^(x_j*log2e + c_f32) * 2^(residual of the rounded offset), folded into -g
    const float neg_g = FAITHFUL ? -g : -g * ex2_approx(fmaf(-lse, kLog2e, -c_f32));
    const GradConsts gk = make_grad_consts(m, logsum, c_f32, neg_g, p.zero);

    const bool same_phase =
        ((reinterpret_cast<uintptr_t>(x) ^ reinterpret_cast<uintptr_t>(g_out)) & 15) == 0;
    if (same_phase) {
      const int mis = static_cast<int>((reinterpret_cast<uintptr_t>(x) & 15) / sizeof(T));
      const int head = mis ? min(E - mis, V) : 0;
      const int nvec = (V - head) / E;
      const int tail0 = head + nvec * E;
      if (tid < head)
        g_out[tid] = Traits<T>::from_float(
            neg_g * prob_of<T, FAITHFUL>(Traits<T>::to_float(x[tid]), m, logsum, c_f32));
      if (tid < V - tail0)
        g_out[tail0 + tid] = Traits<T>::from_float(
            neg_g * prob_of<T, FAITHFUL>(Traits<T>::to_float(x[tail0 + tid]), m, logsum, c_f32));
      const uint4 *src = reinterpret_cast<const uint4 *>(x + head);
      uint4 *dst = reinterpret_cast<uint4 *>(g_out + head);
      int k = tid;
      for (; k + (UNROLL - 1) * THREADS < nvec; k += UNROLL * THREADS) {
        uint4 v[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) v[u] = ldg_stream(src + k + u * THREADS);
#pragma unroll
        for (int u = 0; u < UNROLL; ++u)
          stg_stream(dst + k + u * THREADS, vec_grad<T, FAITHFUL>(v[u], gk));
      }
      for (; k < nvec; k += THREADS)
        stg_stream(dst + k, vec_grad<T, FAITHFUL>(ldg_stream(src + k), gk));
    } else {
      // logits view and gradient tile disagree on the 16-byte phase of this row: element loop
      for (int c = tid; c < V; c += THREADS)
        g_out[c] = Traits<T>::from_float(
            neg_g * prob_of<T, FAITHFUL>(Traits<T>::to_float(x[c]), m, logsum, c_f32));
    }
    // the label column: grad = g - p_y * g (ATen: grad_out - exp(out) * sum(grad_out))
    __syncthreads();
    if (tid == 0) {
      const int64_t y = __ldg(p.labels + __ldg(p.map.seg_label_off + seg) + j);
      if (y >= 0 && y < V) {
        const float py = prob_of<T, FAITHFUL>(Traits<T>::to_float(x[y]), m, logsum, c_f32);
        g_out[y] = Traits<T>::from_float(FAITHFUL ? __fsub_rn(g, __fmul_rn(py, g)) : fmaf(py, neg_g, g));
      }
    }
  }
}

// ---- K1b, chunked (experiment, selected with tuning kernel digit 2): the gradient tile is swept in
// address order.  MEASURED SLOWER on B200 than the one-CTA-per-row kernel above (4.4-5.4 TB/s vs
// 5.7-6.0 TB/s at V = 128257, tools/sweep_k1.py) -- kept for study, not the default.
// The backward needs no per-row reduction (max / logsum come from the forward), so a row does not
// have to be owned by one CTA.  Work unit = (row, chunk of THREADS*UNROLL 16-byte vectors);
// consecutive CTAs take consecutive units, so at any moment the whole grid reads and writes one
// compact window of the tile that moves through memory in address order (what a plain copy does),
// instead of gridDim different rows 256 KB apart.  A tiny prep kernel resolves each row once
// (segment search, label, saved stats, upstream gradient) into a 32-byte record.
struct __align__(16) RowRec {
  int64_t x_off;   // element offset of the logits row
  int64_t g_row;   // row index in the gradient tile
  float m, logsum, g;
  int32_t y;       // label column; -1: out of range (no one-hot term); -2: zero-fill the row
};

__global__ void bwd_row_prep_kernel(const BwdParams p, RowRec *__restrict__ rec) {
  const bool tile_mode = p.n_tile_rows > 0;
  const int64_t n_work = bwd_work_rows(p);
  const int64_t work = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (work >= n_work) return;
  RowRec r;
  r.x_off = 0; r.g_row = work; r.m = 0.f; r.logsum = 0.f; r.g = 0.f; r.y = -2;
  int seg = 0;
  int64_t j = 0;
  bool scored;
  int64_t slot = work;  // where the record goes in the work list
  if (!tile_mode && work >= p.n_rows) {  // listed zero rows come after the scored rows: balanced static stride
    r.g_row = __ldg(p.extra_zero_rows + (work - p.n_rows));
    scored = false;
  } else if (tile_mode) {
    // every tile row is work (the row layout is only known on the device).  The work list is ORDERED: the scored rows
    // first, in flat row order, then the zero rows -- the persistent kernel's static stride then sees equally expensive
    // rows next to each other (rows in tile order gave +-40% scored rows per CTA in the PPO shape)
    scored = false;
    int64_t scored_before = 0;
    if (p.map.n_seg > 0 && work >= __ldg(p.seg_tile_row)) {
      seg = upper_segment(p.seg_tile_row, p.map.n_seg, work);
      j = work - __ldg(p.seg_tile_row + seg);
      const int64_t first = __ldg(p.map.seg_cum + seg), cnt = __ldg(p.map.seg_cum + seg + 1) - first;
      scored = j < cnt;
      scored_before = first + min(j, cnt);
    }
    const int64_t total_scored = __ldg(p.map.seg_cum + p.map.n_seg);
    slot = scored ? scored_before : total_scored + (work - scored_before);
  } else {
    seg = upper_segment(p.map.seg_cum, p.map.n_seg, work);
    j = work - __ldg(p.map.seg_cum + seg);
    r.g_row = __ldg(p.seg_tile_row + seg) + j;
    scored = true;
  }
  if (scored) {
    const int64_t flat = __ldg(p.map.seg_cum + seg) + j;
    float g = 1.f;
    if (p.grad_rows) g *= load_as_float(p.grad_rows, __ldg(p.map.seg_out_off + seg) + j, p.grad_rows_dtype);
    if (p.grad_seg) g *= __ldg(p.grad_seg + seg);
    if (p.grad_scale) g *= load_as_float(p.grad_scale, 0, p.grad_scale_dtype);
    const int64_t y = __ldg(p.labels + __ldg(p.map.seg_label_off + seg) + j);
    if (p.use_ignore && y == p.ignore_index) g = 0.f;
    if (g != 0.f) {  // g == 0 (masked / prompt / ignored rows): plain zero row
      r.x_off = __ldg(p.map.seg_logit_off + seg) + j * p.row_stride;
      r.m = __ldg(p.stat_max + flat);
      r.logsum = __ldg(p.stat_logsum + flat);
      r.g = g;
      r.y = (y >= 0 && y < p.V) ? static_cast<int32_t>(y) : -1;
    }
  }
  rec[slot] = r;
}

template <typename T, int THREADS, int UNROLL, bool FAITHFUL>
__global__ void __launch_bounds__(THREADS)
    logprob_bwd_chunk_kernel(const T *__restrict__ logits, T *__restrict__ grad, int64_t grad_row_stride, int V,
                             const RowRec *__restrict__ rec, int64_t n_work, int upr, float zero) {
  constexpr int E = Traits<T>::kVec;
  constexpr int CH = THREADS * UNROLL;
  const int tid = threadIdx.x;
  const int64_t n_units = n_work * upr;
  for (int64_t u = blockIdx.x; u < n_units; u += gridDim.x) {
    const int64_t r = u / upr;
    const int c = static_cast<int>(u - r * upr);
    const int4 r0 = __ldg(reinterpret_cast<const int4 *>(rec + r));
    const int4 r1 = __ldg(reinterpret_cast<const int4 *>(rec + r) + 1);
    const int64_t x_off = (static_cast<int64_t>(static_cast<uint32_t>(r0.y)) << 32) | static_cast<uint32_t>(r0.x);
    const int64_t g_row = (static_cast<int64_t>(static_cast<uint32_t>(r0.w)) << 32) | static_cast<uint32_t>(r0.z);
    const float m = __int_as_float(r1.x), logsum = __int_as_float(r1.y), g = __int_as_float(r1.z);
    const int y = r1.w;
    T *g_out = grad + g_row * grad_row_stride;
    const int mis = static_cast<int>((reinterpret_cast<uintptr_t>(g_out) & 15) / sizeof(T));
    // vector v of the row's 16-byte-aligned span covers elements [v*E - mis, v*E - mis + E)
    uint4 *gspan = reinterpret_cast<uint4 *>(g_out - mis);
    const int v0 = c * CH + tid;
    if (y == -2) {
#pragma unroll
      for (int q = 0; q < UNROLL; ++q) {
        const int v = v0 + q * THREADS;
        const int e0 = v * E - mis;
        if (e0 >= 0 && e0 + E <= V) {
          stg_stream(gspan + v, make_uint4(0, 0, 0, 0));
        } else {
          for (int e = max(e0, 0); e < min(e0 + E, V); ++e) g_out[e] = Traits<T>::from_float(0.f);
        }
      }
      continue;
    }
    const T *x = logits + x_off;
    const float lse = m + logsum;
    const float c_f32 = -lse * kLog2e;
    const float neg_g = FAITHFUL ? -g : -g * ex2_approx(fmaf(-lse, kLog2e, -c_f32));
    const GradConsts gk = make_grad_consts(m, logsum, c_f32, neg_g, zero);
    const bool same_phase = ((reinterpret_cast<uintptr_t>(x) ^ reinterpret_cast<uintptr_t>(g_out)) & 15) == 0;
    if (same_phase) {
      const uint4 *xspan = reinterpret_cast<const uint4 *>(x - mis);
      const int yv = (y >= 0) ? (y + mis) / E : -1;
      uint4 val[UNROLL];
#pragma unroll
      for (int q = 0; q < UNROLL; ++q) {
        const int v = v0 + q * THREADS;
        const int e0 = v * E - mis;
        if (e0 >= 0 && e0 + E <= V) val[q] = ldg_stream(xspan + v);
      }
#pragma unroll
      for (int q = 0; q < UNROLL; ++q) {
        const int v = v0 + q * THREADS;
        const int e0 = v * E - mis;
        if (e0 >= 0 && e0 + E <= V) {
          uint4 o = vec_grad<T, FAITHFUL>(val[q], gk);
          if (v == yv) patch_label<T, FAITHFUL>(o, val[q], y - e0, m, logsum, c_f32, neg_g, g);
          stg_stream(gspan + v, o);
        } else {  // row head / tail: the vector sticks out of the row
          for (int e = max(e0, 0); e < min(e0 + E, V); ++e)
            g_out[e] = Traits<T>::from_float(
                grad_of<T, FAITHFUL>(Traits<T>::to_float(x[e]), m, logsum, c_f32, neg_g, g, e == y));
        }
      }
    } else {
      // logits view and gradient tile disagree on the 16-byte phase of this row: element loop
      const int e_lo = max(c * CH * E - mis, 0);
      const int e_hi = min((c + 1) * CH * E - mis, V);
      for (int e = e_lo + tid; e < e_hi; e += THREADS)
        g_out[e] = Traits<T>::from_float(
            grad_of<T, FAITHFUL>(Traits<T>::to_float(x[e]), m, logsum, c_f32, neg_g, g, e == y));
    }
  }
}

// ---- K1b, TMA-staged (default for 16-byte-phase-compatible tiles) ---------------------------------
// Micro-benchmark on B200 (tools/micro/copy_bw.cu, 8 GiB read + 8 GiB write): the same one-CTA-per-row
// access structure as the LDG kernel above tops out at 5.97-6.30 TB/s for a PURE copy, while the copy
// engine (cp.async.bulk global->smem, smem->global, 64 KB in flight per SM) reaches 6.59 TB/s =
// cudaMemcpy speed.  So the backward moves its data with the TMA engine in both directions and the SM
// only touches shared memory:
//   producer lane : RowRec -> cp.async.bulk loads of 16 KB chunks of the row's aligned body into a ring
//                   (full mbarriers, expect_tx), and -- lagging LAG chunks behind -- cp.async.bulk
//                   STORES of the chunks the consumers have finished (done mbarriers); zero rows are
//                   stored straight from a zeroed shared-memory buffer, no SM data path at all;
//   8 consumer warps: LDS.128 -> grad math (f32x2, Veltkamp rounding) -> STS.128 in place, one-hot label
//                   patched in registers, fence.proxy.async, arrive(done).
// Rows whose logits and gradient addresses disagree modulo 16 fall back to an element loop.
template <typename T, int CONSUMERS, int STAGES, int UNROLL, int LAG, bool FAITHFUL>
__global__ void __launch_bounds__(CONSUMERS + 32)
    logprob_bwd_tma_kernel(const T *__restrict__ logits, T *__restrict__ grad, int64_t grad_row_stride, int V,
                           const RowRec *__restrict__ rec, int64_t n_work, float zero) {
  constexpr int E = Traits<T>::kVec;
  constexpr int STAGE_VECS = CONSUMERS * UNROLL;
  static_assert(LAG >= 1 && LAG < STAGES, "LAG must leave at least one free stage");
  extern __shared__ __align__(128) uint8_t smem_raw[];
  uint4 *ring = reinterpret_cast<uint4 *>(smem_raw);
  uint4 *zero_buf = ring + static_cast<size_t>(STAGES) * STAGE_VECS;
  uint64_t *full = reinterpret_cast<uint64_t *>(zero_buf + STAGE_VECS);
  uint64_t *done = full + STAGES;
  uint64_t *st_dst = done + STAGES;                             // destination of the chunk held by each stage
  uint32_t *st_bytes = reinterpret_cast<uint32_t *>(st_dst + STAGES);
  const int tid = threadIdx.x;
  for (int i = tid; i < STAGE_VECS; i += CONSUMERS + 32) zero_buf[i] = make_uint4(0, 0, 0, 0);
  if (tid == 0) {
    for (int i = 0; i < STAGES; ++i) {
      bulk::mbar_init(full + i, 1);
      bulk::mbar_init(done + i, CONSUMERS / kWarp);
    }
    bulk::fence_barrier_init();
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // zero_buf is read by the async proxy
  __syncthreads();

  if (tid >= CONSUMERS) {
    // ------------------------------ producer lane ------------------------------
    if (tid != CONSUMERS) return;
    int64_t it = 0;       // chunks loaded so far
    int64_t retired = 0;  // chunks stored so far
    auto retire_one = [&]() {
      const int s = static_cast<int>(retired % STAGES);
      bulk::mbar_wait(done + s, static_cast<uint32_t>((retired / STAGES) & 1));
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(st_dst[s]),
                   "r"(bulk::smem_u32(ring + static_cast<size_t>(s) * STAGE_VECS)), "r"(st_bytes[s])
                   : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      ++retired;
    };
    for (int64_t r = blockIdx.x; r < n_work; r += gridDim.x) {
      const int4 r0 = __ldg(reinterpret_cast<const int4 *>(rec + r));
      const int4 r1 = __ldg(reinterpret_cast<const int4 *>(rec + r) + 1);
      const int64_t x_off = (static_cast<int64_t>(static_cast<uint32_t>(r0.y)) << 32) | static_cast<uint32_t>(r0.x);
      const int64_t g_row = (static_cast<int64_t>(static_cast<uint32_t>(r0.w)) << 32) | static_cast<uint32_t>(r0.z);
      const int y = r1.w;
      T *g_out = grad + g_row * grad_row_stride;
      const int mis = static_cast<int>((reinterpret_cast<uintptr_t>(g_out) & 15) / sizeof(T));
      const int head = mis ? min(E - mis, V) : 0;
      const int nvec = (V - head) / E;
      const int tail0 = head + nvec * E;
      uint4 *gbody = reinterpret_cast<uint4 *>(g_out + head);
      if (y == -2) {  // zero row: the copy engine writes it from the zero buffer
        for (int e = 0; e < head; ++e) g_out[e] = Traits<T>::from_float(0.f);
        for (int e = tail0; e < V; ++e) g_out[e] = Traits<T>::from_float(0.f);
        for (int v0 = 0; v0 < nvec; v0 += STAGE_VECS) {
          const uint32_t bytes = static_cast<uint32_t>(min(STAGE_VECS, nvec - v0)) * 16u;
          asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gbody + v0),
                       "r"(bulk::smem_u32(zero_buf)), "r"(bytes)
                       : "memory");
        }
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        continue;
      }
      const T *x = logits + x_off;
      if (((reinterpret_cast<uintptr_t>(x) ^ reinterpret_cast<uintptr_t>(g_out)) & 15) != 0) continue;  // consumers' element loop
      const uint4 *xbody = reinterpret_cast<const uint4 *>(x + head);
      for (int v0 = 0; v0 < nvec; v0 += STAGE_VECS) {
        const uint32_t bytes = static_cast<uint32_t>(min(STAGE_VECS, nvec - v0)) * 16u;
        while (it - retired >= LAG) retire_one();  // keep at most LAG chunks between load and store
        const int s = static_cast<int>(it % STAGES);
        // the stage's previous chunk (it - STAGES) was handed to the copy engine at least STAGES - LAG
        // stores ago: wait until the engine has finished READING it (later groups may stay pending)
        asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(STAGES - LAG) : "memory");
        st_dst[s] = reinterpret_cast<uint64_t>(gbody + v0);
        st_bytes[s] = bytes;
        bulk::mbar_expect_tx(full + s, bytes);
        bulk::bulk_g2s(ring + static_cast<size_t>(s) * STAGE_VECS, xbody + v0, bytes, full + s);
        ++it;
      }
    }
    while (retired < it) retire_one();
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // smem must outlive the engine's reads / the stores
    return;
  }

  // ------------------------------ consumer warps ------------------------------
  int64_t it = 0;
  for (int64_t r = blockIdx.x; r < n_work; r += gridDim.x) {
    const int4 r0 = __ldg(reinterpret_cast<const int4 *>(rec + r));
    const int4 r1 = __ldg(reinterpret_cast<const int4 *>(rec + r) + 1);
    const int y = r1.w;
    if (y == -2) continue;
    const int64_t x_off = (static_cast<int64_t>(static_cast<uint32_t>(r0.y)) << 32) | static_cast<uint32_t>(r0.x);
    const int64_t g_row = (static_cast<int64_t>(static_cast<uint32_t>(r0.w)) << 32) | static_cast<uint32_t>(r0.z);
    const float m = __int_as_float(r1.x), logsum = __int_as_float(r1.y), g = __int_as_float(r1.z);
    T *g_out = grad + g_row * grad_row_stride;
    const T *x = logits + x_off;
    const float lse = m + logsum;
    const float c_f32 = -lse * kLog2e;
    const float neg_g = FAITHFUL ? -g : -g * ex2_approx(fmaf(-lse, kLog2e, -c_f32));
    const GradConsts gk = make_grad_consts(m, logsum, c_f32, neg_g, zero);
    if (((reinterpret_cast<uintptr_t>(x) ^ reinterpret_cast<uintptr_t>(g_out)) & 15) != 0) {
      for (int e = tid; e < V; e += CONSUMERS)
        g_out[e] = Traits<T>::from_float(grad_of<T, FAITHFUL>(Traits<T>::to_float(x[e]), m, logsum, c_f32, neg_g, g, e == y));
      continue;
    }
    const int mis = static_cast<int>((reinterpret_cast<uintptr_t>(g_out) & 15) / sizeof(T));
    const int head = mis ? min(E - mis, V) : 0;
    const int nvec = (V - head) / E;
    const int tail0 = head + nvec * E;
    if (tid < head)
      g_out[tid] = Traits<T>::from_float(grad_of<T, FAITHFUL>(Traits<T>::to_float(x[tid]), m, logsum, c_f32, neg_g, g, tid == y));
    if (tid < V - tail0)
      g_out[tail0 + tid] = Traits<T>::from_float(
          grad_of<T, FAITHFUL>(Traits<T>::to_float(x[tail0 + tid]), m, logsum, c_f32, neg_g, g, tail0 + tid == y));
    const int yv = (y >= head && y < tail0) ? (y - head) / E : -1;  // body vector holding the label column
    for (int v0 = 0; v0 < nvec; v0 += STAGE_VECS) {
      const int n = min(STAGE_VECS, nvec - v0);
      const int s = static_cast<int>(it % STAGES);
      bulk::mbar_wait(full + s, static_cast<uint32_t>((it / STAGES) & 1));
      uint4 *buf = ring + static_cast<size_t>(s) * STAGE_VECS;
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        const int k = tid + u * CONSUMERS;
        if (k < n) {
          const uint4 in = buf[k];
          uint4 o = vec_grad<T, FAITHFUL>(in, gk);
          if (v0 + k == yv) patch_label<T, FAITHFUL>(o, in, (y - head) - (v0 + k) * E, m, logsum, c_f32, neg_g, g);
          buf[k] = o;
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the copy engine
      __syncwarp();
      if ((tid & 31) == 0) bulk::mbar_arrive(done + s);
      ++it;
    }
  }
}

// ---- host side ----------------------------------------------------------------------------
// Tuning knobs of the DIAGNOSTIC entry points aa_logprob_set_tuning{,_bwd}: process-wide by design (sweeps set them once,
// before a run; the trainers never touch them).  Atomics make a setter racing with launches on another thread well
// defined: such a launch may see the old or the new shape, both valid -- results never depend on the knobs.
static std::atomic<int> g_variant{0};        // forward (and backward unless overridden)
static std::atomic<int> g_ctas_per_sm{0};
static std::atomic<int> g_bwd_variant{-1};   // -1: follow the forward setting
static std::atomic<int> g_bwd_ctas_per_sm{0};
static inline int fwd_variant() { return g_variant.load(std::memory_order_relaxed); }
static inline int fwd_ctas() { return g_ctas_per_sm.load(std::memory_order_relaxed); }
static inline int bwd_variant() {
  const int v = g_bwd_variant.load(std::memory_order_relaxed);
  return v >= 0 ? v : fwd_variant();
}
static inline int bwd_ctas() {
  return g_bwd_variant.load(std::memory_order_relaxed) >= 0 ? g_bwd_ctas_per_sm.load(std::memory_order_relaxed) : fwd_ctas();
}

// tuning: g_variant = kernel variant (units digit) + 10 * shape code.  Forward shape codes (16-bit logits):
//   0: 128 thr x 8 vec, one CTA per row (default)   1: 256 x 8   2: 512 x 4   3: 128 x 8   4: 256 x 2   5: 512 x 2
//   7: the launch before this layout: 128 x 8, a persistent grid of 16 CTAs/SM (9 fit), static row stride -- kept to
//      A/B against the default in one process (bench.py --variant 70); the backward treats 7 as its default.
// A persistent grid (codes 1-5, f32 logits, and code 0 with ctas_per_sm > 0) holds ctas_per_sm CTAs per SM, clamped
// to the CTAs that are resident at once; 0 means all that fit.
constexpr int kFwdLegacyShape = 7;

template <typename T, int THREADS, int UNROLL>
static int launch_fwd_shape(const FwdParams &p, int per_sm, cudaStream_t st, bool fit_resident = true) {
  auto kern = logprob_fwd_kernel<T, THREADS, UNROLL>;
  int64_t grid;
  if (per_sm < 0) {
    grid = p.n_rows < 0x7fffffff ? p.n_rows : 0x7fffffff;  // one CTA per row (the kernel strides past a full grid)
  } else {
    if (fit_resident) {
      const int resident = resident_ctas(reinterpret_cast<const void *>(kern), THREADS, 0);
      if (per_sm == 0 || per_sm > resident) per_sm = resident;
    }
    grid = static_cast<int64_t>(sm_count()) * per_sm;
    if (grid > p.n_rows) grid = p.n_rows;
  }
  kern<<<static_cast<unsigned>(grid), THREADS, 0, st>>>(p);
  return check_launch("aa_logprob_fwd");
}

template <typename T>
static int launch_fwd_bulk(const FwdParams &p, cudaStream_t st) {
  constexpr int CONSUMERS = 256, STAGES = 4, UNROLL = 4;
  constexpr size_t smem = static_cast<size_t>(STAGES) * CONSUMERS * UNROLL * 16 + 2 * STAGES * sizeof(uint64_t);
  auto kern = logprob_fwd_bulk_kernel<T, CONSUMERS, STAGES, UNROLL>;
  static std::atomic<bool> configured{false};  // the attribute is idempotent: a race sets it twice, harmlessly
  if (!configured.load(std::memory_order_relaxed)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) {
      set_error("aa_logprob_fwd(bulk): cannot reserve %zu B of shared memory: %s", smem, cudaGetErrorString(e));
      return static_cast<int>(e);
    }
    configured.store(true, std::memory_order_relaxed);
  }
  const int resident = resident_ctas(reinterpret_cast<const void *>(kern), CONSUMERS + 32, smem);
  const int per_sm = (fwd_ctas() > 0 && fwd_ctas() < resident) ? fwd_ctas() : resident;
  int64_t grid = static_cast<int64_t>(sm_count()) * per_sm;
  if (grid > p.n_rows) grid = p.n_rows;
  kern<<<static_cast<unsigned>(grid), CONSUMERS + 32, smem, st>>>(p);
  return check_launch("aa_logprob_fwd(bulk)");
}

template <typename T>
static int launch_fwd(const FwdParams &p, cudaStream_t st) {
  if ((fwd_variant() % 10) == 1) return launch_fwd_bulk<T>(p, st);
  const int shape = (fwd_variant() / 10) % 10;
  const int per_sm = fwd_ctas();
  if constexpr (sizeof(T) == 2) {
    switch (shape) {
      case 1: return launch_fwd_shape<T, 256, 8>(p, per_sm, st);
      case 2: return launch_fwd_shape<T, 512, 4>(p, per_sm, st);
      case 3: return launch_fwd_shape<T, 128, 8>(p, per_sm, st);
      case 4: return launch_fwd_shape<T, 256, 2>(p, per_sm, st);
      case 5: return launch_fwd_shape<T, 512, 2>(p, per_sm, st);
      case kFwdLegacyShape: return launch_fwd_shape<T, 128, 8>(p, per_sm > 0 ? per_sm : 16, st, false);
      default: break;
    }
    // default (16-bit logits): 128 threads x 8 vectors, one CTA per row.  The block scheduler starts a row's CTA
    // whenever a resident one retires, so the rows go to whichever SM is free: a dynamic hand-out that needs no
    // work counter and is independent of other launches on other streams.  A static split of the rows over a
    // persistent grid finishes at the pace of the slowest SM.  Measured on the C2 tile (tools/k1_residency_ab.py,
    // DESIGN.md §3): one CTA per row reads 6.35 TB/s, the old 16-CTAs/SM persistent grid 5.90-6.03, a resident-sized
    // persistent grid (9 CTAs/SM) 5.82-5.85.
    return launch_fwd_shape<T, 128, 8>(p, per_sm > 0 ? per_sm : -1, st);
  }
  return launch_fwd_shape<T, 256, 4>(p, per_sm, st);
}

template <typename T, int THREADS, int UNROLL>
static int launch_bwd_shape(const BwdParams &p, int mode, int per_sm, cudaStream_t st) {
  const int64_t n_work = bwd_work_rows(p);
  int64_t grid = static_cast<int64_t>(sm_count()) * per_sm;
  if (grid > n_work) grid = n_work;
  const bool faithful = (mode == AA_MODE_FAITHFUL) && sizeof(T) == 2;
  if (faithful)
    logprob_bwd_kernel<T, THREADS, UNROLL, true><<<static_cast<unsigned>(grid), THREADS, 0, st>>>(p);
  else
    logprob_bwd_kernel<T, THREADS, UNROLL, false><<<static_cast<unsigned>(grid), THREADS, 0, st>>>(p);
  return check_launch("aa_logprob_bwd");
}

template <typename T, int THREADS, int UNROLL>
static int launch_bwd_chunk_shape(const BwdParams &p, int mode, int per_sm, RowRec *rec, cudaStream_t st) {
  constexpr int E = Traits<T>::kVec;
  const int64_t n_work = bwd_work_rows(p);
  bwd_row_prep_kernel<<<static_cast<unsigned>((n_work + 255) / 256), 256, 0, st>>>(p, rec);
  int rc = check_launch("aa_logprob_bwd(prep)");
  if (rc) return rc;
  const int span_vecs = (p.V + 2 * (E - 1)) / E + 1;
  const int upr = (span_vecs + THREADS * UNROLL - 1) / (THREADS * UNROLL);
  const int64_t n_units = n_work * upr;
  int64_t grid = static_cast<int64_t>(sm_count()) * per_sm;
  if (grid > n_units) grid = n_units;
  const bool faithful = (mode == AA_MODE_FAITHFUL) && sizeof(T) == 2;
  const T *lg = reinterpret_cast<const T *>(p.logits);
  T *gr = reinterpret_cast<T *>(p.grad_logits);
  if (faithful)
    logprob_bwd_chunk_kernel<T, THREADS, UNROLL, true>
        <<<static_cast<unsigned>(grid), THREADS, 0, st>>>(lg, gr, p.grad_row_stride, p.V, rec, n_work, upr, p.zero);
  else
    logprob_bwd_chunk_kernel<T, THREADS, UNROLL, false>
        <<<static_cast<unsigned>(grid), THREADS, 0, st>>>(lg, gr, p.grad_row_stride, p.V, rec, n_work, upr, p.zero);
  return check_launch("aa_logprob_bwd(chunk)");
}

template <typename T>
static int launch_bwd_chunk(const BwdParams &p, int mode, RowRec *rec, cudaStream_t st) {
  const int shape = (bwd_variant() / 10) % 10;
  const int per_sm = bwd_ctas() > 0 ? bwd_ctas() : 8;
  if constexpr (sizeof(T) == 2) {
    switch (shape) {
      case 1: return launch_bwd_chunk_shape<T, 256, 8>(p, mode, per_sm, rec, st);
      case 2: return launch_bwd_chunk_shape<T, 512, 4>(p, mode, bwd_ctas() > 0 ? bwd_ctas() : 4, rec, st);
      case 3: return launch_bwd_chunk_shape<T, 128, 8>(p, mode, bwd_ctas() > 0 ? bwd_ctas() : 16, rec, st);
      case 4: return launch_bwd_chunk_shape<T, 256, 2>(p, mode, per_sm, rec, st);
      case 5: return launch_bwd_chunk_shape<T, 512, 2>(p, mode, bwd_ctas() > 0 ? bwd_ctas() : 4, rec, st);
      default: break;
    }
  }
  return launch_bwd_chunk_shape<T, 256, 4>(p, mode, per_sm, rec, st);
}

template <typename T, int CONSUMERS, int STAGES, int UNROLL, int LAG>
static int launch_bwd_tma_shape(const BwdParams &p, int mode, int per_sm, RowRec *rec, cudaStream_t st) {
  const int64_t n_work = bwd_work_rows(p);
  bwd_row_prep_kernel<<<static_cast<unsigned>((n_work + 255) / 256), 256, 0, st>>>(p, rec);
  int rc = check_launch("aa_logprob_bwd(prep)");
  if (rc) return rc;
  constexpr size_t smem = static_cast<size_t>(STAGES + 1) * CONSUMERS * UNROLL * 16 + STAGES * (8 + 8 + 8 + 4) + 16;
  const bool faithful = (mode == AA_MODE_FAITHFUL) && sizeof(T) == 2;
  auto kf = logprob_bwd_tma_kernel<T, CONSUMERS, STAGES, UNROLL, LAG, true>;
  auto kn = logprob_bwd_tma_kernel<T, CONSUMERS, STAGES, UNROLL, LAG, false>;
  static std::atomic<bool> configured{false};  // the attribute is idempotent: a race sets it twice, harmlessly
  if (!configured.load(std::memory_order_relaxed)) {
    cudaError_t e = cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(kn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) {
      set_error("aa_logprob_bwd(tma): cannot reserve %zu B of shared memory: %s", smem, cudaGetErrorString(e));
      return static_cast<int>(e);
    }
    configured.store(true, std::memory_order_relaxed);
  }
  int64_t grid = static_cast<int64_t>(sm_count()) * per_sm;
  if (grid > n_work) grid = n_work;
  const T *lg = reinterpret_cast<const T *>(p.logits);
  T *gr = reinterpret_cast<T *>(p.grad_logits);
  if (faithful)
    kf<<<static_cast<unsigned>(grid), CONSUMERS + 32, smem, st>>>(lg, gr, p.grad_row_stride, p.V, rec, n_work, p.zero);
  else
    kn<<<static_cast<unsigned>(grid), CONSUMERS + 32, smem, st>>>(lg, gr, p.grad_row_stride, p.V, rec, n_work, p.zero);
  return check_launch("aa_logprob_bwd(tma)");
}

// shape codes of the TMA-staged backward (stages x stage size, lag, default CTAs/SM):
//   0 (default): 4 x 8 KB, lag 3, 3 CTAs/SM   1: 4 x 16 KB, lag 2, 2   2: 4 x 8 KB, lag 3, 3 (= default)
//   3: 6 x 8 KB, lag 4, 2                     4: 3 x 16 KB, lag 2, 2   5: 8 x 8 KB, lag 6, 2   6: 4 x 16 KB, lag 3, 2
// Measured (bench.py, sustained, 67.2 GB per launch): 4x8KB/lag3 x3 CTAs -> 10.37 ms = 6.48 TB/s (0.986 of the
// measured copy peak); x4 CTAs 5.92; 4x16KB/lag3 x2 CTAs 6.38, x3 5.69; 6x8KB x3 5.94; LDG row kernel 5.79.
template <typename T>
static int launch_bwd_tma(const BwdParams &p, int mode, RowRec *rec, cudaStream_t st) {
  const int shape = (bwd_variant() / 10) % 10;
  const int c = bwd_ctas();
  switch (shape) {
    case 1: return launch_bwd_tma_shape<T, 256, 4, 4, 2>(p, mode, c > 0 ? c : 2, rec, st);
    case 3: return launch_bwd_tma_shape<T, 256, 6, 2, 4>(p, mode, c > 0 ? c : 2, rec, st);
    case 4: return launch_bwd_tma_shape<T, 256, 3, 4, 2>(p, mode, c > 0 ? c : 2, rec, st);
    case 5: return launch_bwd_tma_shape<T, 256, 8, 2, 6>(p, mode, c > 0 ? c : 2, rec, st);
    case 6: return launch_bwd_tma_shape<T, 256, 4, 4, 3>(p, mode, c > 0 ? c : 2, rec, st);
    default: break;
  }
  return launch_bwd_tma_shape<T, 256, 4, 2, 3>(p, mode, c > 0 ? c : 3, rec, st);
}

template <typename T>
static int launch_bwd(const BwdParams &p, int mode, cudaStream_t st) {
  const int shape = (bwd_variant() / 10) % 10;
  const int per_sm = bwd_ctas() > 0 ? bwd_ctas() : 6;
  if constexpr (sizeof(T) == 2) {
    switch (shape) {
      case 1: return launch_bwd_shape<T, 256, 8>(p, mode, per_sm, st);
      case 2: return launch_bwd_shape<T, 512, 4>(p, mode, bwd_ctas() > 0 ? bwd_ctas() : 3, st);
      case 3: return launch_bwd_shape<T, 128, 8>(p, mode, bwd_ctas() > 0 ? bwd_ctas() : 12, st);
      case 4: return launch_bwd_shape<T, 256, 2>(p, mode, per_sm, st);
      case 5: return launch_bwd_shape<T, 512, 2>(p, mode, bwd_ctas() > 0 ? bwd_ctas() : 3, st);
      default: break;
    }
  }
  // default (16-bit logits).  The read+write stream is sensitive to how much is in flight per SM and the
  // optimum depends on the compute per byte of the variant (tools/sweep_k1.py, V = 128257, reproducible
  // to 1%; torch's copy_ reaches 6.6 TB/s on the same boxes):
  //   FAITHFUL (Veltkamp rounding, ~7 instr/elem): 512 thr x 4 vec x 3 CTAs/SM -> 5.74 TB/s sustained in
  //     bench.py (5.86-5.91 burst); 512x2x4 -> 5.44 sustained (5.89 burst); 512x2x3 -> 5.40 burst.
  //   F32 mode (~3.5 instr/elem): 512x2x3 -> 5.93 TB/s burst (x4: 5.56).
  if constexpr (sizeof(T) == 2) {
    if (mode == AA_MODE_FAITHFUL) return launch_bwd_shape<T, 512, 4>(p, mode, bwd_ctas() > 0 ? bwd_ctas() : 3, st);
    return launch_bwd_shape<T, 512, 2>(p, mode, bwd_ctas() > 0 ? bwd_ctas() : 3, st);
  }
  return launch_bwd_shape<T, 256, 4>(p, mode, bwd_ctas() > 0 ? bwd_ctas() : 4, st);
}

}  // namespace aa

using namespace aa;

extern "C" int aa_logprob_set_tuning(int variant, int ctas_per_sm) {
  AA_REQUIRE(variant >= 0 && variant < 100 && variant % 10 <= 3, AA_ERR_ARG,
             "aa_logprob_set_tuning: variant = kernel digit (0..3) + 10 * shape code");
  g_variant = variant;
  g_ctas_per_sm = ctas_per_sm;
  g_bwd_variant = -1;
  return AA_OK;
}

extern "C" int aa_logprob_set_tuning_bwd(int variant, int ctas_per_sm) {
  AA_REQUIRE(variant >= -1 && variant < 100 && (variant < 0 || variant % 10 <= 3), AA_ERR_ARG,
             "aa_logprob_set_tuning_bwd: variant = -1 (follow forward) or kernel + 10 * shape code");
  g_bwd_variant = variant;
  g_bwd_ctas_per_sm = ctas_per_sm;
  return AA_OK;
}

extern "C" int aa_logprob_fwd(const void *logits, int logits_dtype, int64_t row_stride, int32_t V,
                              const int64_t *labels, int64_t ignore_index, int32_t use_ignore,
                              int32_t n_segments, int64_t n_rows,
                              const int64_t *seg_logit_off, const int64_t *seg_label_off,
                              const int64_t *seg_out_off, const int64_t *seg_cum, void *out,
                              int out_dtype, float *stat_max, float *stat_logsum, int32_t *status,
                              void *stream) {
  AA_REQUIRE(V > 0 && n_segments >= 0 && n_rows >= 0, AA_ERR_ARG, "aa_logprob_fwd: bad sizes");
  if (n_rows == 0 || n_segments == 0) return AA_OK;
  AA_REQUIRE(logits && labels && out && seg_logit_off && seg_label_off && seg_out_off && seg_cum,
             AA_ERR_ARG, "aa_logprob_fwd: null pointer");
  AA_REQUIRE((stat_max == nullptr) == (stat_logsum == nullptr), AA_ERR_ARG,
             "aa_logprob_fwd: stat_max and stat_logsum go together");
  AA_REQUIRE(out_dtype == AA_BF16 || out_dtype == AA_F16 || out_dtype == AA_F32, AA_ERR_DTYPE,
             "aa_logprob_fwd: bad out_dtype %d", out_dtype);
  const int esz = dtype_size(logits_dtype);
  AA_REQUIRE(reinterpret_cast<uintptr_t>(logits) % esz == 0, AA_ERR_ALIGN,
             "aa_logprob_fwd: logits not element-aligned");
  FwdParams p{logits, row_stride, V, labels, ignore_index, use_ignore,
              RowMap{seg_logit_off, seg_label_off, seg_out_off, seg_cum, n_segments},
              n_rows, out, out_dtype, stat_max, stat_logsum, status, kLog2e};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (logits_dtype) {
    case AA_BF16: return launch_fwd<__nv_bfloat16>(p, st);
    case AA_F16: return launch_fwd<__half>(p, st);
    case AA_F32: return launch_fwd<float>(p, st);
  }
  set_error("aa_logprob_fwd: unsupported logits dtype %d", logits_dtype);
  return AA_ERR_DTYPE;
}

extern "C" int aa_zero_rows(void *tile, int dtype, int64_t row_stride, int32_t V, int64_t n_tile_rows,
                            const int64_t *spans_host, int32_t n_spans, void *stream) {
  AA_REQUIRE(V > 0 && row_stride >= V && n_spans >= 0 && n_tile_rows >= 0, AA_ERR_ARG, "aa_zero_rows: bad sizes");
  if (n_spans == 0) return AA_OK;
  AA_REQUIRE(tile && spans_host, AA_ERR_ARG, "aa_zero_rows: null pointer");
  AA_REQUIRE(dtype == AA_BF16 || dtype == AA_F16 || dtype == AA_F32, AA_ERR_DTYPE, "aa_zero_rows: bad dtype");
  const size_t esz = (dtype == AA_F32) ? 4 : 2;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const uintptr_t lo = reinterpret_cast<uintptr_t>(tile);
  const uintptr_t hi = lo + static_cast<size_t>(n_tile_rows) * V * esz;  // contiguous tiles only
  constexpr uintptr_t kAlign = 256;
  for (int32_t i = 0; i < n_spans; ++i) {
    const int64_t first = spans_host[2 * i], n = spans_host[2 * i + 1];
    AA_REQUIRE(first >= 0 && n >= 0 && first + n <= n_tile_rows, AA_ERR_ARG, "aa_zero_rows: bad span %d", i);
    if (n == 0) continue;
    cudaError_t e;
    if (row_stride == V) {
      // Rows of an odd vocabulary (V = 128257) start 2-byte aligned, and a memset whose ends are not aligned runs
      // at a fraction of the copy engine's rate.  The rows next to a span are rewritten in full by the kernel that
      // follows in stream order, so the span is widened to 256-byte boundaries (inside the tile).
      uintptr_t a = (lo + static_cast<size_t>(first) * V * esz) & ~(kAlign - 1);
      uintptr_t b = (lo + static_cast<size_t>(first + n) * V * esz + kAlign - 1) & ~(kAlign - 1);
      if (a < lo) a = lo;
      if (b > hi) b = hi;
      e = cudaMemsetAsync(reinterpret_cast<void *>(a), 0, b - a, st);
    } else {
      char *dst = static_cast<char *>(tile) + static_cast<size_t>(first) * row_stride * esz;
      e = cudaMemset2DAsync(dst, static_cast<size_t>(row_stride) * esz, 0, static_cast<size_t>(V) * esz,
                            static_cast<size_t>(n), st);
    }
    if (e != cudaSuccess) {
      set_error("aa_zero_rows: %s", cudaGetErrorString(e));
      return static_cast<int>(e);
    }
  }
  return AA_OK;
}

extern "C" int aa_logprob_bwd(const void *logits, int logits_dtype, int64_t row_stride, int32_t V,
                              const int64_t *labels, int64_t ignore_index, int32_t use_ignore,
                              int32_t n_segments, int64_t n_rows,
                              const int64_t *seg_logit_off, const int64_t *seg_label_off,
                              const int64_t *seg_out_off, const int64_t *seg_cum,
                              const int64_t *seg_tile_row, const float *stat_max,
                              const float *stat_logsum, const void *grad_rows, int grad_rows_dtype,
                              const float *grad_seg, const void *grad_scale, int grad_scale_dtype, void *grad_logits,
                              int64_t grad_row_stride, int64_t n_tile_rows, const int64_t *extra_zero_rows,
                              int64_t n_extra_zero_rows, void *row_scratch, int mode, void *stream) {
  AA_REQUIRE(V > 0 && n_segments >= 0 && n_rows >= 0 && n_tile_rows >= 0 && n_extra_zero_rows >= 0, AA_ERR_ARG,
             "aa_logprob_bwd: bad sizes");
  AA_REQUIRE(n_extra_zero_rows == 0 || (n_tile_rows == 0 && extra_zero_rows), AA_ERR_ARG,
             "aa_logprob_bwd: extra_zero_rows needs n_tile_rows == 0 and a device row list");
  if (n_segments == 0) n_rows = 0;
  if (n_tile_rows == 0 && n_rows == 0 && n_extra_zero_rows == 0) return AA_OK;
  AA_REQUIRE(grad_logits, AA_ERR_ARG, "aa_logprob_bwd: null grad_logits");
  if (n_segments > 0)
    AA_REQUIRE(logits && labels && seg_logit_off && seg_label_off && seg_out_off && seg_cum &&
                   seg_tile_row && stat_max && stat_logsum,
               AA_ERR_ARG, "aa_logprob_bwd: null pointer");
  AA_REQUIRE(mode == AA_MODE_FAITHFUL || mode == AA_MODE_F32, AA_ERR_ARG, "aa_logprob_bwd: bad mode");
  AA_REQUIRE(!grad_scale || grad_scale_dtype == AA_BF16 || grad_scale_dtype == AA_F16 || grad_scale_dtype == AA_F32,
             AA_ERR_DTYPE, "aa_logprob_bwd: bad grad_scale dtype");
  BwdParams p{logits, row_stride, V, labels, ignore_index, use_ignore,
              RowMap{seg_logit_off, seg_label_off, seg_out_off, seg_cum, n_segments},
              n_rows, seg_tile_row, stat_max, stat_logsum, grad_rows, grad_rows_dtype, grad_seg,
              grad_scale, grad_scale_dtype, grad_logits, grad_row_stride, n_tile_rows, 0.0f, extra_zero_rows, n_extra_zero_rows};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (row_scratch && (bwd_variant() % 10) <= 1) {  // kernel digit 0 / 1: TMA-staged backward (the default)
    AA_REQUIRE((reinterpret_cast<uintptr_t>(row_scratch) & 15) == 0, AA_ERR_ALIGN,
               "aa_logprob_bwd: row_scratch must be 16-byte aligned");
    RowRec *rec = static_cast<RowRec *>(row_scratch);
    switch (logits_dtype) {
      case AA_BF16: return launch_bwd_tma<__nv_bfloat16>(p, mode, rec, st);
      case AA_F16: return launch_bwd_tma<__half>(p, mode, rec, st);
      case AA_F32: return launch_bwd_tma<float>(p, mode, rec, st);
    }
  }
  if (row_scratch && (bwd_variant() % 10) == 2) {  // kernel digit 2: address-ordered chunked sweep (slower on B200, kept for study)
    AA_REQUIRE((reinterpret_cast<uintptr_t>(row_scratch) & 15) == 0, AA_ERR_ALIGN,
               "aa_logprob_bwd: row_scratch must be 16-byte aligned");
    RowRec *rec = static_cast<RowRec *>(row_scratch);
    switch (logits_dtype) {
      case AA_BF16: return launch_bwd_chunk<__nv_bfloat16>(p, mode, rec, st);
      case AA_F16: return launch_bwd_chunk<__half>(p, mode, rec, st);
      case AA_F32: return launch_bwd_chunk<float>(p, mode, rec, st);
    }
  }
  switch (logits_dtype) {
    case AA_BF16: return launch_bwd<__nv_bfloat16>(p, mode, st);
    case AA_F16: return launch_bwd<__half>(p, mode, st);
    case AA_F32: return launch_bwd<float>(p, mode, st);
  }
  set_error("aa_logprob_bwd: unsupported logits dtype %d", logits_dtype);
  return AA_ERR_DTYPE;
}

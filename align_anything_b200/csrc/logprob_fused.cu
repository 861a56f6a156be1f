// logprob_fused.cu -- K1f: log-probs, the loss's per-token gradient and the gradient tile in ONE pass over the logits tile,
// for losses that are (masked) means of per-token terms: the PPO actor loss (described below), the causal-LM cross-entropy
// (aa_logprob_ce_fused: trainers/text_to_text/sft.py:95-98, ppo.py:400-408) and the GRPO loss (aa_logprob_grpo_fused:
// trainers/text_to_text/grpo.py:290-312).  The three differ only in the record the prep kernel writes per row and in the
// per-token function the boundary thread calls (csrc/ppo_math.cuh).
//
// Reference: trainers/text_image_to_text/ppo.py:296-316 (text: trainers/text_to_text/ppo.py:336-349):
//     logits = actor(**batch).logits ; log_probs = gather_log_probabilities(logits[b, :-1][-R:], ids[b, 1:][-R:])
//     actor_loss = actor_loss_fn(log_probs, old_log_probs, advantages, mask) ; actor_model.backward(actor_loss)
// i.e. K1 (read the scored rows) -> K5 -> K1b (read the scored rows AGAIN, write the gradient tile).
//
// The clipped-ratio objective is a masked MEAN of per-token terms: d loss / d log_prob[b, t] depends on that token's own
// log-prob, on (old_log_prob, advantage, mask)[b, t] and on the row's mask count -- all known before the forward.  So
// the gradient row can be produced right after the row's (max, logsum), while the row is still on the chip:
//
//   per scored row, one CTA:   phase A  stream the row through a shared-memory ring (cp.async.bulk), online softmax
//                              boundary one thread: log-prob -> actor_token() -> g = d loss / d log-prob
//                              phase B  stream the SAME row again -- 304 KB at V = 152064, read a few microseconds ago
//                                       by this CTA, so the copy engine finds it in the 126 MB L2 (phase-A loads carry
//                                       an L2 evict_last policy, phase-B loads and the stores evict_first) --
//                                       g * (onehot - softmax) in place in shared memory, cp.async.bulk stores.
//
// HBM traffic per scored row: V*e read + V*e written instead of 2*V*e read + V*e written (K1 + K1b); unscored tile rows
// are written by the copy engine from a zeroed buffer, as in K1b.  The loss VALUE is still reduced by K5 from the
// log-probs this kernel writes (a 16 us launch); autograd's backward returns the tile produced here, multiplied in
// place by the incoming scalar only if that is not 1 (aa_scale_tile: every CTA reads the scalar and leaves).
#include <atomic>
#include <cstdlib>

#include "common.cuh"
#include "logprob_math.cuh"
#include "ppo_math.cuh"

namespace aa {

struct FusedActorParams {
  const void *logits;
  int64_t row_stride;
  int V;
  const int64_t *labels;
  RowMap map;
  const int64_t *seg_tile_row;
  int seq;  // tile rows per segment (n_tile_rows / n_seg)
  void *out;
  int out_dtype;
  float *stat_max, *stat_logsum;  // optional
  const void *old;
  int64_t old_stride;
  const void *adv;
  int64_t adv_stride;
  int adv_dtype;
  const uint8_t *mask;
  int64_t mask_stride;
  int W;
  float clip;
  int rx, rp;
  void *grad;
  int64_t grad_row_stride;
  int32_t *status;
  float log2e, zero;
  int hint;  // L2 policy of the bulk copies: 0 none, 1 phase A evict_last / phase B + stores evict_first
  int interleave;  // > 0: size of the persistent grid -- the work list alternates `interleave` scored rows / zero rows
  // kind 1 (cross-entropy, aa_logprob_ce_fused): every row whose label != ignore_index has the SAME upstream gradient
  // *ce_coeff = -loss_scale / n_valid (written by ce_coeff_kernel); old / adv / mask are unused
  // kind 2 (GRPO, aa_logprob_grpo_fused): old = reference log-probs, adv = ONE fp32 advantage per segment, clip = beta,
  // a token counts while j < row_end[segment], 1 / *total is d loss / d per-token loss (grpo_mask_kernel wrote both)
  int kind;
  int64_t ignore_index;
  const float *ce_coeff;
  const int32_t *row_end;
  const float *total;
};

// One record per gradient-tile row, in the order the persistent kernel walks them.  The scored rows are bound by
// instruction issue / MUFU (two exp per logit in one kernel), the zero rows are pure copy-engine stores: the list
// alternates G scored rows and G zero rows (G = grid size), so every CTA's producer lane fires the stores of a zero
// row while its consumer warps are still busy with the scored row before it -- the zero rows ride in the DRAM
// bandwidth the compute-bound rows leave unused.  (interleave == 0: scored rows first, zero rows after, as in K1b.)
struct __align__(16) FusedRec {
  int64_t x_off;    // element offset of the logits row
  int64_t g_row;    // row index in the gradient tile
  int64_t out_idx;  // element index of the log-prob in `out` (and of old / adv / mask relative to their row starts)
  float old, adv, g_rs;
  int32_t y;        // label column; -1: out of range; -2: zero row
  int32_t flat;     // index into stat_max / stat_logsum
  int32_t on;       // mask bit
};
static_assert(sizeof(FusedRec) == 48, "FusedRec is read as three 16-byte vectors");

// grid (ceil(seq / 256), n_seg): block (c, seg) resolves tile rows [256 c, 256 c + 256) of sample `seg`.
__global__ void __launch_bounds__(256) fused_actor_prep_kernel(const FusedActorParams p, FusedRec *__restrict__ rec) {
  __shared__ float scratch[33];
  const int seg = blockIdx.y, tid = threadIdx.x;
  const int k = blockIdx.x * 256 + tid;
  float cnt = 0.f;
  if (p.kind == 0) {
    for (int t = tid; t < p.W; t += 256) cnt += p.mask[seg * p.mask_stride + t] ? 1.f : 0.f;
    cnt = block_sum<256>(cnt, scratch);
  }
  if (k >= p.seq) return;
  const int64_t work = static_cast<int64_t>(seg) * p.seq + k;
  const int64_t first_flat = __ldg(p.map.seg_cum + seg);
  const int64_t n = __ldg(p.map.seg_cum + seg + 1) - first_flat;
  const int64_t total = __ldg(p.map.seg_cum + p.map.n_seg);
  const int64_t j = work - __ldg(p.seg_tile_row + seg);
  const bool scored = j >= 0 && j < n;
  const int64_t scored_before = first_flat + min(max(j, static_cast<int64_t>(0)), n);
  int64_t slot;
  if (p.interleave > 0) {
    const int64_t G = p.interleave, Z = static_cast<int64_t>(p.map.n_seg) * p.seq - total;
    if (scored) {
      const int64_t i = first_flat + j;
      slot = i + min((i / G) * G, Z);                // zero rows of the earlier rounds come first
    } else {
      const int64_t z = work - scored_before;
      slot = min((z / G + 1) * G, total) + z;        // scored rows of this and the earlier rounds come first
    }
  } else {
    slot = scored ? first_flat + j : total + (work - scored_before);
  }
  FusedRec r;
  r.x_off = 0; r.g_row = work; r.out_idx = 0; r.old = 0.f; r.adv = 0.f; r.g_rs = 0.f; r.y = -2; r.flat = 0; r.on = 0;
  if (scored) {
    const int64_t y = __ldg(p.labels + __ldg(p.map.seg_label_off + seg) + j);
    if (p.kind != 1 || y != p.ignore_index) {  // cross-entropy: an ignored position is a zero row (its log-prob stays 0: no traffic)
      r.x_off = __ldg(p.map.seg_logit_off + seg) + j * p.row_stride;
      r.out_idx = __ldg(p.map.seg_out_off + seg) + j;
      r.y = (y >= 0 && y < p.V) ? static_cast<int32_t>(y) : -1;
      r.flat = static_cast<int32_t>(first_flat + j);
      if (p.kind == 0) {
        r.old = load_as_float(p.old, seg * p.old_stride + j, p.out_dtype);
        r.adv = load_as_float(p.adv, seg * p.adv_stride + j, p.adv_dtype);
        r.g_rs = actor_row_coeff(cnt, p.map.n_seg, p.rp);
        r.on = p.mask[seg * p.mask_stride + j] ? 1 : 0;
      } else if (p.kind == 2) {
        r.old = load_as_float(p.old, seg * p.old_stride + j, p.out_dtype);
        r.adv = reinterpret_cast<const float *>(p.adv)[seg];
        r.g_rs = 1.f / __ldg(p.total);
        r.on = (j < __ldg(p.row_end + seg)) ? 1 : 0;
      } else {
        r.g_rs = __ldg(p.ce_coeff);
        r.on = 1;
      }
    }
  }
  rec[slot] = r;
}

namespace bulk {
__device__ __forceinline__ uint64_t policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void bulk_g2s_hint(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar,
                                              uint64_t pol) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
      : "memory");
}
__device__ __forceinline__ void bulk_s2g(void *dst_gmem, const void *src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_s2g_hint(void *dst_gmem, const void *src_smem, uint32_t bytes, uint64_t pol) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(dst_gmem),
               "r"(smem_u32(src_smem)), "r"(bytes), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
}  // namespace bulk

// vec_grad (logprob_math.cuh) with the reference's 16-bit rounding of the log-softmax done by ONE F2FP.PACK_AB per pair
// (+ two ALU unpacks) instead of the Veltkamp split on the FMA pipe (FFMA2 + 2 FADD2): the same bits for finite values,
// -inf logits need no clamp (HMNMX2), and three instructions per pair move from the FMA-heavy pipe -- the busiest one
// of this kernel, 57 % -- to the ALU pipe (36 %).  K1b keeps the split: it is HBM-bound with the XU pipe as runner-up.
#ifndef AA_K1F_PACK_ROUND
#define AA_K1F_PACK_ROUND 1
#endif
template <typename T, bool FAITHFUL>
__device__ __forceinline__ uint4 vec_grad_pk(const uint4 &v, const GradConsts &k) {
  if constexpr (sizeof(T) == 4 || !FAITHFUL || !AA_K1F_PACK_ROUND) {
    return vec_grad<T, FAITHFUL>(v, k);
  } else {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float lo, hi;
      unpack2<T>(w[i], lo, hi);
      f2_unpack(f2_sub(f2_sub(f2_pack(lo, hi), k.m2), k.ls2), lo, hi);
      unpack2<T>(pack2<T>(lo, hi), lo, hi);  // round_T((x - max) - logsum): what ATen's backward re-reads
      f2_unpack(f2_mul(f2_ex2(f2_mul(f2_pack(lo, hi), f2_splat(kLog2e))), k.ng2), lo, hi);
      o[i] = pack2<T>(lo, hi);
    }
    return make_uint4(o[0], o[1], o[2], o[3]);
  }
}

template <typename T, int CONSUMERS, int STAGES, int UNROLL, int LAG, bool FAITHFUL>
__global__ void __launch_bounds__(CONSUMERS + 32)
    logprob_actor_fused_kernel(const FusedActorParams p, const FusedRec *__restrict__ rec, int64_t n_work) {
  constexpr int E = Traits<T>::kVec;
  constexpr int STAGE_VECS = CONSUMERS * UNROLL;
  constexpr int NW = CONSUMERS / kWarp;
  static_assert(LAG >= 2 && LAG < STAGES, "phase A holds two stages at a time; LAG must leave at least one free stage");
  extern __shared__ __align__(128) uint8_t smem_raw[];
  uint4 *ring = reinterpret_cast<uint4 *>(smem_raw);
  uint4 *zero_buf = ring + static_cast<size_t>(STAGES) * STAGE_VECS;
  uint64_t *full = reinterpret_cast<uint64_t *>(zero_buf + STAGE_VECS);
  uint64_t *done = full + STAGES;
  uint64_t *st_dst = done + STAGES;  // destination of the chunk held by each stage (phase B), 0 for phase A
  uint32_t *st_bytes = reinterpret_cast<uint32_t *>(st_dst + STAGES);
  __shared__ float sh_m[32], sh_s[32], sh_b[4];
  const int tid = threadIdx.x;
  const int V = p.V;
  const T *__restrict__ logits = reinterpret_cast<const T *>(p.logits);
  T *__restrict__ grad = reinterpret_cast<T *>(p.grad);
  for (int i = tid; i < STAGE_VECS; i += CONSUMERS + 32) zero_buf[i] = make_uint4(0, 0, 0, 0);
  if (tid == 0) {
    for (int i = 0; i < STAGES; ++i) {
      bulk::mbar_init(full + i, 1);
      bulk::mbar_init(done + i, NW);
    }
    bulk::fence_barrier_init();
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // zero_buf is read by the async proxy
  __syncthreads();

  if (tid >= CONSUMERS) {
    // ------------------------------ producer lane ------------------------------
    if (tid != CONSUMERS) return;
    const uint64_t pol_keep = bulk::policy_evict_last(), pol_drop = bulk::policy_evict_first();
    // ring positions are kept as (stage, parity) pairs stepped by hand: `it % STAGES` with a 64-bit counter and
    // STAGES = 6 is a ~40-instruction division per chunk (seen in the SASS of the first version)
    int inflight = 0;                     // chunks loaded and not yet handed back
    int ld_stage = 0;                     // stage of the next load
    int rt_stage = 0;                     // stage of the next chunk to hand back (phase A: freed; phase B: stored)
    uint32_t rt_phase = 0;
    auto retire_one = [&]() {
      const int s = rt_stage;
      bulk::mbar_wait(done + s, rt_phase);
      if (st_bytes[s]) {
        void *dst = reinterpret_cast<void *>(st_dst[s]);
        if (p.hint)
          bulk::bulk_s2g_hint(dst, ring + static_cast<size_t>(s) * STAGE_VECS, st_bytes[s], pol_drop);
        else
          bulk::bulk_s2g(dst, ring + static_cast<size_t>(s) * STAGE_VECS, st_bytes[s]);
      }
      bulk::commit_group();  // one (possibly empty) group per chunk: wait_group.read below counts chunks
      --inflight;
      if (++rt_stage == STAGES) {
        rt_stage = 0;
        rt_phase ^= 1u;
      }
    };
    // zero rows are not stored in one burst: their chunks are fed to the copy engine one per chunk load of the scored
    // row that follows, so the engine's queue never holds a whole 300 KB row in front of the loads the consumers wait for
    uint4 *zq_dst = nullptr;
    int zq_left = 0;  // vectors of the pending zero row not yet handed to the copy engine
    auto zero_some = [&](int max_chunks) {
      while (zq_left > 0 && max_chunks-- > 0) {
        const int n = min(STAGE_VECS, zq_left);
        if (p.hint)
          bulk::bulk_s2g_hint(zq_dst, zero_buf, static_cast<uint32_t>(n) * 16u, pol_drop);
        else
          bulk::bulk_s2g(zq_dst, zero_buf, static_cast<uint32_t>(n) * 16u);
        zq_dst += n;
        zq_left -= n;
      }
    };
    for (int64_t r = blockIdx.x; r < n_work; r += gridDim.x) {
      const int4 r0 = __ldg(reinterpret_cast<const int4 *>(rec + r));
      const int4 r2 = __ldg(reinterpret_cast<const int4 *>(rec + r) + 2);
      const int64_t x_off = (static_cast<int64_t>(static_cast<uint32_t>(r0.y)) << 32) | static_cast<uint32_t>(r0.x);
      const int64_t g_row = (static_cast<int64_t>(static_cast<uint32_t>(r0.w)) << 32) | static_cast<uint32_t>(r0.z);
      const int y = r2.y, on = r2.w;
      T *g_out = grad + g_row * p.grad_row_stride;
      const T *x = logits + x_off;
      const bool same_phase = ((reinterpret_cast<uintptr_t>(x) ^ reinterpret_cast<uintptr_t>(g_out)) & 15) == 0;
      // geometry of the row the chunks come from (scored rows: the logits row; it shares g_out's 16-byte phase)
      const uintptr_t ref = (y == -2) ? reinterpret_cast<uintptr_t>(g_out) : reinterpret_cast<uintptr_t>(x);
      const int mis = static_cast<int>((ref & 15) / sizeof(T));
      const int head = mis ? min(E - mis, V) : 0;
      const int nvec = (V - head) / E;
      const int tail0 = head + nvec * E;
      const uint4 *xbody = reinterpret_cast<const uint4 *>(x + head);
      uint4 *gbody = reinterpret_cast<uint4 *>(g_out + head);
      if (y != -2 && same_phase) {
        for (int ph = 0; ph < (on ? 2 : 1); ++ph) {
          for (int v0 = 0; v0 < nvec; v0 += STAGE_VECS) {
            const uint32_t bytes = static_cast<uint32_t>(min(STAGE_VECS, nvec - v0)) * 16u;
            while (inflight >= LAG) retire_one();
            const int s = ld_stage;
            // the stage's previous chunk was handed to the copy engine at least STAGES - LAG groups ago: wait until the
            // engine has finished READING it (later groups may stay pending)
            asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(STAGES - LAG) : "memory");
            st_dst[s] = reinterpret_cast<uint64_t>(gbody + v0);
            st_bytes[s] = ph ? bytes : 0u;
            bulk::mbar_expect_tx(full + s, bytes);
            if (p.hint)
              bulk::bulk_g2s_hint(ring + static_cast<size_t>(s) * STAGE_VECS, xbody + v0, bytes, full + s,
                                  ph ? pol_drop : pol_keep);
            else
              bulk::bulk_g2s(ring + static_cast<size_t>(s) * STAGE_VECS, xbody + v0, bytes, full + s);
            ++inflight;
            if (++ld_stage == STAGES) ld_stage = 0;
            zero_some(1);  // joins the group of the next retired chunk
          }
        }
      }
      if (y == -2 || (!on && same_phase)) {  // zero row: the copy engine writes it from the zero buffer
        zero_some(1 << 30);                  // (whatever is left of the previous one first)
        for (int e = 0; e < head; ++e) g_out[e] = Traits<T>::from_float(0.f);
        for (int e = tail0; e < V; ++e) g_out[e] = Traits<T>::from_float(0.f);
        zq_dst = gbody;
        zq_left = nvec;
      }
    }
    zero_some(1 << 30);
    bulk::commit_group();
    while (inflight > 0) retire_one();
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // smem must outlive the engine's reads / the stores
    return;
  }

  // ------------------------------ consumer warps ------------------------------
  const f32x2 L2 = f2_splat(p.log2e);
  const int lane = tid & 31, wid = tid >> 5;
  int stage = 0;       // ring position of the next chunk, stepped by hand (see the producer)
  uint32_t phase = 0;
  for (int64_t r = blockIdx.x; r < n_work; r += gridDim.x) {
    const int4 r0 = __ldg(reinterpret_cast<const int4 *>(rec + r));
    const int4 r1 = __ldg(reinterpret_cast<const int4 *>(rec + r) + 1);
    const int4 r2 = __ldg(reinterpret_cast<const int4 *>(rec + r) + 2);
    const int y = r2.y;
    if (y == -2) continue;
    const int64_t x_off = (static_cast<int64_t>(static_cast<uint32_t>(r0.y)) << 32) | static_cast<uint32_t>(r0.x);
    const int64_t g_row = (static_cast<int64_t>(static_cast<uint32_t>(r0.w)) << 32) | static_cast<uint32_t>(r0.z);
    const int64_t out_idx = (static_cast<int64_t>(static_cast<uint32_t>(r1.y)) << 32) | static_cast<uint32_t>(r1.x);
    const float old = __int_as_float(r1.z), adv = __int_as_float(r1.w), g_rs = __int_as_float(r2.x);
    const int flat = r2.z;
    const bool on = r2.w != 0;
    T *g_out = grad + g_row * p.grad_row_stride;
    const T *x = logits + x_off;
    const bool same_phase = ((reinterpret_cast<uintptr_t>(x) ^ reinterpret_cast<uintptr_t>(g_out)) & 15) == 0;
    const int mis = static_cast<int>((reinterpret_cast<uintptr_t>(x) & 15) / sizeof(T));
    const int head = mis ? min(E - mis, V) : 0;
    const int nvec = (V - head) / E;
    const int tail0 = head + nvec * E;

    float xy = 0.f;
    if (tid == 0) xy = (y >= 0) ? Traits<T>::to_float(x[y]) : NAN;  // label column, issued before the streaming loop

    // ---- phase A: (max, sum exp) of the row ----
    float m = -INFINITY, s = 0.f;
    if (same_phase) {
      if (tid < head) lse_push(m, s, Traits<T>::to_float(x[tid]));
      if (tid < V - tail0) lse_push(m, s, Traits<T>::to_float(x[tail0 + tid]));
      // two stages per fold: the running-max rescale (one MUFU, a compare and a select) is paid per 4 vectors
      for (int v0 = 0; v0 < nvec; v0 += 2 * STAGE_VECS) {
        const int n0 = min(STAGE_VECS, nvec - v0);
        const int n1 = min(STAGE_VECS, max(nvec - v0 - STAGE_VECS, 0));  // 0: the row ends in the first stage
        const int st0 = stage;
        const uint32_t ph0 = phase;
        int st1 = st0 + 1;
        uint32_t ph1 = ph0;
        if (st1 == STAGES) {
          st1 = 0;
          ph1 ^= 1u;
        }
        uint4 v[2 * UNROLL];
        bulk::mbar_wait(full + st0, ph0);
        const uint4 *buf0 = ring + static_cast<size_t>(st0) * STAGE_VECS;
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
          const int k = tid + u * CONSUMERS;
          v[u] = (k < n0) ? buf0[k] : bulk::neg_inf_vec<T>();
        }
        if (n1 > 0) {
          bulk::mbar_wait(full + st1, ph1);
          const uint4 *buf1 = ring + static_cast<size_t>(st1) * STAGE_VECS;
#pragma unroll
          for (int u = 0; u < UNROLL; ++u) {
            const int k = tid + u * CONSUMERS;
            v[UNROLL + u] = (k < n1) ? buf1[k] : bulk::neg_inf_vec<T>();
          }
        } else {
#pragma unroll
          for (int u = 0; u < UNROLL; ++u) v[UNROLL + u] = bulk::neg_inf_vec<T>();
        }
        // order this warp's generic-proxy reads of the stages before the copy engine's next write to them
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
          bulk::mbar_arrive(done + st0);
          if (n1 > 0) bulk::mbar_arrive(done + st1);
        }
        fold_batch<T, 2 * UNROLL>(v, m, s, L2);
        stage = st1;
        phase = ph1;
        if (n1 > 0 && ++stage == STAGES) {
          stage = 0;
          phase ^= 1u;
        }
      }
    } else {  // logits view and gradient tile disagree on the 16-byte phase of this row: element loops, no staging
      for (int e = tid; e < V; e += CONSUMERS) lse_push(m, s, Traits<T>::to_float(x[e]));
    }
    // merge the partials of the CONSUMERS threads (named barrier 1: the producer warp is not part of it)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float m2 = __shfl_xor_sync(0xffffffffu, m, o);
      const float s2 = __shfl_xor_sync(0xffffffffu, s, o);
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
        const float m2 = __shfl_xor_sync(0xffffffffu, m, o);
        const float s2 = __shfl_xor_sync(0xffffffffu, s, o);
        lse_merge(m, s, m2, s2);
      }
      if (lane == 0) {
        // ---- boundary: log-prob -> d loss / d log-prob of this token ----
        const float logsum = logf(s);
        float lp = (xy - m) - logsum;  // same association as ATen's `x - max - log(sum)`
        if (y < 0) {
          lp = NAN;
          if (p.status) atomicOr(p.status, AA_STATUS_LABEL_OOB);
        }
        store_from_float(p.out, out_idx, p.out_dtype, lp);
        if (p.stat_max) {
          p.stat_max[flat] = m;
          p.stat_logsum[flat] = logsum;
        }
        float obj, g = g_rs;  // cross-entropy: the same -loss_scale / n_valid for every scored row
        if (p.kind == 0) actor_token(round_to(lp, p.out_dtype), old, adv, on, g_rs, p.clip, p.rx, p.rp, obj, g);
        if (p.kind == 2) grpo_token(round_to(lp, p.out_dtype), old, adv, on, g_rs, p.clip, p.rx, obj, g);
        sh_b[0] = m;
        sh_b[1] = logsum;
        sh_b[2] = g;
      }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(CONSUMERS) : "memory");
    if (!on) {  // the producer zero-fills the row (same_phase) ...
      if (!same_phase)
        for (int e = tid; e < V; e += CONSUMERS) g_out[e] = Traits<T>::from_float(0.f);
      continue;
    }
    m = sh_b[0];
    const float logsum = sh_b[1], g = sh_b[2];

    // ---- phase B: g * (onehot - softmax), the row comes from L2 ----
    const float lse = m + logsum;
    const float c_f32 = -lse * kLog2e;
    const float neg_g = FAITHFUL ? -g : -g * ex2_approx(fmaf(-lse, kLog2e, -c_f32));
    const GradConsts gk = make_grad_consts(m, logsum, c_f32, neg_g, p.zero);
    const bool dead = (g == 0.f);  // clipped token: 0 * softmax, written as +0 like K1b's zero rows
    if (!same_phase) {
      for (int e = tid; e < V; e += CONSUMERS)
        g_out[e] = Traits<T>::from_float(
            dead ? 0.f : grad_of<T, FAITHFUL>(Traits<T>::to_float(x[e]), m, logsum, c_f32, neg_g, g, e == y));
      continue;
    }
    if (tid < head)
      g_out[tid] = Traits<T>::from_float(
          dead ? 0.f : grad_of<T, FAITHFUL>(Traits<T>::to_float(x[tid]), m, logsum, c_f32, neg_g, g, tid == y));
    if (tid < V - tail0)
      g_out[tail0 + tid] = Traits<T>::from_float(
          dead ? 0.f
               : grad_of<T, FAITHFUL>(Traits<T>::to_float(x[tail0 + tid]), m, logsum, c_f32, neg_g, g, tail0 + tid == y));
    const int yv = (y >= head && y < tail0) ? (y - head) / E : -1;  // body vector holding the label column
    for (int v0 = 0; v0 < nvec; v0 += STAGE_VECS) {
      const int n = min(STAGE_VECS, nvec - v0);
      const int st = stage;
      bulk::mbar_wait(full + st, phase);
      uint4 *buf = ring + static_cast<size_t>(st) * STAGE_VECS;
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        const int k = tid + u * CONSUMERS;
        if (k < n) {
          if (dead) {
            buf[k] = make_uint4(0, 0, 0, 0);
          } else {
            const uint4 in = buf[k];
            uint4 o = vec_grad_pk<T, FAITHFUL>(in, gk);
            if (v0 + k == yv) patch_label<T, FAITHFUL>(o, in, (y - head) - (v0 + k) * E, m, logsum, c_f32, neg_g, g);
            buf[k] = o;
          }
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the copy engine
      __syncwarp();
      if (lane == 0) bulk::mbar_arrive(done + st);
      if (++stage == STAGES) {
        stage = 0;
        phase ^= 1u;
      }
    }
  }
}

// coeff[0] = -loss_scale / #(labels != ignore_index): the upstream gradient of every scored row of a mean cross-entropy
__global__ void __launch_bounds__(1024) ce_coeff_kernel(const int64_t *__restrict__ labels, int64_t n, int64_t ignore_index,
                                                        float loss_scale, float *__restrict__ coeff) {
  __shared__ float scratch[33];
  float c = 0.f;
  for (int64_t i = threadIdx.x; i < n; i += 1024) c += (__ldg(labels + i) != ignore_index) ? 1.f : 0.f;
  c = block_sum<1024>(c, scratch);
  if (threadIdx.x == 0) coeff[0] = -loss_scale / c;
}

// tile *= scale unless scale == 1 (every thread reads the scalar first: the usual case costs one empty launch)
template <typename T>
__global__ void __launch_bounds__(256) scale_tile_kernel(T *__restrict__ tile, int64_t n, const void *scale, int scale_dtype) {
  const float s = load_as_float(scale, 0, scale_dtype);
  if (s == 1.f) return;
  constexpr int E = Traits<T>::kVec;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  const int64_t t0 = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int mis = static_cast<int>((reinterpret_cast<uintptr_t>(tile) & 15) / sizeof(T));
  const int64_t head = mis ? min(static_cast<int64_t>(E - mis), n) : 0;
  const int64_t nvec = (n - head) / E;
  const int64_t tail0 = head + nvec * E;
  if (t0 < head) tile[t0] = Traits<T>::from_float(Traits<T>::to_float(tile[t0]) * s);
  if (t0 < n - tail0) tile[tail0 + t0] = Traits<T>::from_float(Traits<T>::to_float(tile[tail0 + t0]) * s);
  uint4 *body = reinterpret_cast<uint4 *>(tile + head);
  for (int64_t k = t0; k < nvec; k += stride) {
    uint4 v = body[k];
    if constexpr (sizeof(T) == 4) {
      v.x = __float_as_uint(__uint_as_float(v.x) * s);
      v.y = __float_as_uint(__uint_as_float(v.y) * s);
      v.z = __float_as_uint(__uint_as_float(v.z) * s);
      v.w = __float_as_uint(__uint_as_float(v.w) * s);
    } else {
      uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float lo, hi;
        unpack2<T>(w[i], lo, hi);
        w[i] = pack2<T>(lo * s, hi * s);
      }
      v = make_uint4(w[0], w[1], w[2], w[3]);
    }
    body[k] = v;
  }
}

// ---- host side ----------------------------------------------------------------------------
// Shape of the persistent kernel (experiment switch AA_B200_FUSED_SHAPE, read once).  Measured on the C4 actor tile
// (32 x 513 x 152064 bf16, 8695 scored rows; K1 -> K5 -> K1b: 1.72 ms), zero rows interleaved:
//   6 (default): 992 consumers (31 warps + the producer warp = 1024 threads), 6 x 31 KB stages, lag 4, 1 CTA/SM: 1.41 ms
//                (1.37 ms after call M: ring positions stepped by hand instead of a 64-bit `it % 6`, two stages per
//                fold in phase A, F2FP rounding in phase B),
//                DRAM reads 2.72 GB = the scored rows ONCE (the second pass hits L2), 4.93 GB written
//   1: 512 consumers, 8 x 16 KB, lag 6, 1 CTA/SM: 1.44     4: 992 consumers, 8 x 15.5 KB, lag 6, 1 CTA/SM: 1.47
//   0: 256 consumers, 8 x 8 KB, lag 6, 2 CTAs/SM: 1.59-1.62 (two rows in flight per SM: a third of the second pass
//      misses L2, 3.5-4.1 GB read)     5: 480 consumers, 8 x 7.5 KB, 2 CTAs/SM: 1.61
//   2: 256 consumers, 4 x 8 KB, lag 3, 3 CTAs/SM (K1b's shape): 1.70     3: 256 consumers, 8 x 16 KB, 1 CTA/SM: 1.91
//   7: 736 consumers, 8 x 11.5 KB, 1 CTA/SM: 1.71 (before the interleaving)
// One CTA per SM keeps 148 rows (45 MB) between the two passes; the kernel is bound by the MUFU / conversion pipe and
// instruction issue (two exp per logit + the bf16 pack), not by HBM: ncu shows 47 % XU, IPC 2.5 at the 1.4 GHz the power
// cap leaves.  AA_B200_FUSED_CTAS overrides the CTAs/SM, AA_B200_FUSED_HINT=0 drops the L2 policies (-10 % with two CTAs
// per SM, +-0 with one), AA_B200_FUSED_INTERLEAVE=0 puts the zero rows after the scored rows (1.63 ms for shape 6).
// LOST (profiles/r02_k1f_experiments.txt, call J): phase A straight from global memory as in K1 (LDG.128, no staging) plus
// a dedicated warp writing the zero rows with st.global: 1.59 ms (30 consumer warps per SM do not hide the DRAM latency
// of the LDG pass: IPC 2.0, and a fifth of the second pass misses L2) -- removed from the source.
// ncu --set full of the default shape (profiles/r02_ncu_k1f_summary.md): DRAM 70 %, issue slots 65 % busy, FMA-heavy
// pipe 57 %, XU 48 %; stalls: 21 % not selected, 18 % waiting for a chunk, 12 % math pipe, 10 % MIO.
static int env_int(const char *name, int dflt) {
  const char *v = std::getenv(name);
  return (v && *v) ? std::atoi(v) : dflt;
}

template <typename T, int CONSUMERS, int STAGES, int UNROLL, int LAG>
static int launch_fused_shape(const FusedActorParams &p, int mode, int per_sm, FusedRec *rec, int64_t n_work,
                              cudaStream_t st) {
  constexpr size_t smem = static_cast<size_t>(STAGES + 1) * CONSUMERS * UNROLL * 16 + STAGES * (8 + 8 + 8 + 4) + 16;
  const bool faithful = (mode == AA_MODE_FAITHFUL) && sizeof(T) == 2;
  auto kf = logprob_actor_fused_kernel<T, CONSUMERS, STAGES, UNROLL, LAG, true>;
  auto kn = logprob_actor_fused_kernel<T, CONSUMERS, STAGES, UNROLL, LAG, false>;
  static std::atomic<bool> configured{false};  // the attribute is idempotent: a race sets it twice, harmlessly
  if (!configured.load(std::memory_order_relaxed)) {
    cudaError_t e = cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(kn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) {
      set_error("aa_logprob_actor_fused: cannot reserve %zu B of shared memory: %s", smem, cudaGetErrorString(e));
      return static_cast<int>(e);
    }
    configured.store(true, std::memory_order_relaxed);
  }
  const int resident = resident_ctas(reinterpret_cast<const void *>(faithful ? kf : kn), CONSUMERS + 32, smem);
  if (per_sm > resident) per_sm = resident;
  int64_t grid = static_cast<int64_t>(sm_count()) * per_sm;
  if (grid > n_work) grid = n_work;
  static const int interleave = env_int("AA_B200_FUSED_INTERLEAVE", 1);
  FusedActorParams q = p;
  q.interleave = interleave ? static_cast<int>(grid) : 0;
  const dim3 pgrid((q.seq + 255) / 256, q.map.n_seg);
  fused_actor_prep_kernel<<<pgrid, 256, 0, st>>>(q, rec);
  int rc = check_launch("aa_logprob_actor_fused(prep)");
  if (rc) return rc;
  if (faithful)
    kf<<<static_cast<unsigned>(grid), CONSUMERS + 32, smem, st>>>(q, rec, n_work);
  else
    kn<<<static_cast<unsigned>(grid), CONSUMERS + 32, smem, st>>>(q, rec, n_work);
  return check_launch("aa_logprob_actor_fused");
}

template <typename T>
static int launch_fused(const FusedActorParams &p, int mode, FusedRec *rec, int64_t n_work, cudaStream_t st) {
  static const int shape = env_int("AA_B200_FUSED_SHAPE", 6);
  static const int ctas = env_int("AA_B200_FUSED_CTAS", 0);
  switch (shape) {
    case 0: return launch_fused_shape<T, 256, 8, 2, 6>(p, mode, ctas > 0 ? ctas : 2, rec, n_work, st);
    case 1: return launch_fused_shape<T, 512, 8, 2, 6>(p, mode, ctas > 0 ? ctas : 1, rec, n_work, st);
    case 2: return launch_fused_shape<T, 256, 4, 2, 3>(p, mode, ctas > 0 ? ctas : 3, rec, n_work, st);
    case 3: return launch_fused_shape<T, 256, 8, 4, 6>(p, mode, ctas > 0 ? ctas : 1, rec, n_work, st);
    case 4: return launch_fused_shape<T, 992, 8, 1, 6>(p, mode, ctas > 0 ? ctas : 1, rec, n_work, st);
    case 5: return launch_fused_shape<T, 480, 8, 1, 6>(p, mode, ctas > 0 ? ctas : 2, rec, n_work, st);
    case 7: return launch_fused_shape<T, 736, 8, 1, 6>(p, mode, ctas > 0 ? ctas : 1, rec, n_work, st);
    default: break;
  }
  return launch_fused_shape<T, 992, 6, 2, 4>(p, mode, ctas > 0 ? ctas : 1, rec, n_work, st);
}

static inline bool fdtype_ok(int dt) { return dt == AA_BF16 || dt == AA_F16 || dt == AA_F32; }
static inline int promote_dt(int a, int b) { return (a == b) ? a : AA_F32; }

}  // namespace aa

using namespace aa;

extern "C" int aa_logprob_actor_fused(const void *logits, int logits_dtype, int64_t row_stride, int32_t V,
                                      const int64_t *labels, int32_t n_segments, const int64_t *seg_logit_off,
                                      const int64_t *seg_label_off, const int64_t *seg_out_off, const int64_t *seg_cum,
                                      const int64_t *seg_tile_row, int64_t n_tile_rows, void *log_probs, int lp_dtype,
                                      float *stat_max, float *stat_logsum, const void *old_log_probs, int64_t old_stride,
                                      const void *advantages, int64_t adv_stride, int adv_dtype, const uint8_t *mask,
                                      int64_t mask_stride, int32_t W, float clip_range_ratio, int mode, void *grad_logits,
                                      int64_t grad_row_stride, void *row_scratch, int32_t *status, void *stream) {
  AA_REQUIRE(V > 0 && n_segments > 0 && W > 0 && n_tile_rows > 0 && n_tile_rows % n_segments == 0, AA_ERR_ARG,
             "aa_logprob_actor_fused: bad sizes (the gradient tile holds n_tile_rows / n_segments rows per sample)");
  AA_REQUIRE(logits && labels && seg_logit_off && seg_label_off && seg_out_off && seg_cum && seg_tile_row && log_probs &&
                 old_log_probs && advantages && mask && grad_logits && row_scratch,
             AA_ERR_ARG, "aa_logprob_actor_fused: null pointer");
  AA_REQUIRE((stat_max == nullptr) == (stat_logsum == nullptr), AA_ERR_ARG,
             "aa_logprob_actor_fused: stat_max and stat_logsum go together");
  AA_REQUIRE(fdtype_ok(logits_dtype) && fdtype_ok(lp_dtype) && fdtype_ok(adv_dtype), AA_ERR_DTYPE,
             "aa_logprob_actor_fused: bad dtype");
  AA_REQUIRE(mode == AA_MODE_FAITHFUL || mode == AA_MODE_F32, AA_ERR_ARG, "aa_logprob_actor_fused: bad mode");
  AA_REQUIRE((reinterpret_cast<uintptr_t>(row_scratch) & 15) == 0, AA_ERR_ALIGN,
             "aa_logprob_actor_fused: row_scratch must be 16-byte aligned");
  AA_REQUIRE(n_tile_rows / n_segments < (1ll << 31) && n_tile_rows < (1ll << 31), AA_ERR_ARG,
             "aa_logprob_actor_fused: tile too large");
  const bool f = (mode == AA_MODE_FAITHFUL);
  static const int hint = env_int("AA_B200_FUSED_HINT", 1);
  FusedActorParams p{logits, row_stride, V, labels,
                     RowMap{seg_logit_off, seg_label_off, seg_out_off, seg_cum, n_segments}, seg_tile_row,
                     static_cast<int>(n_tile_rows / n_segments), log_probs, lp_dtype, stat_max, stat_logsum,
                     old_log_probs, old_stride, advantages, adv_stride, adv_dtype, mask, mask_stride, W,
                     clip_range_ratio, f ? lp_dtype : AA_F32, f ? promote_dt(lp_dtype, adv_dtype) : AA_F32,
                     grad_logits, grad_row_stride, status, kLog2e, 0.0f, hint, 0, 0, 0, nullptr, nullptr, nullptr};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  FusedRec *rec = static_cast<FusedRec *>(row_scratch);
  switch (logits_dtype) {
    case AA_BF16: return launch_fused<__nv_bfloat16>(p, mode, rec, n_tile_rows, st);
    case AA_F16: return launch_fused<__half>(p, mode, rec, n_tile_rows, st);
    case AA_F32: return launch_fused<float>(p, mode, rec, n_tile_rows, st);
  }
  return AA_ERR_DTYPE;
}

extern "C" int aa_logprob_ce_fused(const void *logits, int logits_dtype, int64_t row_stride, int32_t V,
                                  const int64_t *labels, int64_t n_labels, int64_t ignore_index, int32_t n_segments,
                                  const int64_t *seg_logit_off, const int64_t *seg_label_off, const int64_t *seg_out_off,
                                  const int64_t *seg_cum, const int64_t *seg_tile_row, int64_t n_tile_rows,
                                  float *log_probs, float loss_scale, void *grad_logits, int64_t grad_row_stride,
                                  void *row_scratch, float *coeff_scratch, int32_t *status, void *stream) {
  AA_REQUIRE(V > 0 && n_segments > 0 && n_labels > 0 && n_tile_rows > 0 && n_tile_rows % n_segments == 0, AA_ERR_ARG,
             "aa_logprob_ce_fused: bad sizes (the gradient tile holds n_tile_rows / n_segments rows per segment)");
  AA_REQUIRE(logits && labels && seg_logit_off && seg_label_off && seg_out_off && seg_cum && seg_tile_row && log_probs &&
                 grad_logits && row_scratch && coeff_scratch,
             AA_ERR_ARG, "aa_logprob_ce_fused: null pointer");
  AA_REQUIRE(fdtype_ok(logits_dtype), AA_ERR_DTYPE, "aa_logprob_ce_fused: bad dtype");
  AA_REQUIRE((reinterpret_cast<uintptr_t>(row_scratch) & 15) == 0, AA_ERR_ALIGN,
             "aa_logprob_ce_fused: row_scratch must be 16-byte aligned");
  AA_REQUIRE(n_tile_rows < (1ll << 31), AA_ERR_ARG, "aa_logprob_ce_fused: tile too large");
  static const int hint = env_int("AA_B200_FUSED_HINT", 1);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ce_coeff_kernel<<<1, 1024, 0, st>>>(labels, n_labels, ignore_index, loss_scale, coeff_scratch);
  int rc = check_launch("aa_logprob_ce_fused(count)");
  if (rc) return rc;
  FusedActorParams p{logits, row_stride, V, labels,
                     RowMap{seg_logit_off, seg_label_off, seg_out_off, seg_cum, n_segments}, seg_tile_row,
                     static_cast<int>(n_tile_rows / n_segments), log_probs, AA_F32, nullptr, nullptr,
                     nullptr, 0, nullptr, 0, AA_F32, nullptr, 0, 0, 0.f, AA_F32, AA_F32,
                     grad_logits, grad_row_stride, status, kLog2e, 0.0f, hint, 0, 1, ignore_index, coeff_scratch, nullptr, nullptr};
  FusedRec *rec = static_cast<FusedRec *>(row_scratch);
  switch (logits_dtype) {
    case AA_BF16: return launch_fused<__nv_bfloat16>(p, AA_MODE_F32, rec, n_tile_rows, st);
    case AA_F16: return launch_fused<__half>(p, AA_MODE_F32, rec, n_tile_rows, st);
    case AA_F32: return launch_fused<float>(p, AA_MODE_F32, rec, n_tile_rows, st);
  }
  return AA_ERR_DTYPE;
}

extern "C" int aa_logprob_grpo_fused(const void *logits, int logits_dtype, int64_t row_stride, int32_t V,
                                    const int64_t *labels, int32_t n_segments, const int64_t *seg_logit_off,
                                    const int64_t *seg_label_off, const int64_t *seg_out_off, const int64_t *seg_cum,
                                    const int64_t *seg_tile_row, int64_t n_tile_rows, void *log_probs, int lp_dtype,
                                    const void *ref_log_probs, int64_t ref_stride, const float *advantages,
                                    const int64_t *completion_tokens, int64_t tok_stride, int64_t eos_id, int32_t K,
                                    float beta, int mode, void *grad_logits, int64_t grad_row_stride, void *row_scratch,
                                    int32_t *row_end, float *total, uint32_t *counter, int32_t *status, void *stream) {
  AA_REQUIRE(V > 0 && n_segments > 0 && K > 0 && n_tile_rows > 0 && n_tile_rows % n_segments == 0, AA_ERR_ARG,
             "aa_logprob_grpo_fused: bad sizes (the gradient tile holds n_tile_rows / n_segments rows per sample)");
  AA_REQUIRE(logits && labels && seg_logit_off && seg_label_off && seg_out_off && seg_cum && seg_tile_row && log_probs &&
                 ref_log_probs && advantages && completion_tokens && grad_logits && row_scratch && row_end && total && counter,
             AA_ERR_ARG, "aa_logprob_grpo_fused: null pointer");
  AA_REQUIRE(fdtype_ok(logits_dtype) && fdtype_ok(lp_dtype), AA_ERR_DTYPE, "aa_logprob_grpo_fused: bad dtype");
  AA_REQUIRE(mode == AA_MODE_FAITHFUL || mode == AA_MODE_F32, AA_ERR_ARG, "aa_logprob_grpo_fused: bad mode");
  AA_REQUIRE((reinterpret_cast<uintptr_t>(row_scratch) & 15) == 0, AA_ERR_ALIGN,
             "aa_logprob_grpo_fused: row_scratch must be 16-byte aligned");
  AA_REQUIRE(n_tile_rows < (1ll << 31), AA_ERR_ARG, "aa_logprob_grpo_fused: tile too large");
  const bool f = (mode == AA_MODE_FAITHFUL);
  static const int hint = env_int("AA_B200_FUSED_HINT", 1);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  grpo_mask_kernel<128><<<n_segments, 128, 0, st>>>(completion_tokens, tok_stride, n_segments, K, eos_id, row_end, total, counter);
  int rc = check_launch("aa_logprob_grpo_fused(mask)");
  if (rc) return rc;
  FusedActorParams p{logits, row_stride, V, labels,
                     RowMap{seg_logit_off, seg_label_off, seg_out_off, seg_cum, n_segments}, seg_tile_row,
                     static_cast<int>(n_tile_rows / n_segments), log_probs, lp_dtype, nullptr, nullptr,
                     ref_log_probs, ref_stride, advantages, 0, AA_F32, nullptr, 0, K, beta, f ? lp_dtype : AA_F32,
                     f ? lp_dtype : AA_F32, grad_logits, grad_row_stride, status, kLog2e, 0.0f, hint, 0, 2, 0, nullptr,
                     row_end, total};
  FusedRec *rec = static_cast<FusedRec *>(row_scratch);
  switch (logits_dtype) {
    case AA_BF16: return launch_fused<__nv_bfloat16>(p, mode, rec, n_tile_rows, st);
    case AA_F16: return launch_fused<__half>(p, mode, rec, n_tile_rows, st);
    case AA_F32: return launch_fused<float>(p, mode, rec, n_tile_rows, st);
  }
  return AA_ERR_DTYPE;
}

extern "C" int aa_scale_tile(void *tile, int dtype, int64_t n, const void *scale, int scale_dtype, void *stream) {
  AA_REQUIRE(n >= 0 && fdtype_ok(dtype) && fdtype_ok(scale_dtype), AA_ERR_ARG, "aa_scale_tile: bad arguments");
  if (n == 0) return AA_OK;
  AA_REQUIRE(tile && scale, AA_ERR_ARG, "aa_scale_tile: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const unsigned grid = static_cast<unsigned>(sm_count()) * 8u;
  switch (dtype) {
    case AA_BF16: scale_tile_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(static_cast<__nv_bfloat16 *>(tile), n, scale, scale_dtype); break;
    case AA_F16: scale_tile_kernel<__half><<<grid, 256, 0, st>>>(static_cast<__half *>(tile), n, scale, scale_dtype); break;
    default: scale_tile_kernel<float><<<grid, 256, 0, st>>>(static_cast<float *>(tile), n, scale, scale_dtype);
  }
  return check_launch("aa_scale_tile");
}

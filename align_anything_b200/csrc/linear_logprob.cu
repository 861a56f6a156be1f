// linear_logprob.cu -- K6 (SURVEY.md 8f rank 1): lm_head x log-prob in ONE kernel, no (rows, V) logits tile.
//
//   logp[r] = log_softmax(hidden[r, :] @ weight^T)[label[r]]          hidden (N, H) bf16, weight (V, H) bf16
//
// i.e. `gather_log_probabilities(lm_head(hidden), labels)` (utils/tools.py:402-413 on the output of the
// model's nn.Linear lm_head, callers trainers/text_to_text/dpo.py:128, ppo.py:266-267) for rows that carry no
// gradient (reference model, rollout scoring).  The GEMM runs on the 5th-generation tensor cores:
//
//   warp 0   : TMA producer -- cp.async.bulk.tensor 2-D boxes (64 x 128 of hidden, 64 x 256 of weight, 128-byte
//              swizzle) into a 4-stage shared-memory ring, mbarrier expect_tx / complete_tx
//   warp 1   : allocates 512 TMEM columns, one lane issues tcgen05.mma.cta_group::1.kind::f16
//              (M = 128, N = 256, K = 16, bf16 x bf16 -> fp32 in TMEM); tcgen05.commit frees the ring stage /
//              publishes the accumulator
//   warps 2-5: epilogue, one thread per row: tcgen05.ld 32 columns at a time, round to bf16 (the rounding point
//              of the reference's nn.Linear), online (max, sum-exp) update, label-column pick; the two 256-column
//              accumulators alternate so the epilogue of vocabulary tile j overlaps the MMAs of tile j + 1
//
// One CTA owns 128 rows and sweeps the whole vocabulary, so (max, sum) never leave registers; concurrently
// running CTAs sweep the weight in step, which keeps it L2-resident (1.05 GB is read ~once from HBM).
// Both operands are K-major with 16-byte aligned rows (H * 2 bytes), so TMA applies although V = 128257 is odd:
// the odd leading dimension only ever existed in the logits tile, which is never written here (cuBLAS runs the
// same GEMM at ~150 TFLOP/s because of it, see DESIGN.md section 8).
#include <stdlib.h>

#include <atomic>

#include "umma.cuh"

namespace aa {
namespace k6 {

using namespace umma;  // BM / BN / BK / UMMA_K, mbarrier + TMA + tcgen05 wrappers, descriptors (shared with linear_backward.cu)

constexpr int STAGES = 4;
constexpr int THREADS = 192;  // warp 0 TMA, warp 1 MMA, warps 2..5 epilogue
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /* alignment slack */ + 256 /* barriers */;
constexpr uint32_t kIdesc = instr_desc(0, 0);  // both operands K-major

__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) { return desc_k_major(smem_addr); }
__device__ __forceinline__ void umma_f16(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t accumulate) {
  mma_f16(tmem_c, da, db, kIdesc, accumulate);
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) { mma_commit(bar); }

struct Params {
  const int64_t *labels;
  int64_t n_rows;
  int V, H;
  void *out;
  int out_dtype;
  float *stat_max, *stat_logsum;
  int faithful;  // 0: F32 (no rounding); 1: FAITHFUL (logits and log-softmax rounded to bf16); 2: CE (logits only)
  int32_t *status;
  int v_splits, tiles_per_split;  // blockIdx.y sweeps vocabulary tiles [y * tiles_per_split, ...)
  int rot_groups;                 // CTAs start their sweep (m_tile % rot_groups) * rot_step tiles into the range
  int rot_step;
  int group_tiles, m_tiles;       // linear block id -> (row-tile group, split, row tile in group); see the host code
  float *partial;                 // v_splits > 1: (row, split) -> {max, sum, label logit}
};

// Params::faithful of an entry point's `mode`: AA_MODE_CE rounds the logits like nn.Linear's bf16 output but keeps the
// log-softmax (and, in K6b, p) in fp32, so that d(logits) = g * (onehot - p) is rounded once, at the bf16 store -- what
// transformers' ForCausalLMLoss computes on `logits.float()`
inline int rounding(int mode) { return mode == AA_MODE_FAITHFUL ? 1 : mode == AA_MODE_CE ? 2 : 0; }

// d(logits) tile store of K6b: the upstream gradient per row and the padded bf16 buffer
struct GradParams {
  const void *grad_rows;  // upstream d loss / d logp per row
  int grad_rows_dtype;
  __nv_bfloat16 *dlogits; // (n_rows, ld) bf16, ld >= ceil(V / 256) * 256, multiple of 8
  int64_t ld;
  int store_policy;       // 1 = plain 16-byte stores (default); 0 / 2: experiments (AA_K6B_STORE), see the epilogue
};

// K6 (DLOGITS = false) and K6b (DLOGITS = true) are ONE kernel: same TMA producer, same MMA issuer, same two
// alternating TMEM accumulators; they differ in what the four epilogue warps do with a finished 128 x 256 logits tile --
// fold it into the running (max, sum-exp, label logit) of the row, or turn it into d(logits) with the statistics K6
// saved and store it as bf16.
//
// PAIR = true (default since the A/B of round 2: K6 10.2-10.6 ms against 11.6-11.9 ms for single CTAs on 16 376 rows, K6b
// 12.4-12.8 against 13.7-13.9, profiles/r02_k6_pair_ab.txt; AA_B200_K6_PAIR=0 selects single CTAs; launched as clusters
// of 2): the CTA-pair form of the same kernel
// (tcgen05 cta_group::2, see linear_backward.cu): the pair owns 256 rows, each CTA stages its 128 hidden rows and HALF of
// the 256-row weight tile (32 KB per k-block instead of 48 KB -> a 6-deep ring), the leader issues M = 256 MMAs, each
// CTA's epilogue warps consume the 128 x 256 accumulator slice in their own TMEM exactly as before.
template <bool DLOGITS, bool PAIR>
__global__ void __launch_bounds__(THREADS, 1)
    linear_logprob_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                          const Params p, const GradParams gp) {
  constexpr int NST = PAIR ? 6 : STAGES;
  constexpr int SB = PAIR ? (A_BYTES + B_BYTES / 2) : STAGE_BYTES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t *tiles = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t *full = reinterpret_cast<uint64_t *>(tiles + NST * SB);
  uint64_t *empty = full + NST;
  uint64_t *acc_full = empty + NST;   // [2]
  uint64_t *acc_empty = acc_full + 2;    // [2]
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(acc_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // block id -> (group of `group_tiles` row tiles) x (vocabulary split) x (row tile in the group): the CTAs that are
  // resident together work on few row tiles (their hidden-state tiles, 1 MB each and re-read for every vocabulary
  // tile, must stay in L2 next to the weight tiles of the moment) and on all splits of those rows
  // PAIR: `unit` counts CTA pairs and p.m_tiles / p.group_tiles count 256-row pair tiles; rank picks the 128-row half
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const bool leader = rank == 0;
  const int unit = PAIR ? static_cast<int>(blockIdx.x) / 2 : static_cast<int>(blockIdx.x);
  const int per_group = p.group_tiles * p.v_splits;
  const int grp = unit / per_group, rem = unit % per_group;
  const int m_unit = grp * p.group_tiles + rem % p.group_tiles;
  const int split = rem / p.group_tiles;
  if (m_unit >= p.m_tiles) return;  // tail of the last group (uniform per CTA / per pair, before any barrier / TMEM use)
  const int m_tile = PAIR ? 2 * m_unit + static_cast<int>(rank) : m_unit;
  const int m0 = m_tile * BM;
  const int all_tiles = (p.V + BN - 1) / BN;
  const int t0 = split * p.tiles_per_split;
  const int n_tiles = min(all_tiles - t0, p.tiles_per_split);  // >= 1 by construction of the grid
  const int k_blocks = p.H / BK;
  // The online softmax is order independent, so every CTA may sweep its vocabulary range from a different start:
  // at any moment `rot_groups` different weight tiles are hot in L2 instead of one that all SMs hammer.
  const int rot = (p.rot_groups > 1) ? static_cast<int>((m_unit % p.rot_groups) * p.rot_step) % n_tiles : 0;

  if (threadIdx.x == 0) {
    for (int i = 0; i < NST; ++i) {
      mbar_init(full + i, 1);
      mbar_init(empty + i, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(acc_full + i, 1);
      mbar_init(acc_empty + i, PAIR ? 256 : 128);  // PAIR: the leader's barrier collects both CTAs' epilogue threads
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {  // whole warp: allocate all 512 TMEM columns (two 256-column accumulators)
    if (PAIR) tmem_alloc_512_pair(tmem_slot); else tmem_alloc_512(tmem_slot);
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------- TMA producer -------------------------------
    if (lane == 0) {
      int64_t it = 0;
      for (int nt = 0; nt < n_tiles; ++nt) {
        for (int kb = 0; kb < k_blocks; ++kb, ++it) {
          const int s = static_cast<int>(it % NST);
          const uint32_t ph = static_cast<uint32_t>((it / NST) & 1);
          mbar_wait(empty + s, ph ^ 1u);
          uint8_t *a = tiles + s * SB, *b = a + A_BYTES;
          const int v_row0 = (t0 + (nt + rot) % n_tiles) * BN;
          if (PAIR) {  // both CTAs' bytes are credited to the LEADER's full barrier; map_b has 128-row boxes
            if (leader) mbar_expect_tx(full + s, 2 * SB);
            const uint32_t bar = mapa_u32(full + s, 0);
            tma_load_2d_pair(a, &map_a, kb * BK, m0, bar);
            tma_load_2d_pair(b, &map_b, kb * BK, v_row0 + static_cast<int>(rank) * (BN / 2), bar);
          } else {
            mbar_expect_tx(full + s, STAGE_BYTES);
            tma_load_2d(a, &map_a, kb * BK, m0, full + s);
            tma_load_2d(b, &map_b, kb * BK, v_row0, full + s);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------- MMA issuer (PAIR: the leader CTA only) ------
    if (lane == 0 && leader) {
      int64_t it = 0;
      for (int nt = 0; nt < n_tiles; ++nt) {
        const int acc = nt & 1;
        const uint32_t aph = static_cast<uint32_t>((nt >> 1) & 1);
        mbar_wait(acc_empty + acc, aph ^ 1u);  // the epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t tmem_c = tmem_base + static_cast<uint32_t>(acc * BN);
        for (int kb = 0; kb < k_blocks; ++kb, ++it) {
          const int s = static_cast<int>(it % NST);
          const uint32_t ph = static_cast<uint32_t>((it / NST) & 1);
          mbar_wait(full + s, ph);
          tc_fence_after();
          const uint32_t a = smem_u32(tiles + s * SB), b = a + A_BYTES;
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            if (PAIR)
              mma_f16_pair(tmem_c, umma_desc(a + k * UMMA_K * 2), umma_desc(b + k * UMMA_K * 2), instr_desc_pair(0, 0),
                           (kb | k) != 0 ? 1u : 0u);
            else
              umma_f16(tmem_c, umma_desc(a + k * UMMA_K * 2), umma_desc(b + k * UMMA_K * 2), (kb | k) != 0 ? 1u : 0u);
          }
          if (PAIR) mma_commit_pair(empty + s); else umma_commit(empty + s);  // frees the ring stage (in both CTAs)
        }
        if (PAIR) mma_commit_pair(acc_full + acc); else umma_commit(acc_full + acc);  // accumulator complete
      }
    }
  } else if constexpr (!DLOGITS) {
    // ------------------------------- K6 epilogue: one thread per row, online log-sum-exp ----------------
    const int q = warp & 3;  // TMEM lane quadrant this warp may read
    const int row_in_tile = q * 32 + lane;
    const int64_t row = static_cast<int64_t>(m0) + row_in_tile;
    const bool live = row < p.n_rows;
    const int64_t label = live ? __ldg(p.labels + row) : -1;
    if (live && (label < 0 || label >= p.V) && p.status) atomicOr(p.status, AA_STATUS_LABEL_OOB);
    float m = -INFINITY, s = 0.f, x_label = -INFINITY;
    for (int nt = 0; nt < n_tiles; ++nt) {
      const int acc = nt & 1;
      const uint32_t aph = static_cast<uint32_t>((nt >> 1) & 1);
      mbar_wait(acc_full + acc, aph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(acc * BN);
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        uint32_t v[32];
        tmem_ld32(taddr + static_cast<uint32_t>(c * 32), v);
        const int col0 = (t0 + (nt + rot) % n_tiles) * BN + c * 32;
        float x[32];
        float cmax = -INFINITY;
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          float f0 = __uint_as_float(v[j]), f1 = __uint_as_float(v[j + 1]);
          if (p.faithful) round_bf16_pair(f0, f1);  // nn.Linear returns bf16
          if (col0 + j >= p.V) f0 = -INFINITY;      // vocabulary tail (TMA zero-filled the rows)
          if (col0 + j + 1 >= p.V) f1 = -INFINITY;
          x[j] = f0;
          x[j + 1] = f1;
          cmax = fmaxf(cmax, fmaxf(f0, f1));
        }
        const int rel = static_cast<int>(label - col0);
        if (rel >= 0 && rel < 32) {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (j == rel) x_label = x[j];
        }
        if (cmax > m) {  // m == -inf implies s == 0
          s *= ex2_approx((m - cmax) * kLog2e);
          m = cmax;
        }
        float add = 0.f;
#pragma unroll
        for (int j = 0; j < 32; ++j) add += ex2_approx((x[j] - m) * kLog2e);
        s += add;
      }
      tc_fence_before();
      if (PAIR && !leader) mbar_arrive_cluster(mapa_u32(acc_empty + acc, 0)); else mbar_arrive(acc_empty + acc);
    }
    if (live && p.v_splits > 1) {
      float *dst = p.partial + (row * p.v_splits + split) * 3;
      dst[0] = m;
      dst[1] = s;
      dst[2] = x_label;
    } else if (live) {
      const float logsum = logf(s);
      float lp = (x_label - m) - logsum;
      if (label < 0 || label >= p.V) lp = __int_as_float(0x7fc00000);
      if (p.faithful == 1) lp = __bfloat162float(__float2bfloat16_rn(lp));
      store_from_float(p.out, row, p.out_dtype, lp);
      if (p.stat_max) p.stat_max[row] = m;
      if (p.stat_logsum) p.stat_logsum[row] = logsum;
    }
  } else {
    // ------------------------------- K6b epilogue: one thread per row, d(logits) tile store ----------------
    // d(logits)[row, col] = g * ([col == label] - p),  p = exp(round_bf16((x - max) - logsum)) in FAITHFUL mode
    // (what ATen's backward sees: it re-reads the rounded log-softmax), written as bf16 into the padded buffer
    const int q = warp & 3;
    const int row_in_tile = q * 32 + lane;
    const int64_t row = static_cast<int64_t>(m0) + row_in_tile;
    const bool live = row < p.n_rows;
    const int64_t label = live ? __ldg(p.labels + row) : -1;
    const float m = live ? __ldg(p.stat_max + row) : 0.f;
    const float logsum = live ? __ldg(p.stat_logsum + row) : 0.f;
    const float g = live ? load_as_float(gp.grad_rows, row, gp.grad_rows_dtype) : 0.f;
    const float neg_g = -g;
    __nv_bfloat16 *drow = gp.dlogits + row * gp.ld;
    for (int nt = 0; nt < n_tiles; ++nt) {
      const int acc = nt & 1;
      const uint32_t aph = static_cast<uint32_t>((nt >> 1) & 1);
      mbar_wait(acc_full + acc, aph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(acc * BN);
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        uint32_t v[32];
        tmem_ld32(taddr + static_cast<uint32_t>(c * 32), v);
        const int col0 = (t0 + (nt + rot) % n_tiles) * BN + c * 32;
        const int64_t rel64 = label - col0;  // label column inside this chunk, or out of [0, 32)
        const int rel = (rel64 >= 0 && rel64 < 32) ? static_cast<int>(rel64) : -1;
        const int vlim = p.V - col0;         // columns >= vlim are padding
        float d[32];
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          float xs[2] = {__uint_as_float(v[j]), __uint_as_float(v[j + 1])};
          if (p.faithful) round_bf16_pair(xs[0], xs[1]);
          float ls[2] = {(xs[0] - m) - logsum, (xs[1] - m) - logsum};
          if (p.faithful == 1) round_bf16_pair(ls[0], ls[1]);
          d[j] = ex2_approx(ls[0] * kLog2e) * neg_g;  // -(p * g), every column but the label's
          d[j + 1] = ex2_approx(ls[1] * kLog2e) * neg_g;
        }
        if (rel >= 0) {  // this row's label column is in the chunk (1 row in ~4000): g - p * g, the same two roundings
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (j == rel) d[j] = __fadd_rn(d[j], g);
        }
        if (vlim < 32) {  // last vocabulary tile: pad columns of the buffer stay zero
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (j >= vlim) d[j] = 0.f;
        }
        uint32_t o[16];
#pragma unroll
        for (int j = 0; j < 32; j += 2) o[j / 2] = pack2<__nv_bfloat16>(d[j], d[j + 1]);
        if (live && gp.store_policy == 1) {
          uint4 *dst = reinterpret_cast<uint4 *>(drow + col0);  // ld and col0 are multiples of 8 elements: 16-byte aligned
          dst[0] = make_uint4(o[0], o[1], o[2], o[3]);
          dst[1] = make_uint4(o[4], o[5], o[6], o[7]);
          dst[2] = make_uint4(o[8], o[9], o[10], o[11]);
          dst[3] = make_uint4(o[12], o[13], o[14], o[15]);
        } else if (live && gp.store_policy == 2) {  // experiment: streaming (evict-first) stores
          uint4 *dst = reinterpret_cast<uint4 *>(drow + col0);
          __stcs(dst + 0, make_uint4(o[0], o[1], o[2], o[3]));
          __stcs(dst + 1, make_uint4(o[4], o[5], o[6], o[7]));
          __stcs(dst + 2, make_uint4(o[8], o[9], o[10], o[11]));
          __stcs(dst + 3, make_uint4(o[12], o[13], o[14], o[15]));
        } else if (live && o[0] == 0x12345678u && o[15] == 0x9abcdef0u) {  // experiment 0: no stores (keeps the math alive)
          *reinterpret_cast<uint4 *>(drow + col0) = make_uint4(o[0], o[1], o[2], o[3]);
        }
      }
      tc_fence_before();
      if (PAIR && !leader) mbar_arrive_cluster(mapa_u32(acc_empty + acc, 0)); else mbar_arrive(acc_empty + acc);
    }
  }

  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();
  if (warp == 1) {
    if (PAIR) tmem_dealloc_512_pair(tmem_base); else tmem_dealloc_512(tmem_base);
  }
}

// v_splits > 1: merge the per-split (max, sum, label logit) of each row
__global__ void linear_logprob_merge_kernel(const Params p) {
  const int64_t row = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (row >= p.n_rows) return;
  const float *src = p.partial + row * p.v_splits * 3;
  float m = -INFINITY, x_label = -INFINITY;
  for (int i = 0; i < p.v_splits; ++i) {
    m = fmaxf(m, src[3 * i]);
    x_label = fmaxf(x_label, src[3 * i + 2]);  // exactly one split holds the label column
  }
  float s = 0.f;
  for (int i = 0; i < p.v_splits; ++i) s += src[3 * i + 1] * ex2_approx((src[3 * i] - m) * kLog2e);
  const int64_t label = __ldg(p.labels + row);
  const float logsum = logf(s);
  float lp = (x_label - m) - logsum;
  if (label < 0 || label >= p.V) lp = __int_as_float(0x7fc00000);
  if (p.faithful == 1) lp = __bfloat162float(__float2bfloat16_rn(lp));
  store_from_float(p.out, row, p.out_dtype, lp);
  if (p.stat_max) p.stat_max[row] = m;
  if (p.stat_logsum) p.stat_logsum[row] = logsum;
}

// (rows, H) bf16 row-major -> boxes of 64 (K) x box_rows, 128-byte swizzle, out-of-range rows read as zero
static int make_map(CUtensorMap *map, const void *base, int64_t rows, int H, int64_t row_stride, int box_rows) {
  return make_map_2d(map, base, H, rows, row_stride, box_rows, "aa_linear_logprob_fwd");
}

// ---- host: scheduling and launch shared by K6 / K6b, single-CTA and CTA-pair forms ----------------------------------
// One unit (a CTA, or a CTA pair in the PAIR form) owns 128 (256) rows x a range of vocabulary tiles and keeps (max,
// sum) in registers.  The L2 working set decides the speed (ncu, 128 row tiles resident at once: 67 GB of DRAM reads
// for 1.2 GB of operands, L2 hit rate 42% -- the 1 MB hidden-state tile of every resident CTA is re-read for each
// vocabulary tile, 128 of them plus the weight tiles do not fit the 126 MB L2).  So the resident wave is shaped as
// `group` row units x `splits` vocabulary ranges: with S resident units (148 CTAs / 74 pairs) S/8 .. S/4 row units keep
// 18-37 MB of hidden tiles hot and each weight tile is shared by as many units; with fewer row units than S/8 the
// vocabulary is spread over the idle SMs.  Measured on B200 (tools/debug/k6_sweep.py, H = 4096, V = 128257, single
// CTAs): 128 row tiles: 1 split 1124, 18 x 8 1469 TFLOP/s; 1024 row tiles: 1 split 1029, 37 x 4 1204, 37 x 8 1381.
struct Schedule {
  int64_t splits, group, n_groups, units;
  int tps;
};
struct Env {  // scheduling overrides for sweeps, read ONCE per process (thread-safe magic static)
  int min_splits, rot, rot_step, group, pair, store;
  Env() {
    const char *e1 = getenv("AA_K6_MIN_SPLITS"), *e2 = getenv("AA_K6_ROT"), *e3 = getenv("AA_K6_ROT_STEP"),
               *e4 = getenv("AA_K6_GROUP"), *e5 = getenv("AA_B200_K6_PAIR"), *e6 = getenv("AA_K6B_STORE");
    store = e6 ? atoi(e6) : 1;
    min_splits = e1 ? atoi(e1) : 0;
    rot = e2 ? atoi(e2) : 1;
    rot_step = e3 ? atoi(e3) : 1;
    group = e4 ? atoi(e4) : 0;
    pair = e5 ? atoi(e5) : 1;
  }
};
static const Env &env() {
  static const Env e;
  return e;
}
static Schedule make_schedule(int64_t n_rows, int V, bool pair, bool may_split, int64_t partial_floats) {
  const int rows_per_unit = pair ? 2 * BM : BM;
  const int S = pair ? sm_count() / 2 : sm_count();
  Schedule sc;
  sc.units = (n_rows + rows_per_unit - 1) / rows_per_unit;
  const int all_tiles = (V + BN - 1) / BN;
  sc.splits = 1;
  sc.group = sc.units;
  if (may_split) {
    if (sc.units < S / 8) {
      sc.splits = S / sc.units;
    } else {
      // Every live unit does the same work (tiles-per-split vocabulary tiles), so the kernel takes
      // ceil(units * splits / S) rounds of `tps` tiles: pick the split count around 8 that wastes the least of the
      // last round (ncu r02, 8320 rows x 8 splits = 520 units on 148 SMs: 3.51 rounds run as 4, SMs active 86%,
      // tensor pipe 74% of elapsed against 93% for the 1024-unit forward).
      int64_t best = 8, best_cost = INT64_MAX;
      for (int64_t s = 6; s <= 12; ++s) {
        const int64_t tps = (all_tiles + s - 1) / s;
        const int64_t live = sc.units * ((all_tiles + tps - 1) / tps);
        const int64_t cost = ((live + S - 1) / S) * tps * 64 + (s > 8 ? s - 8 : 8 - s);  // rounds x tiles, ties -> 8
        if (cost < best_cost) best_cost = cost, best = s;
      }
      sc.splits = best;
      sc.group = (sc.units >= S) ? S / 4 : S / 8;
      if (sc.units < S) sc.group = S / sc.splits;
    }
    if (env().min_splits > 0) sc.splits = env().min_splits;
    if (env().group > 0) sc.group = env().group;
    if (sc.splits > all_tiles) sc.splits = all_tiles;
    if (sc.splits < 1) sc.splits = 1;
    while (partial_floats >= 0 && sc.splits > 1 && n_rows * sc.splits * 3 > partial_floats) --sc.splits;
    if (sc.group > sc.units) sc.group = sc.units;
    if (sc.group < 1) sc.group = 1;
  }
  sc.tps = static_cast<int>((all_tiles + sc.splits - 1) / sc.splits);
  sc.splits = (all_tiles + sc.tps - 1) / sc.tps;  // no empty split
  sc.n_groups = (sc.units + sc.group - 1) / sc.group;
  return sc;
}

template <bool DLOGITS>
static int launch(const void *hidden, int64_t n_rows, int H, int64_t hidden_row_stride, const void *weight, int V,
                  int64_t weight_row_stride, Params p, const GradParams &gp, const Schedule &sc, bool pair, cudaStream_t st,
                  const char *who) {
  CUtensorMap map_a, map_b;
  int rc = make_map(&map_a, hidden, n_rows, H, hidden_row_stride, BM);
  if (rc) return rc;
  rc = make_map(&map_b, weight, V, H, weight_row_stride, pair ? BN / 2 : BN);  // PAIR: each CTA stages half of the tile
  if (rc) return rc;
  p.v_splits = static_cast<int>(sc.splits);
  p.tiles_per_split = sc.tps;
  p.group_tiles = static_cast<int>(sc.group);
  p.m_tiles = static_cast<int>(sc.units);
  const unsigned units = static_cast<unsigned>(sc.n_groups * sc.group * sc.splits);
  if (!pair) {
    auto kern = linear_logprob_kernel<DLOGITS, false>;
    static std::atomic<bool> configured{false};  // once per process (idempotent; a race sets it twice, harmlessly)
    if (!configured.load(std::memory_order_relaxed)) {
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
      if (e != cudaSuccess) {
        set_error("%s: %s", who, cudaGetErrorString(e));
        return static_cast<int>(e);
      }
      configured.store(true, std::memory_order_relaxed);
    }
    kern<<<units, THREADS, SMEM_BYTES, st>>>(map_a, map_b, p, gp);
    return check_launch(who);
  }
  auto kern = linear_logprob_kernel<DLOGITS, true>;
  constexpr int kPairSmem = 6 * (A_BYTES + B_BYTES / 2) + 1024 + 256;
  static std::atomic<bool> configured_pair{false};
  if (!configured_pair.load(std::memory_order_relaxed)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kPairSmem);
    if (e != cudaSuccess) {
      set_error("%s(pair): %s", who, cudaGetErrorString(e));
      return static_cast<int>(e);
    }
    configured_pair.store(true, std::memory_order_relaxed);
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * units);
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = kPairSmem;
  cfg.stream = st;
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.x = 2;
  attr.val.clusterDim.y = 1;
  attr.val.clusterDim.z = 1;
  cfg.attrs = &attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, map_a, map_b, p, gp);
  if (e != cudaSuccess) {
    set_error("%s(pair): %s", who, cudaGetErrorString(e));
    return static_cast<int>(e);
  }
  return check_launch(who);
}

}  // namespace k6
}  // namespace aa

using namespace aa;

extern "C" int aa_linear_logprob_fwd(const void *hidden, int64_t n_rows, int32_t H, int64_t hidden_row_stride,
                                     const void *weight, int32_t V, int64_t weight_row_stride, const int64_t *labels,
                                     void *out, int out_dtype, float *stat_max, float *stat_logsum, float *partial,
                                     int64_t partial_floats, int mode, int32_t *status, void *stream) {
  AA_REQUIRE(n_rows >= 0 && H > 0 && V > 0, AA_ERR_ARG, "aa_linear_logprob_fwd: bad sizes");
  if (n_rows == 0) return AA_OK;
  AA_REQUIRE(hidden && weight && labels && out, AA_ERR_ARG, "aa_linear_logprob_fwd: null pointer");
  AA_REQUIRE(H % k6::BK == 0, AA_ERR_UNSUPPORTED, "aa_linear_logprob_fwd: H=%d must be a multiple of %d", H, k6::BK);
  AA_REQUIRE((reinterpret_cast<uintptr_t>(hidden) & 15) == 0 && (reinterpret_cast<uintptr_t>(weight) & 15) == 0 &&
                 hidden_row_stride % 8 == 0 && weight_row_stride % 8 == 0 && hidden_row_stride >= H && weight_row_stride >= H,
             AA_ERR_ALIGN, "aa_linear_logprob_fwd: operands must be 16-byte aligned with 16-byte row strides");
  AA_REQUIRE(out_dtype == AA_BF16 || out_dtype == AA_F32, AA_ERR_DTYPE, "aa_linear_logprob_fwd: out must be bf16 or f32");
  AA_REQUIRE(mode == AA_MODE_FAITHFUL || mode == AA_MODE_F32 || mode == AA_MODE_CE, AA_ERR_ARG, "aa_linear_logprob_fwd: bad mode");
  AA_REQUIRE(n_rows < (int64_t(1) << 31) - k6::BM, AA_ERR_UNSUPPORTED, "aa_linear_logprob_fwd: too many rows");
  const bool pair = k6::env().pair > 0;
  const k6::Schedule sc = k6::make_schedule(n_rows, V, pair, partial != nullptr, partial_floats);
  k6::Params p{labels, n_rows, V, H, out, out_dtype, stat_max, stat_logsum, k6::rounding(mode), status,
               1, 1, k6::env().rot, k6::env().rot_step, 1, 1, partial};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = k6::launch<false>(hidden, n_rows, H, hidden_row_stride, weight, V, weight_row_stride, p,
                             k6::GradParams{nullptr, AA_F32, nullptr, 0, 1}, sc, pair, st, "aa_linear_logprob_fwd");
  p.v_splits = static_cast<int>(sc.splits);  // the merge kernel reads the split count
  const int64_t splits = sc.splits;
  if (rc || splits == 1) return rc;
  k6::linear_logprob_merge_kernel<<<static_cast<unsigned>((n_rows + 255) / 256), 256, 0, st>>>(p);
  return check_launch("aa_linear_logprob_fwd(merge)");
}


extern "C" int aa_linear_dlogits(const void *hidden, int64_t n_rows, int32_t H, int64_t hidden_row_stride,
                                 const void *weight, int32_t V, int64_t weight_row_stride, const int64_t *labels,
                                 const float *stat_max, const float *stat_logsum, const void *grad_rows,
                                 int grad_rows_dtype, void *dlogits, int64_t ld, int mode, void *stream) {
  AA_REQUIRE(n_rows >= 0 && H > 0 && V > 0, AA_ERR_ARG, "aa_linear_dlogits: bad sizes");
  if (n_rows == 0) return AA_OK;
  AA_REQUIRE(hidden && weight && labels && stat_max && stat_logsum && grad_rows && dlogits, AA_ERR_ARG,
             "aa_linear_dlogits: null pointer");
  AA_REQUIRE(H % k6::BK == 0, AA_ERR_UNSUPPORTED, "aa_linear_dlogits: H=%d must be a multiple of %d", H, k6::BK);
  const int all_tiles = (V + k6::BN - 1) / k6::BN;
  AA_REQUIRE(ld >= static_cast<int64_t>(all_tiles) * k6::BN && ld % 8 == 0 && (reinterpret_cast<uintptr_t>(dlogits) & 15) == 0,
             AA_ERR_ALIGN, "aa_linear_dlogits: ld must be >= ceil(V / 256) * 256, a multiple of 8, buffer 16-byte aligned");
  AA_REQUIRE((reinterpret_cast<uintptr_t>(hidden) & 15) == 0 && (reinterpret_cast<uintptr_t>(weight) & 15) == 0 &&
                 hidden_row_stride % 8 == 0 && weight_row_stride % 8 == 0 && hidden_row_stride >= H && weight_row_stride >= H,
             AA_ERR_ALIGN, "aa_linear_dlogits: operands must be 16-byte aligned with 16-byte row strides");
  AA_REQUIRE(grad_rows_dtype == AA_BF16 || grad_rows_dtype == AA_F16 || grad_rows_dtype == AA_F32, AA_ERR_DTYPE,
             "aa_linear_dlogits: bad grad dtype");
  AA_REQUIRE(mode == AA_MODE_FAITHFUL || mode == AA_MODE_F32 || mode == AA_MODE_CE, AA_ERR_ARG, "aa_linear_dlogits: bad mode");
  AA_REQUIRE(n_rows < (int64_t(1) << 31) - k6::BM, AA_ERR_UNSUPPORTED, "aa_linear_dlogits: too many rows");
  const bool pair = k6::env().pair > 0;
  const k6::Schedule sc = k6::make_schedule(n_rows, V, pair, true, -1);
  k6::Params p{labels, n_rows, V, H, nullptr, AA_BF16, const_cast<float *>(stat_max), const_cast<float *>(stat_logsum),
               k6::rounding(mode), nullptr, 1, 1, 1, 1, 1, 1, nullptr};
  k6::GradParams gp{grad_rows, grad_rows_dtype, static_cast<__nv_bfloat16 *>(dlogits), ld, k6::env().store};
  return k6::launch<true>(hidden, n_rows, H, hidden_row_stride, weight, V, weight_row_stride, p, gp, sc, pair,
                          static_cast<cudaStream_t>(stream), "aa_linear_dlogits");
}

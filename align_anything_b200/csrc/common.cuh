// common.cuh -- shared device helpers for libaa_b200 (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/aa_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libaa_b200 is written for sm_100a (B200) only"
#endif

namespace aa {

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;
constexpr int kWarp = 32;

// ---- host-side error plumbing (capi.cu) ------------------------------------------------
void set_error(const char *fmt, ...);
int check_launch(const char *what);  // cudaGetLastError -> 0 or positive code (+ message)
int sm_count();
// CTAs of `kernel` that fit on one SM at `threads` threads and `smem` bytes of dynamic shared memory on the current
// device (cudaOccupancyMaxActiveBlocksPerMultiprocessor, queried once per kernel, shape and device).  Persistent
// kernels size their grid with it: a CTA beyond it waits for a resident one to retire and runs in a thinner second
// wave.
int resident_ctas(const void *kernel, int threads, size_t smem);

#define AA_REQUIRE(cond, code, ...)     \
  do {                                  \
    if (!(cond)) {                      \
      ::aa::set_error(__VA_ARGS__);     \
      return (code);                    \
    }                                   \
  } while (0)

// ---- dtype traits -----------------------------------------------------------------------
template <typename T>
struct Traits;

template <>
struct Traits<__nv_bfloat16> {
  static constexpr int kCode = AA_BF16;
  static constexpr int kVec = 8;  // elements per 16-byte vector
  __device__ static __forceinline__ float to_float(__nv_bfloat16 v) { return __bfloat162float(v); }
  __device__ static __forceinline__ __nv_bfloat16 from_float(float v) { return __float2bfloat16_rn(v); }
  __device__ static __forceinline__ float round(float v) {
    return __bfloat162float(__float2bfloat16_rn(v));
  }
};
template <>
struct Traits<__half> {
  static constexpr int kCode = AA_F16;
  static constexpr int kVec = 8;
  __device__ static __forceinline__ float to_float(__half v) { return __half2float(v); }
  __device__ static __forceinline__ __half from_float(float v) { return __float2half_rn(v); }
  __device__ static __forceinline__ float round(float v) { return __half2float(__float2half_rn(v)); }
};
template <>
struct Traits<float> {
  static constexpr int kCode = AA_F32;
  static constexpr int kVec = 4;
  __device__ static __forceinline__ float to_float(float v) { return v; }
  __device__ static __forceinline__ float from_float(float v) { return v; }
  __device__ static __forceinline__ float round(float v) { return v; }
};

// Round `v` to the precision of dtype code `dt` (bf16 / f16), identity for f32.
__device__ __forceinline__ float round_to(float v, int dt) {
  if (dt == AA_BF16) return __bfloat162float(__float2bfloat16_rn(v));
  if (dt == AA_F16) return __half2float(__float2half_rn(v));
  return v;
}

// Generic typed scalar load / store through a dtype code (cold paths: the PPO scalars).
__device__ __forceinline__ float load_as_float(const void *p, int64_t i, int dt) {
  if (dt == AA_BF16) return __bfloat162float(reinterpret_cast<const __nv_bfloat16 *>(p)[i]);
  if (dt == AA_F16) return __half2float(reinterpret_cast<const __half *>(p)[i]);
  return reinterpret_cast<const float *>(p)[i];
}
__device__ __forceinline__ void store_from_float(void *p, int64_t i, int dt, float v) {
  if (dt == AA_BF16)
    reinterpret_cast<__nv_bfloat16 *>(p)[i] = __float2bfloat16_rn(v);
  else if (dt == AA_F16)
    reinterpret_cast<__half *>(p)[i] = __float2half_rn(v);
  else
    reinterpret_cast<float *>(p)[i] = v;
}
__host__ __device__ __forceinline__ int dtype_size(int dt) { return dt == AA_F32 ? 4 : 2; }

// ---- unpack one 32-bit word holding two 16-bit floats -----------------------------------
template <typename T>
__device__ __forceinline__ void unpack2(uint32_t w, float &lo, float &hi);
template <>
__device__ __forceinline__ void unpack2<__nv_bfloat16>(uint32_t w, float &lo, float &hi) {
  lo = __uint_as_float(w << 16);
  hi = __uint_as_float(w & 0xffff0000u);
}
template <>
__device__ __forceinline__ void unpack2<__half>(uint32_t w, float &lo, float &hi) {
  __half2 h = *reinterpret_cast<__half2 *>(&w);
  float2 f = __half22float2(h);
  lo = f.x;
  hi = f.y;
}
template <typename T>
__device__ __forceinline__ uint32_t pack2(float lo, float hi);
template <>
__device__ __forceinline__ uint32_t pack2<__nv_bfloat16>(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);  // .x = lo (low 16 bits)
  return *reinterpret_cast<uint32_t *>(&h);
}
template <>
__device__ __forceinline__ uint32_t pack2<__half>(float lo, float hi) {
  __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t *>(&h);
}
// round two fp32 values to bf16 (RN-even) and back: ONE F2FP.PACK_AB + two ALU unpacks instead of two F2F on the
// quarter-rate XU pipe that the exp2 of the same epilogue needs
__device__ __forceinline__ void round_bf16_pair(float &a, float &b) {
  unpack2<__nv_bfloat16>(pack2<__nv_bfloat16>(a, b), a, b);
}

// ---- streaming 128-bit global access (read-once / write-once tiles) ---------------------
// load policy (compile-time experiment knob): 0 = nc + L1::no_allocate + L2::256B prefetch (default),
// 1 = same without the 256B prefetch hint, 2 = L2::evict_first, 3 = L1::no_allocate + L2::evict_first + 256B
#ifndef AA_LDG_POLICY
#define AA_LDG_POLICY 0
#endif
__device__ __forceinline__ uint4 ldg_stream(const uint4 *p) {
  uint4 r;
#if AA_LDG_POLICY == 0
  asm("ld.global.nc.L1::no_allocate.L2::256B.v4.u32 {%0,%1,%2,%3}, [%4];"
#elif AA_LDG_POLICY == 1
  asm("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
#elif AA_LDG_POLICY == 2
  asm("ld.global.nc.L1::no_allocate.L2::evict_first.v4.u32 {%0,%1,%2,%3}, [%4];"
#else
  asm("ld.global.nc.L1::no_allocate.L2::evict_first.L2::256B.v4.u32 {%0,%1,%2,%3}, [%4];"
#endif
      : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
      : "l"(p));
  return r;
}
// store policy (compile-time experiment knob, see tools/sweep_k1.py): 0 = .cs (evict-first),
// 1 = default write-back, 2 = .L1::no_allocate, 3 = .wt
#ifndef AA_STG_POLICY
#define AA_STG_POLICY 0
#endif
__device__ __forceinline__ void stg_stream(uint4 *p, const uint4 &v) {
#if AA_STG_POLICY == 0
  asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
#elif AA_STG_POLICY == 1
  asm volatile("st.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
#elif AA_STG_POLICY == 2
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
#else
  asm volatile("st.global.wt.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
#endif
}

__device__ __forceinline__ float ex2_approx(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// ---- packed fp32 pairs (Blackwell f32x2: FADD2 / FMUL2 / FFMA2, one issue slot for two lanes of math) ----
// The log-prob kernels are bound by instruction issue once the SM clock drops under the power cap
// (1.72 GHz sustained vs 1.95 GHz burst), so the per-element fp32 ops are issued two at a time.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 f2_pack(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(f32x2 v, float &lo, float &hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 f2_splat(float v) { return f2_pack(v, v); }
__device__ __forceinline__ f32x2 f2_add(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 f2_sub(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 f2_mul(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 f2_fma(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ f32x2 f2_ex2(f32x2 t) {
  float a, b;
  f2_unpack(t, a, b);
  return f2_pack(ex2_approx(a), ex2_approx(b));
}
// Round both lanes to 8 significant bits (= bf16 round-to-nearest) WITHOUT the conversion unit:
// Veltkamp splitting, hi = c - (c - x) with c = x * (2^16 + 1).  Three FMA-pipe ops per pair instead
// of an F2FP round trip on the XU pipe (which MUFU.EX2 already keeps ~70% busy in the backward).
// Bit-identical to __float2bfloat16_rn for normal numbers (checked on 5M samples); inputs must be
// finite (callers clamp -inf logits to -1e30 first).
// `zero2` must be a RUN-TIME +0.0 pair (kernel parameter): ptxas contracts mul.rn.f32x2 + sub.rn.f32x2
// into FFMA2 (observed with CUDA 12.9: d = fma(x, 65537, -x)), which destroys the split; producing c
// with an FMA whose addend the compiler cannot see through leaves nothing to contract.
__device__ __forceinline__ f32x2 f2_round_bf16(f32x2 x, f32x2 zero2) {
  const f32x2 c = f2_fma(x, f2_splat(65537.f), zero2);
  return f2_sub(c, f2_sub(c, x));
}
// Same for fp16 precision (11 significant bits): c = x * (2^13 + 1); valid inside fp16's normal range.
__device__ __forceinline__ f32x2 f2_round_f16(f32x2 x, f32x2 zero2) {
  const f32x2 c = f2_fma(x, f2_splat(8193.f), zero2);
  return f2_sub(c, f2_sub(c, x));
}

// 2^t on the FMA / ALU pipes (no MUFU): Cody-Waite split t = n + f, f in [-0.5, 0.5], degree-5 minimax
// polynomial with c0 == 1 exactly (so 2^0 == 1 exactly, like MUFU.EX2), exponent patched in with one
// integer add.  Max relative error 1.9e-7 (MUFU.EX2: 2^-22 = 2.4e-7).  An experiment to unload the
// MUFU pipe (16/clk/SM on B200, 73% busy in the forward per ncu); it measured slower (logprob.cu,
// AA_FWD_POLY_WORDS) and is off by default.
__device__ __forceinline__ float ex2_poly(float t) {
  float tc;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(tc) : "f"(t), "f"(-126.f));  // NaN stays NaN
  const float r = tc + 12582912.f;                                    // 1.5 * 2^23: rounds to nearest integer
  const float f = tc - (r - 12582912.f);
  float p = 1.328307088e-03f;
  p = fmaf(p, f, 9.671507403e-03f);
  p = fmaf(p, f, 5.550670624e-02f);
  p = fmaf(p, f, 2.402224243e-01f);
  p = fmaf(p, f, 6.931470037e-01f);
  p = fmaf(p, f, 1.0f);
  return __int_as_float(__float_as_int(p) + (__float_as_int(r) << 23));
}

// Packed version of ex2_poly: two lanes per instruction for the range reduction and the Horner chain.
__device__ __forceinline__ f32x2 f2_ex2_poly(f32x2 t) {
  float ta, tb;
  f2_unpack(t, ta, tb);
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(ta) : "f"(ta), "f"(-126.f));
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(tb) : "f"(tb), "f"(-126.f));
  const f32x2 tc = f2_pack(ta, tb);
  const f32x2 magic = f2_splat(12582912.f);
  const f32x2 r = f2_add(tc, magic);
  const f32x2 f = f2_sub(tc, f2_sub(r, magic));
  f32x2 p = f2_splat(1.328307088e-03f);
  p = f2_fma(p, f, f2_splat(9.671507403e-03f));
  p = f2_fma(p, f, f2_splat(5.550670624e-02f));
  p = f2_fma(p, f, f2_splat(2.402224243e-01f));
  p = f2_fma(p, f, f2_splat(6.931470037e-01f));
  p = f2_fma(p, f, f2_splat(1.0f));
  float pa, pb, ra, rb;
  f2_unpack(p, pa, pb);
  f2_unpack(r, ra, rb);
  return f2_pack(__int_as_float(__float_as_int(pa) + (__float_as_int(ra) << 23)),
                 __int_as_float(__float_as_int(pb) + (__float_as_int(rb) << 23)));
}

// ---- warp / block reductions ------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int warp_max_i(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Deterministic block sum (fixed tree); result valid in every thread.  `scratch` >= 33 floats.
template <int THREADS>
__device__ __forceinline__ float block_sum(float v, float *scratch) {
  constexpr int W = THREADS / kWarp;
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < kWarp) {
    float t = threadIdx.x < W ? scratch[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0) scratch[32] = t;
  }
  __syncthreads();
  float r = scratch[32];
  __syncthreads();
  return r;
}

// Online-softmax partials are kept as (m, s) with s = sum_i 2^((x_i - m)*log2e).  The subtraction is
// done BEFORE the scaling (FADD + FMUL instead of one FFMA): x_i - m is exact for the element that
// attains the maximum, so its term is exactly 1 -- like ATen's exp(x - max) -- and a saturated row
// yields sum == 1.0f and a log-prob of exactly 0, which the multimodal PPO trainer's
// `response_mask = (log_probs != 0)` (trainers/text_image_to_text/ppo.py:250) depends on; it is also
// accurate for logits of any magnitude.
// Invariant: a partial whose max is -inf has s == 0.
__device__ __forceinline__ float lse_rescale(float m_old, float m_new) {
  if (m_old == m_new) return 1.f;
  if (m_old == -INFINITY) return 0.f;  // s == 0 anyway; avoids inf - inf
  return ex2_approx((m_old - m_new) * kLog2e);
}

// Merge two partials.
__device__ __forceinline__ void lse_merge(float &m, float &s, float m2, float s2) {
  const float mn = fmaxf(m, m2);
  s = s * lse_rescale(m, mn) + s2 * lse_rescale(m2, mn);
  m = mn;
}

// Fold one scalar element (the <8-element head / tail of an unaligned row).
__device__ __forceinline__ void lse_push(float &m, float &s, float x) {
  if (x == -INFINITY) return;  // exp(-inf) = 0: keeps the invariant
  lse_merge(m, s, x, 1.f);
}

// largest s in [0, n) with arr[s] <= key (arr ascending, arr[0] <= key)
__device__ __forceinline__ int upper_segment(const int64_t *__restrict__ arr, int n, int64_t key) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    int mid = (lo + hi + 1) >> 1;
    if (__ldg(arr + mid) <= key)
      lo = mid;
    else
      hi = mid - 1;
  }
  return lo;
}

// "last block done" helper: returns true in every thread of the block that arrives last.
// `counter` must be zero before the first launch; the last block re-zeroes it.
__device__ __forceinline__ bool last_block_arrives(uint32_t *counter, uint32_t n_blocks) {
  __shared__ bool is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t prev = atomicAdd(counter, 1u);
    is_last = (prev == n_blocks - 1);
    if (is_last) *counter = 0u;
  }
  __syncthreads();
  if (is_last) __threadfence();
  return is_last;
}

// ---- one-shot all-reduce of a packed metric vector over NVLink peer memory -----------------------------
// Every rank owns one symmetric buffer (torch.distributed._symmetric_memory: peer-mapped over NVLink /
// NVSwitch) laid out as  float slots[2][world][kCollLanes]  followed by  uint32 flags[world].
// A call with epoch e: each rank STORES its n floats into slot [e & 1][rank] of EVERY peer's buffer
// (plain st.global on the peer-mapped pointer = NVLink write), fences system-wide, raises flag[rank] = e on
// every peer, waits until all `world` flags in its OWN buffer have reached e, then reduces the `world`
// slots locally (lanes in max_mask: MAX, others: mean -- the AVG / MAX of utils/multi_process.py:74-89).
// No NCCL launch, no extra kernel: it runs in the tail of the kernel that produced the vector (K2's last
// block, the PPO metric packer).  Double-buffered by epoch parity; epochs increase by 1 per call on
// every rank (same number of steps on every rank, as DistributedSampler guarantees).
constexpr int kCollLanes = 16;
struct CollParams {
  float *const *peer_bufs;  // device array [world] of peer-mapped buffer pointers (this rank's included)
  int rank, world;
  uint32_t epoch;
  uint32_t max_mask;        // bit t set: lane t is reduced with MAX instead of mean
};

__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// Called by ONE block (>= 32 threads), all threads of its first warp; `vals` (local, n <= kCollLanes) in,
// reduced values out through `out`.
__device__ __forceinline__ void p2p_allreduce_packed(const CollParams &c, const float *vals, float *out, int n) {
  const int lane = threadIdx.x;
  if (lane >= kWarp) return;
  const int par = static_cast<int>(c.epoch & 1u);
  const size_t slot_floats = static_cast<size_t>(c.world) * kCollLanes;
  // 1. push my vector to every peer (lane t carries element t)
  if (lane < n) {
    const float v = vals[lane];
    for (int p = 0; p < c.world; ++p)
      c.peer_bufs[p][par * slot_floats + static_cast<size_t>(c.rank) * kCollLanes + lane] = v;
  }
  __threadfence_system();
  __syncwarp();
  // 2. raise my flag on every peer (lane p signals peer p)
  if (lane < c.world) {
    uint32_t *flags = reinterpret_cast<uint32_t *>(c.peer_bufs[lane] + 2 * slot_floats);
    st_release_sys(flags + c.rank, c.epoch);
  }
  // 3. wait for everybody's flag in MY buffer (lane p waits for rank p)
  float *mine = c.peer_bufs[c.rank];
  if (lane < c.world) {
    const uint32_t *flag = reinterpret_cast<const uint32_t *>(mine + 2 * slot_floats) + lane;
    while (static_cast<int32_t>(ld_acquire_sys(flag) - c.epoch) < 0) __nanosleep(64);
  }
  __syncwarp();
  // 4. reduce locally
  if (lane < n) {
    const volatile float *slots = mine + par * slot_floats;
    float acc = slots[lane];
    const bool is_max = (c.max_mask >> lane) & 1u;
    for (int r = 1; r < c.world; ++r) {
      const float v = slots[static_cast<size_t>(r) * kCollLanes + lane];
      acc = is_max ? fmaxf(acc, v) : acc + v;
    }
    out[lane] = is_max ? acc : acc / static_cast<float>(c.world);
  }
}

}  // namespace aa

// Causal flash attention for sm_100a: tcgen05 MMAs with fp32 scores / outputs in tensor memory, TMA loads straight out of
// the packed qkv projection buffer, one query (or key) row per thread so row statistics need no shuffles.
//
// Replaces the reference's F.scaled_dot_product_attention call (peft_pretraining/modeling_llama.py:241-247 and
// modeling_pythia.py attention) for head_dim <= 64.  Three kernels:
//
//   attn_fwd_kernel      CTA = (128 queries, head, batch); per 64 keys:  S = Q·Kᵀ -> online softmax -> O += P·V
//   attn_bwd_dq_kernel   CTA = (128 queries, head, batch); per 64 keys:  S, dP = dO·Vᵀ -> dS -> dQ += dS·K
//   attn_bwd_dkv_kernel  CTA = (128 keys, head, batch); per 64 queries:  Sᵀ = K·Qᵀ, dPᵀ = V·dOᵀ -> Pᵀ, dSᵀ -> dV += Pᵀ·dO, dK += dSᵀ·Q
//
// Roles inside a CTA: warps 0-3 = 128 "row" threads (thread i <-> TMEM lane i), warp 4 lane 0 = TMA + MMA issue.
// Shared-memory tiles are 64 columns (128 bytes) wide with the 128-byte swizzle, so the same [64 x 64] tile serves as a K-major
// operand (reduction over head_dim) and as an MN-major operand (reduction over its rows) by descriptor alone.
#include <cuda.h>

#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <stdexcept>
#include <unordered_map>

#include "attention.h"
#include "common.cuh"
#include "sm100.cuh"
#include "tensormap.h"

namespace rb {

using namespace sm100;

namespace {

constexpr int BQ = 128;  // rows owned by the row threads (queries in fwd / dq, keys in dkv)
constexpr int BK = 64;   // columns per step (keys in fwd / dq, queries in dkv)
constexpr int kTile128 = 128 * 128;  // bytes of a [128 x 64] bf16 tile
constexpr int kTile64 = 64 * 128;    // bytes of a [64 x 64] bf16 tile
// The driver keeps kernels that allocate tensor memory at one resident CTA per SM (occupancy calculator: 1, independent of
// shared memory and registers), so the latency hiding comes from several independent "groups" inside one CTA: each group is
// 4 row warps + 1 control warp working on its own (batch, head, block) item with its own shared-memory region, barriers and
// tensor-memory columns.
#ifndef RB_ATTN_GROUPS_FWD
#define RB_ATTN_GROUPS_FWD 1
#define RB_ATTN_GROUPS_BWD 1
#endif
constexpr int kFwdGroups = RB_ATTN_GROUPS_FWD, kDqGroups = RB_ATTN_GROUPS_BWD, kDkvGroups = RB_ATTN_GROUPS_BWD;  // measured: 3/2/2 groups per CTA 88 / 232 us vs 1 group (several CTAs per SM) 79 / 210 us
constexpr int pow2_cols(int c) { return c <= 32 ? 32 : c <= 64 ? 64 : c <= 128 ? 128 : c <= 256 ? 256 : 512; }
constexpr int kFwdGroupBytes = 2 * kTile128 + 4 * kTile64 + 1024;                  // Q, K/V stages, P, barriers
constexpr int kDqGroupBytes = 3 * kTile128 + 4 * kTile64 + 1024;                   // Q, dO, K/V stages, dS, barriers
constexpr int kDkvGroupBytes = 4 * kTile128 + 4 * kTile64 + 1024 + 1024;           // K, V, Q/dO stages, Pt, dSt, lse/delta, barriers
constexpr float kNegInf = -1e30f;

__device__ __forceinline__ uint64_t desc_k(const uint8_t* tile, int kstep) {  // K-major operand, 16 columns per MMA
  return make_desc_sw128(smem_u32(tile) + kstep * 32, 16, 1024);
}
__device__ __forceinline__ uint64_t desc_mn(const uint8_t* tile, int kstep) {  // MN-major operand, 16 rows per MMA
  return make_desc_sw128(smem_u32(tile) + kstep * 2048, 8192, 1024);
}

#ifndef RB_ATTN_SLEEP_NS
#define RB_ATTN_SLEEP_NS 0
#endif
__device__ __forceinline__ void attn_wait(uint64_t* bar, uint32_t parity) {
  if constexpr (RB_ATTN_SLEEP_NS > 0) mbar_wait_sleep(bar, parity, RB_ATTN_SLEEP_NS);
  else mbar_wait(bar, parity);
}

// The control warp walks its loop with all 32 lanes (uniform control flow: ptxas keeps shared-memory addresses, descriptors and TMEM
// addresses in uniform registers) and ONE elected lane issues the TMA / tcgen05 instructions.  Under an `if (lane == 0)` branch
// every UTMALDG / UTCHMMA is wrapped in an ELECT + R2UR + BRA.U.ANY loop (~17 extra dependent instructions per MMA).
#define RB_ONE_LANE(...)          \
  do {                            \
    if (elect_one()) { __VA_ARGS__ } \
    __syncwarp();                 \
  } while (0)

__device__ __forceinline__ float fast_exp2(float x) {  // one MUFU.EX2, no range fix-up (inputs are <= ~8, -inf -> 0)
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// row `r` of a [128 x 64] bf16 tile (128-byte swizzle): 8 chunks of 8 values
__device__ __forceinline__ void store_row64(uint8_t* tile, int r, const float* v) {
  uint8_t* rowp = tile + r * 128;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    float f[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] = v[q * 8 + i];
    *reinterpret_cast<uint4*>(rowp + ((q ^ (r & 7)) << 4)) = pack8(f);
  }
}

__device__ __forceinline__ void ld64(uint32_t taddr, float* v) {  // 64 fp32 columns of this thread's TMEM lane
  uint32_t a[32], b[32];
  tmem_ld_32x32b_x32(taddr, a);
  tmem_ld_32x32b_x32(taddr + 32, b);
  tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    v[i] = __uint_as_float(a[i]);
    v[32 + i] = __uint_as_float(b[i]);
  }
}

__device__ __forceinline__ void ld32(uint32_t taddr, float* v) {  // 32 fp32 columns of this thread's TMEM lane
  uint32_t a[32];
  tmem_ld_32x32b_x32(taddr, a);
  tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(a[i]);
}
// half `hf` (32 values = 4 chunks of 8) of row `r` of a [128 x 64] bf16 tile (128-byte swizzle)
__device__ __forceinline__ void store_row32(uint8_t* tile, int r, int hf, const float* v) {
  uint8_t* rowp = tile + r * 128;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float f[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] = v[q * 8 + i];
    *reinterpret_cast<uint4*>(rowp + (((hf * 4 + q) ^ (r & 7)) << 4)) = pack8(f);
  }
}
// The backward kernels have no row reductions (lse and delta are inputs), so TWO warps share every row: warp w and w + 4 own
// the same TMEM lanes and split the 64 columns of a step.  Halves the per-thread work of the S / dP -> dS dependency chain
// that bounds these kernels (ncu round 2: 15 % warps active, 60 % of the stall samples waiting on the chain).
constexpr int kBwdRowWarps = 8;

struct FwdArgs {
  long long* trace;  // diagnostics: clock64 stamps of the heaviest CTA (bench/attn_trace.py); normally null
  bf16* out;
  long long ld_out;
  float* lse;
  int B, T, nh, hd;
  float scale_log2;
};

// =============================================================================================== forward
__global__ void __launch_bounds__((4 * kFwdGroups + kFwdGroups) * 32, kFwdGroups == 1 ? 3 : 1) attn_fwd_kernel(const __grid_constant__ CUtensorMap map_qkv, const FwdArgs p) {
  constexpr int NG = kFwdGroups;
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;  // warp index known uniform to ptxas
  if (threadIdx.x == 0) pdl_launch_dependents();
  const bool is_ctrl = warp >= 4 * NG;
  const int g = is_ctrl ? warp - 4 * NG : warp >> 2;  // group of this warp
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem0 = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem = smem0 + g * kFwdGroupBytes;
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + kTile128;      // 2 stages
  uint8_t* sV = sK + 2 * kTile64;   // 2 stages
  uint8_t* sP = sV + 2 * kTile64;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + kTile128);
  uint64_t* q_full = bars;
  uint64_t* kv_full = bars + 1;
  uint64_t* kv_free = bars + 3;
  uint64_t* s_full = bars + 5;
  uint64_t* p_ready = bars + 6;
  uint64_t* o_full = bars + 7;
  uint64_t* s_free = bars + 9;  // (bars + 8 is the tensor-memory slot of group 0)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem0 + 2 * kTile128 + 4 * kTile64 + 64);  // in group 0's barrier page

  // work item of this group: (query block, head, batch), heaviest (latest) query blocks first
  const int nqb = (p.T + BQ - 1) / BQ;
  const long long per = (long long)p.B * p.nh;
  const long long item = (long long)blockIdx.x * NG + g;
  const bool active = item < per * nqb;
  const int qb = active ? nqb - 1 - int(item / per) : 0;
  const int head = int((item % per) % p.nh), b = active ? int((item % per) / p.nh) : 0;
  const int t0 = qb * BQ;
  const int kv_end = min(p.T, t0 + BQ);
  const int n_kv = active ? (kv_end + BK - 1) / BK : 0;
  const int row0 = b * p.T;

  if (is_ctrl && lane == 0) {
    mbar_init(q_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_free[i], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(p_ready, 128);
    mbar_init(o_full, 1);
    mbar_init(s_free, 128);
    fence_barrier_init();
    tma_prefetch_desc(&map_qkv);
  }
  if (warp == 4 * NG) {
    tmem_alloc(tmem_slot, pow2_cols(NG * 128));  // per group: S in columns 0-63, O in columns 64-127
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0) + g * 128;
  pdl_wait();

  if (is_ctrl) {
    if (active) {
      auto load_kv = [&](int jj, int st) {
        RB_ONE_LANE(mbar_arrive_expect_tx(&kv_full[st], 2 * kTile64);
                    tma_load_3d(&map_qkv, &kv_full[st], sK + st * kTile64, 0, p.nh + head, row0 + jj * BK);
                    tma_load_3d(&map_qkv, &kv_full[st], sV + st * kTile64, 0, 2 * p.nh + head, row0 + jj * BK););
      };
      RB_ONE_LANE(mbar_arrive_expect_tx(q_full, kTile128);
                  tma_load_3d(&map_qkv, q_full, sQ, 0, head, row0 + t0);
                  tma_load_3d(&map_qkv, q_full, sQ + kTile64, 0, head, row0 + t0 + 64););
      load_kv(0, 0);
      if (n_kv > 1) load_kv(1, 1);
      constexpr uint32_t idesc_s = make_idesc_bf16(128, 64, 0, 0);
      constexpr uint32_t idesc_pv = make_idesc_bf16(128, 64, 0, 1);
      auto issue_s = [&](int st) {
        RB_ONE_LANE(
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_f16_ss(tmem_base, desc_k(sQ, k), desc_k(sK + st * kTile64, k), idesc_s, k != 0);
            umma_commit(s_full););
      };
      attn_wait(q_full, 0);
      attn_wait(&kv_full[0], 0);
      tc_fence_after();
      issue_s(0);
      for (int jj = 0; jj < n_kv; ++jj) {
        const int st = jj & 1;
        // The scores of the next step are issued as soon as the row threads hold S(jj) in registers (s_free, a few hundred cycles
        // into the step), not when they finish the step: QKᵀ latency and the wake-up of this warp leave the per-step chain
        // (forward 69.6 -> 65.6 us at the 250m shape, 198.7 -> 176.2 us at T = 2048).  The same change in the dK/dV kernel was
        // measured slower (162.8 -> 166.9 us: it needs a second guard on the Pᵀ / dSᵀ tiles) and is not applied there.
        if (jj + 1 < n_kv) {
          attn_wait(s_free, jj & 1);
          attn_wait(&kv_full[st ^ 1], ((jj + 1) >> 1) & 1);
          tc_fence_after();
          issue_s(st ^ 1);
        }
        attn_wait(p_ready, jj & 1);
        tc_fence_after();
        // this step's P·V: its completion (o_full) gates the reuse of P and a rescale of O
        RB_ONE_LANE(
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_f16_ss(tmem_base + 64, desc_k(sP, k), desc_mn(sV + st * kTile64, k), idesc_pv, (jj | k) != 0);  // O accumulates in TMEM
            umma_commit(o_full);
            umma_commit(&kv_free[st]););
        if (jj + 2 < n_kv) {
          attn_wait(&kv_free[st], (jj >> 1) & 1);
          load_kv(jj + 2, st);
        }
      }
    }
  } else {
    const int r = threadIdx.x & 127;
    const int t = t0 + r;
    const uint32_t lane_addr = tmem_addr(tmem_base, (warp & 3) * 32, 0);
    // The output accumulates in tensor memory across key steps.  The running maximum used for the exponentials ("m") is
    // only raised -- and O rescaled by a TMEM load / multiply / store -- when a step's maximum exceeds it by more than
    // 2^8; any reference maximum is mathematically valid as long as exp2 stays in range, and the same m enters l.
    float m = kNegInf, l = 0.f;
    // in-kernel clock64 trace (bench/attn_trace.py): compiled in only with -DRB_ATTN_TRACE -- even predicated off, its five
    // stores + clock reads per step showed up as issue slots and `lg` stalls in the ncu source view of the production build
#ifdef RB_ATTN_TRACE
    const bool tr = p.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0;
#define ATR(slot) do { if (tr) p.trace[(slot) * 64 + jj] = clock64(); } while (0)
    if (tr) p.trace[7 * 64] = clock64();
#else
#define ATR(slot) do { } while (0)
#endif
    for (int jj = 0; jj < n_kv; ++jj) {
      const int k0 = jj * BK;
      ATR(0);
      attn_wait(s_full, jj & 1);
      tc_fence_after();
      ATR(1);
      float s[64];
      ld64(lane_addr, s);
      tc_fence_before();
      mbar_arrive(s_free);  // S is in registers: the control warp may overwrite the tensor-memory buffer with the next step's scores
      ATR(2);
      const bool edge = (k0 + BK - 1 > t0) || (k0 + BK > p.T);  // diagonal block or ragged tail (uniform in the CTA)
      float mx = kNegInf;  // maxima are tracked on the raw scores; the softmax scale is folded into the exp2 argument
      if (edge) {
        const int lim = min(t, p.T - 1) - k0;  // last valid column of this row in the block
#pragma unroll
        for (int c = 0; c < 64; ++c) {
          s[c] = c <= lim ? s[c] : kNegInf;
          mx = fmaxf(mx, s[c]);
        }
      } else {
        float m0 = s[0], m1 = s[1], m2 = s[2], m3 = s[3];  // four independent chains instead of one 64-deep dependency
#pragma unroll
        for (int c = 4; c < 64; c += 4) {
          m0 = fmaxf(m0, s[c]);
          m1 = fmaxf(m1, s[c + 1]);
          m2 = fmaxf(m2, s[c + 2]);
          m3 = fmaxf(m3, s[c + 3]);
        }
        mx = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
      }
      if (jj > 0) {  // P (and O, for the rescale below) are free once the previous step's P·V has completed
        attn_wait(o_full, (jj - 1) & 1);
        tc_fence_after();
      }
      // Whether a row moves its reference maximum depends on that row's own scores only.  The TMEM round trip below is
      // warp-collective, but rows that do not need it keep m and scale by exactly 1, so a row's result never depends on
      // its warp-mates -- rows of the next batch in a ragged tail tile, or later rows that see later keys.  Rows past T
      // (next-batch queries loaded into the tail tile) never rescale, so their P may overflow to inf and their O / l turn
      // inf or NaN.  That is harmless: P·V is row-local (O row r reads only P row r) and those rows are never stored.
      const bool bump = t < p.T && (mx - m) * p.scale_log2 > 8.0f;
      if (jj == 0) {
        m = mx;  // first step: P·V overwrites O (accumulate = 0), nothing to rescale
      } else if (__any_sync(0xffffffffu, bump)) {
        // rare: bring the rows that need it to their new reference maximum
        const float m_new = bump ? mx : m;
        const float f = bump ? fast_exp2((m - m_new) * p.scale_log2) : 1.0f;
        uint32_t o0[32], o1[32];
        tmem_ld_32x32b_x32(lane_addr + 64, o0);
        tmem_ld_32x32b_x32(lane_addr + 96, o1);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          o0[i] = __float_as_uint(__uint_as_float(o0[i]) * f);
          o1[i] = __float_as_uint(__uint_as_float(o1[i]) * f);
        }
        tmem_st_32x32b_x32(lane_addr + 64, o0);
        tmem_st_32x32b_x32(lane_addr + 96, o1);
        tmem_st_wait();
        l *= f;
        m = m_new;
      }
      const float mc = m * p.scale_log2;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
      for (int c = 0; c < 64; c += 4) {
        s[c] = fast_exp2(fmaf(s[c], p.scale_log2, -mc));
        s[c + 1] = fast_exp2(fmaf(s[c + 1], p.scale_log2, -mc));
        s[c + 2] = fast_exp2(fmaf(s[c + 2], p.scale_log2, -mc));
        s[c + 3] = fast_exp2(fmaf(s[c + 3], p.scale_log2, -mc));
        a0 += s[c];
        a1 += s[c + 1];
        a2 += s[c + 2];
        a3 += s[c + 3];
      }
      l += (a0 + a1) + (a2 + a3);
      ATR(3);
      store_row64(sP, r, s);
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(p_ready);
      ATR(4);
    }
#undef ATR
    float O[64];
    if (active) {
      attn_wait(o_full, (n_kv - 1) & 1);
      tc_fence_after();
      ld64(lane_addr + 64, O);
    }
    if (active && t < p.T) {
      const float inv = 1.0f / l;
      bf16* op = p.out + (long long)(row0 + t) * p.ld_out + head * p.hd;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        if (q * 8 < p.hd) {
          float f[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) f[i] = O[q * 8 + i] * inv;
          *reinterpret_cast<uint4*>(op + q * 8) = pack8(f);
        }
      }
      p.lse[((long long)b * p.nh + head) * p.T + t] = m * p.scale_log2 + log2f(l);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4 * NG) {
    tc_fence_after();
    tmem_dealloc(*tmem_slot, pow2_cols(NG * 128));
  }
}

// =============================================================================================== backward: delta
// delta[b, h, t] = sum_d dO[b, t, h, d] * O[b, t, h, d]
__global__ void __launch_bounds__(256) attn_delta_kernel(const bf16* __restrict__ o, long long ld_o, const bf16* __restrict__ dout,
                                                         long long ld_do, float* __restrict__ delta, int B, int T, int nh, int hd) {
  pdl_wait();
  pdl_launch_dependents();
  const long long total = (long long)B * T * nh;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int h = int(i % nh);
    const long long row = i / nh;
    const bf16* a = o + row * ld_o + h * hd;
    const bf16* g = dout + row * ld_do + h * hd;
    float acc = 0.f;
    for (int q = 0; q < hd; q += 8) {
      float x[8], y[8];
      unpack8(*reinterpret_cast<const uint4*>(a + q), x);
      unpack8(*reinterpret_cast<const uint4*>(g + q), y);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc += x[j] * y[j];
    }
    const long long bb = row / T, t = row % T;
    delta[(bb * nh + h) * T + t] = acc;
  }
}

struct BwdArgs {
  const float* lse;
  const float* delta;
  bf16* dqkv;
  long long ld_dqkv;
  int B, T, nh, hd;
  float scale, scale_log2;
  int store_ds;  // dK/dV kernel also writes its dSᵀ tiles to global memory (consumed by attn_bwd_dq2_kernel)
};

// =============================================================================================== backward: dQ
__global__ void __launch_bounds__((kBwdRowWarps * kDqGroups + kDqGroups) * 32, kDqGroups == 1 ? 2 : 1) attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap map_qkv,
                                                                   const __grid_constant__ CUtensorMap map_do, const BwdArgs p) {
  constexpr int NG = kDqGroups;
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;  // warp index known uniform to ptxas
  if (threadIdx.x == 0) pdl_launch_dependents();
  const bool is_ctrl = warp >= kBwdRowWarps * NG;
  const int g = is_ctrl ? warp - kBwdRowWarps * NG : warp / kBwdRowWarps;  // group of this warp
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem0 = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem = smem0 + g * kDqGroupBytes;
  uint8_t* sQ = smem;
  uint8_t* sdO = sQ + kTile128;
  uint8_t* sK = sdO + kTile128;     // 2 stages
  uint8_t* sV = sK + 2 * kTile64;   // 2 stages
  uint8_t* sdS = sV + 2 * kTile64;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sdS + kTile128);
  uint64_t* q_full = bars;
  uint64_t* kv_full = bars + 1;
  uint64_t* kv_free = bars + 3;
  uint64_t* sdp_full = bars + 5;
  uint64_t* ds_ready = bars + 6;
  uint64_t* dq_full = bars + 7;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem0 + 3 * kTile128 + 4 * kTile64 + 64);

  const int nqb = (p.T + BQ - 1) / BQ;
  const long long per = (long long)p.B * p.nh;
  const long long item = (long long)blockIdx.x * NG + g;
  const bool active = item < per * nqb;
  const int qb = active ? nqb - 1 - int(item / per) : 0;
  const int head = int((item % per) % p.nh), b = active ? int((item % per) / p.nh) : 0;
  const int t0 = qb * BQ;
  const int kv_end = min(p.T, t0 + BQ);
  const int n_kv = active ? (kv_end + BK - 1) / BK : 0;
  const int row0 = b * p.T;

  if (is_ctrl && lane == 0) {
    mbar_init(q_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_free[i], 1);
    }
    mbar_init(sdp_full, 1);
    mbar_init(ds_ready, 32 * kBwdRowWarps);
    mbar_init(dq_full, 1);
    fence_barrier_init();
    tma_prefetch_desc(&map_qkv);
    tma_prefetch_desc(&map_do);
  }
  if (warp == kBwdRowWarps * NG) {
    tmem_alloc(tmem_slot, pow2_cols(NG * 256));  // per group (256 columns): S 0-63, dP 64-127, dQ 128-191
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0) + g * 256;
  pdl_wait();

  if (is_ctrl) {
    if (active) {
      auto load_kv = [&](int jj, int st) {
        RB_ONE_LANE(mbar_arrive_expect_tx(&kv_full[st], 2 * kTile64);
                    tma_load_3d(&map_qkv, &kv_full[st], sK + st * kTile64, 0, p.nh + head, row0 + jj * BK);
                    tma_load_3d(&map_qkv, &kv_full[st], sV + st * kTile64, 0, 2 * p.nh + head, row0 + jj * BK););
      };
      RB_ONE_LANE(mbar_arrive_expect_tx(q_full, 2 * kTile128);
                  tma_load_3d(&map_qkv, q_full, sQ, 0, head, row0 + t0);
                  tma_load_3d(&map_qkv, q_full, sQ + kTile64, 0, head, row0 + t0 + 64);
                  tma_load_3d(&map_do, q_full, sdO, 0, head, row0 + t0);
                  tma_load_3d(&map_do, q_full, sdO + kTile64, 0, head, row0 + t0 + 64););
      load_kv(0, 0);
      if (n_kv > 1) load_kv(1, 1);
      constexpr uint32_t idesc_kk = make_idesc_bf16(128, 64, 0, 0);
      constexpr uint32_t idesc_kmn = make_idesc_bf16(128, 64, 0, 1);
      auto issue_sdp = [&](int st) {
        RB_ONE_LANE(
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_f16_ss(tmem_base, desc_k(sQ, k), desc_k(sK + st * kTile64, k), idesc_kk, k != 0);
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_f16_ss(tmem_base + 64, desc_k(sdO, k), desc_k(sV + st * kTile64, k), idesc_kk, k != 0);
            umma_commit(sdp_full););
      };
      attn_wait(q_full, 0);
      attn_wait(&kv_full[0], 0);
      tc_fence_after();
      issue_sdp(0);
      for (int jj = 0; jj < n_kv; ++jj) {
        const int st = jj & 1;
        attn_wait(ds_ready, jj & 1);
        tc_fence_after();
        RB_ONE_LANE(
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_f16_ss(tmem_base + 128, desc_k(sdS, k), desc_mn(sK + st * kTile64, k), idesc_kmn, (jj | k) != 0);
            umma_commit(&kv_free[st]););
        if (jj + 1 < n_kv) {
          attn_wait(&kv_full[st ^ 1], ((jj + 1) >> 1) & 1);
          tc_fence_after();
          issue_sdp(st ^ 1);  // its commit also covers the dQ MMAs above: dS may be overwritten once sdp_full fires
        } else {
          RB_ONE_LANE(umma_commit(dq_full););
        }
        if (jj + 2 < n_kv) {
          attn_wait(&kv_free[st], (jj >> 1) & 1);
          load_kv(jj + 2, st);
        }
      }
    }
  } else {
    const int r = threadIdx.x & 127, hf = (threadIdx.x >> 7) & 1;  // row of the query block, column half of every step
    const int t = t0 + r;
    const uint32_t lane_addr = tmem_addr(tmem_base, (warp & 3) * 32, hf * 32);
    const long long stat = ((long long)b * p.nh + head) * p.T + t;
    const float lse = (active && t < p.T) ? p.lse[stat] : 0.f;
    const float dl = (active && t < p.T) ? p.delta[stat] : 0.f;
    for (int jj = 0; jj < n_kv; ++jj) {
      const int k0 = jj * BK + hf * 32;
      attn_wait(sdp_full, jj & 1);
      tc_fence_after();
      float s[32], dp[32];
      ld32(lane_addr, s);
      ld32(lane_addr + 64, dp);
      const bool edge = (jj * BK + BK - 1 > t0) || (jj * BK + BK > p.T);
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        float pr = fast_exp2(fmaf(s[c], p.scale_log2, -lse));
        if (edge && (k0 + c > t || k0 + c >= p.T)) pr = 0.f;
        s[c] = pr * (dp[c] - dl) * p.scale;
      }
      store_row32(sdS, r, hf, s);
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(ds_ready);
    }
    float dq[32];
    if (active) {
      attn_wait(dq_full, 0);
      tc_fence_after();
      ld32(lane_addr + 128, dq);
    }
    if (active && t < p.T) {
      bf16* op = p.dqkv + (long long)(row0 + t) * p.ld_dqkv + head * p.hd + hf * 32;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (hf * 32 + q * 8 < p.hd) {
          float f[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) f[i] = dq[q * 8 + i];
          *reinterpret_cast<uint4*>(op + q * 8) = pack8(f);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kBwdRowWarps * NG) {
    tc_fence_after();
    tmem_dealloc(*tmem_slot, pow2_cols(NG * 256));
  }
}

// =============================================================================================== backward: dK, dV
__global__ void __launch_bounds__((kBwdRowWarps * kDkvGroups + kDkvGroups) * 32, kDkvGroups == 1 ? 2 : 1) attn_bwd_dkv_kernel(const __grid_constant__ CUtensorMap map_qkv,
                                                                    const __grid_constant__ CUtensorMap map_do,
                                                                    const __grid_constant__ CUtensorMap map_ds, const BwdArgs p) {
  constexpr int NG = kDkvGroups;
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;  // warp index known uniform to ptxas
  if (threadIdx.x == 0) pdl_launch_dependents();
  const bool is_ctrl = warp >= kBwdRowWarps * NG;
  const int g = is_ctrl ? warp - kBwdRowWarps * NG : warp / kBwdRowWarps;  // group of this warp
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem0 = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem = smem0 + g * kDkvGroupBytes;
  uint8_t* sK = smem;
  uint8_t* sV = sK + kTile128;
  uint8_t* sQ = sV + kTile128;      // 2 stages of [64 queries x 64]
  uint8_t* sdO = sQ + 2 * kTile64;  // 2 stages
  uint8_t* sPt = sdO + 2 * kTile64;
  uint8_t* sdSt = sPt + kTile128;
  float* s_lse = reinterpret_cast<float*>(sdSt + kTile128);  // [2][64]
  float* s_dl = s_lse + 128;                                  // [2][64]
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_dl + 128);
  uint64_t* kv_full = bars;
  uint64_t* q_full = bars + 1;
  uint64_t* q_free = bars + 3;
  uint64_t* sdp_full = bars + 5;
  uint64_t* pds_ready = bars + 6;
  uint64_t* acc_full = bars + 7;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem0 + 4 * kTile128 + 4 * kTile64 + 1024 + 64);

  // work item of this group: (key block, head, batch); early key blocks see the most queries and go first
  const int nkb = (p.T + BQ - 1) / BQ;
  const long long per = (long long)p.B * p.nh;
  const long long item = (long long)blockIdx.x * NG + g;
  const bool active = item < per * nkb;
  const int kb = active ? int(item / per) : 0;
  const int head = int((item % per) % p.nh), b = active ? int((item % per) / p.nh) : 0;
  const int kstart = kb * BQ;
  const int n_q = active ? (p.T - kstart + BK - 1) / BK : 0;  // query steps of 64 starting at the block's first key
  const int row0 = b * p.T;

  if (is_ctrl && lane == 0) {
    mbar_init(kv_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_free[i], 1);
    }
    mbar_init(sdp_full, 1);
    mbar_init(pds_ready, 32 * kBwdRowWarps);
    mbar_init(acc_full, 1);
    fence_barrier_init();
    tma_prefetch_desc(&map_qkv);
    tma_prefetch_desc(&map_do);
    if (p.store_ds) tma_prefetch_desc(&map_ds);
  }
  if (warp == kBwdRowWarps * NG) {
    tmem_alloc(tmem_slot, pow2_cols(NG * 256));  // per group (256 columns): Sᵀ 0-63, dPᵀ 64-127, dV 128-191, dK 192-255
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0) + g * 256;
  pdl_wait();

  if (is_ctrl) {
    if (active) {
      auto load_q = [&](int ii, int st) {
        RB_ONE_LANE(mbar_arrive_expect_tx(&q_full[st], 2 * kTile64);
                    tma_load_3d(&map_qkv, &q_full[st], sQ + st * kTile64, 0, head, row0 + kstart + ii * BK);
                    tma_load_3d(&map_do, &q_full[st], sdO + st * kTile64, 0, head, row0 + kstart + ii * BK););
      };
      RB_ONE_LANE(mbar_arrive_expect_tx(kv_full, 2 * kTile128);
                  tma_load_3d(&map_qkv, kv_full, sK, 0, p.nh + head, row0 + kstart);
                  tma_load_3d(&map_qkv, kv_full, sK + kTile64, 0, p.nh + head, row0 + kstart + 64);
                  tma_load_3d(&map_qkv, kv_full, sV, 0, 2 * p.nh + head, row0 + kstart);
                  tma_load_3d(&map_qkv, kv_full, sV + kTile64, 0, 2 * p.nh + head, row0 + kstart + 64););
      load_q(0, 0);
      if (n_q > 1) load_q(1, 1);
      constexpr uint32_t idesc_kk = make_idesc_bf16(128, 64, 0, 0);
      constexpr uint32_t idesc_kmn = make_idesc_bf16(128, 64, 0, 1);
      auto issue_sdp = [&](int st) {
        RB_ONE_LANE(
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_f16_ss(tmem_base, desc_k(sK, k), desc_k(sQ + st * kTile64, k), idesc_kk, k != 0);
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_f16_ss(tmem_base + 64, desc_k(sV, k), desc_k(sdO + st * kTile64, k), idesc_kk, k != 0);
            umma_commit(sdp_full););
      };
      attn_wait(kv_full, 0);
      attn_wait(&q_full[0], 0);
      tc_fence_after();
      issue_sdp(0);
      for (int ii = 0; ii < n_q; ++ii) {
        const int st = ii & 1;
        attn_wait(pds_ready, ii & 1);
        tc_fence_after();
        RB_ONE_LANE(
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_f16_ss(tmem_base + 128, desc_k(sPt, k), desc_mn(sdO + st * kTile64, k), idesc_kmn, (ii | k) != 0);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_f16_ss(tmem_base + 192, desc_k(sdSt, k), desc_mn(sQ + st * kTile64, k), idesc_kmn, (ii | k) != 0);
            umma_commit(&q_free[st]););
        if (p.store_ds && lane == 0) {  // bulk-store groups are per thread: lane 0 stores, commits and waits
          // dSᵀ tile [128 keys x 64 queries] -> global [b*nh+head][key][query]: the dQ kernel then is a plain TMA -> MMA pipeline
          // (dQ = dS·K) instead of recomputing S and dP (the row threads fenced their writes before arriving on pds_ready)
          tma_store_3d(&map_ds, sdSt, kstart + ii * BK, kstart, b * p.nh + head);
          tma_store_commit();
        }
        __syncwarp();
        if (ii + 1 < n_q) {
          attn_wait(&q_full[st ^ 1], ((ii + 1) >> 1) & 1);
          tc_fence_after();
          if (p.store_ds && lane == 0) tma_store_wait_read<0>();  // the next step's row threads overwrite the tile once sdp_full fires
          __syncwarp();
          issue_sdp(st ^ 1);
        } else {
          RB_ONE_LANE(umma_commit(acc_full););
          if (p.store_ds && lane == 0) tma_store_wait<0>();
          __syncwarp();
        }
        if (ii + 2 < n_q) {
          attn_wait(&q_free[st], (ii >> 1) & 1);
          load_q(ii + 2, st);
        }
      }
    }
  } else {
    const int r = threadIdx.x & 127, hf = (threadIdx.x >> 7) & 1;  // key row of the block, query-column half of every step
    const int kk = kstart + r;  // this thread's key
    const uint32_t lane_addr = tmem_addr(tmem_base, (warp & 3) * 32, hf * 32);
    const long long stat0 = ((long long)b * p.nh + head) * p.T;
    for (int ii = 0; ii < n_q; ++ii) {
      const int q0 = kstart + ii * BK;
      {  // stage the 64 queries' lse / delta (double buffered; the barrier below orders reuse)
        const int w = threadIdx.x & 255;
        if (w < 128) {
          const int c = w & 63;
          const int tq = q0 + c;
          float* dst = (w < 64 ? s_lse : s_dl) + (ii & 1) * 64;
          const float* src = w < 64 ? p.lse : p.delta;
          dst[c] = tq < p.T ? src[stat0 + tq] : 0.f;
        }
      }
      named_bar_sync(1 + g, 32 * kBwdRowWarps);
      const float4* lse4 = reinterpret_cast<const float4*>(s_lse + (ii & 1) * 64 + hf * 32);
      const float4* dl4 = reinterpret_cast<const float4*>(s_dl + (ii & 1) * 64 + hf * 32);
      attn_wait(sdp_full, ii & 1);
      tc_fence_after();
      float s[32], dp[32];
      ld32(lane_addr, s);
      ld32(lane_addr + 64, dp);
      const bool edge = (q0 < kstart + BQ) || (q0 + BK > p.T) || (kstart + BQ > p.T);
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) {
        const float4 l4 = lse4[c4], d4 = dl4[c4];  // 16 vector loads per step instead of 128 scalar broadcasts
        const float ls[4] = {l4.x, l4.y, l4.z, l4.w}, ds[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int c = c4 * 4 + i;
          const int tq = q0 + hf * 32 + c;
          float pr = fast_exp2(fmaf(s[c], p.scale_log2, -ls[i]));
          if (edge && (kk > tq || tq >= p.T || kk >= p.T)) pr = 0.f;
          s[c] = pr;
          dp[c] = pr * (dp[c] - ds[i]) * p.scale;
        }
      }
      store_row32(sPt, r, hf, s);
      store_row32(sdSt, r, hf, dp);
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(pds_ready);
    }
    if (active) {
      attn_wait(acc_full, 0);
      tc_fence_after();
    }
    float acc[32];
#pragma unroll 1
    for (int which = 0; active && which < 2; ++which) {  // 0: dV -> v slot, 1: dK -> k slot
      ld32(lane_addr + 128 + which * 64, acc);
      if (kk < p.T) {
        bf16* op = p.dqkv + (long long)(row0 + kk) * p.ld_dqkv + (long long)((which == 0 ? 2 : 1) * p.nh + head) * p.hd + hf * 32;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (hf * 32 + q * 8 < p.hd) {
            float f[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) f[i] = acc[q * 8 + i];
            *reinterpret_cast<uint4*>(op + q * 8) = pack8(f);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kBwdRowWarps * NG) {
    tc_fence_after();
    tmem_dealloc(*tmem_slot, pow2_cols(NG * 256));
  }
}

// =============================================================================================== backward: dQ from stored dS
// dQ[q, :] = Σ_k dS[q, k] · K[k, :] with dSᵀ tiles written by the dK/dV kernel: no scores, no exponentials, no row-thread work inside
// the loop -- a two-stage TMA -> tcgen05 pipeline per (128 queries, head, batch).  A = dSᵀ tile [128 keys x 128 queries] read MN-major
// (M = queries), B = K tile [128 keys x head_dim] read MN-major (N = head_dim), K = 128 keys per stage.
constexpr int kDq2StageBytes = 2 * kTile128 + 2 * kTile64;   // dSᵀ (two 64-query chunks) + K (two 64-key tiles)
constexpr int kDq2Smem = 2 * kDq2StageBytes + 1024 + 1024;
__global__ void __launch_bounds__(160, 2) attn_bwd_dq2_kernel(const __grid_constant__ CUtensorMap map_qkv, const __grid_constant__ CUtensorMap map_ds,
                                                              const BwdArgs p) {
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;  // warp index known uniform to ptxas
  const bool is_ctrl = warp >= 4;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * kDq2StageBytes);
  uint64_t* full = bars;       // [2]
  uint64_t* free_ = bars + 2;  // [2]
  uint64_t* done = bars + 4;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

  const int nqb = (p.T + BQ - 1) / BQ;
  const long long per = (long long)p.B * p.nh;
  const long long item = blockIdx.x;
  const int qb = nqb - 1 - int(item / per);  // heaviest (latest) query blocks first
  const int head = int((item % per) % p.nh), b = int((item % per) / p.nh);
  const int t0 = qb * BQ;
  const int row0 = b * p.T;
  const int n_kb = qb + 1;  // causal: key blocks 0 .. qb

  if (is_ctrl && lane == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&free_[i], 1);
    }
    mbar_init(done, 1);
    fence_barrier_init();
    tma_prefetch_desc(&map_qkv);
    tma_prefetch_desc(&map_ds);
  }
  if (warp == 4) {
    tmem_alloc(tmem_slot, 64);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  pdl_wait();

  if (is_ctrl) {
    {
      constexpr uint32_t idesc = make_idesc_bf16(128, 64, 1, 1);
      auto load = [&](int kb, int st) {
        uint8_t* sA = smem + st * kDq2StageBytes;
        uint8_t* sB = sA + 2 * kTile128;
        RB_ONE_LANE(mbar_arrive_expect_tx(&full[st], kDq2StageBytes);
                    tma_load_3d(&map_ds, &full[st], sA, t0, kb * BQ, b * p.nh + head);
                    tma_load_3d(&map_ds, &full[st], sA + kTile128, t0 + 64, kb * BQ, b * p.nh + head);
                    tma_load_3d(&map_qkv, &full[st], sB, 0, p.nh + head, row0 + kb * BQ);
                    tma_load_3d(&map_qkv, &full[st], sB + kTile64, 0, p.nh + head, row0 + kb * BQ + 64););
      };
      load(0, 0);
      if (n_kb > 1) load(1, 1);
      for (int kb = 0; kb < n_kb; ++kb) {
        const int st = kb & 1;
        attn_wait(&full[st], (kb >> 1) & 1);
        tc_fence_after();
        const uint32_t sA = smem_u32(smem + st * kDq2StageBytes), sB = sA + 2 * kTile128;
        RB_ONE_LANE(
            const uint64_t da = make_desc_sw128(sA, kTile128, 1024); const uint64_t db = make_desc_sw128(sB, 8192, 1024);
#pragma unroll
            for (int k = 0; k < 8; ++k)  // 16 keys per instruction (2048 B = +128 in the start-address field); A: query chunks of 64 are
              umma_f16_ss(tmem_base, da + 128 * k, db + 128 * k, idesc, (kb | k) != 0);  // 16 KB apart, 8-key groups 1 KB apart
            umma_commit(&free_[st]););
        if (kb + 2 < n_kb) {
          attn_wait(&free_[st], (kb >> 1) & 1);
          load(kb + 2, st);
        }
      }
      RB_ONE_LANE(umma_commit(done););
    }
  } else {
    const int r = threadIdx.x & 127;
    const int t = t0 + r;
    attn_wait(done, 0);
    tc_fence_after();
    float dq[64];
    ld64(tmem_addr(tmem_base, (warp & 3) * 32, 0), dq);
    if (t < p.T) {
      bf16* op = p.dqkv + (long long)(row0 + t) * p.ld_dqkv + head * p.hd;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        if (q * 8 < p.hd) {
          float f[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) f[i] = dq[q * 8 + i];
          *reinterpret_cast<uint4*>(op + q * 8) = pack8(f);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 64);
  }
}

// ---------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------
struct HeadMapKey {
  const void* ptr;
  long long ld, rows;
  int hd, heads;
  bool operator==(const HeadMapKey& o) const { return ptr == o.ptr && ld == o.ld && rows == o.rows && hd == o.hd && heads == o.heads; }
};
struct HeadMapHash {
  size_t operator()(const HeadMapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.ptr);
    h ^= std::hash<long long>()(k.ld * 1315423911ll + k.rows) + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2);
    h ^= std::hash<long long>()(((long long)k.hd << 32) | (unsigned)k.heads) + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2);
    return h;
  }
};
std::unordered_map<HeadMapKey, CUtensorMap, HeadMapHash> g_head_maps;
std::mutex g_head_maps_mu;

// [rows, heads*hd] bf16 (row stride ld) viewed as [hd, heads, rows]; box = 64 x 1 x 64 rows
CUtensorMap head_map(const void* ptr, long long ld, long long rows, int hd, int heads) {
  HeadMapKey key{ptr, ld, rows, hd, heads};
  {
    std::lock_guard<std::mutex> lk(g_head_maps_mu);
    auto it = g_head_maps.find(key);
    if (it != g_head_maps.end()) return it->second;
  }
  CUtensorMap m = make_map_3d_bf16(ptr, hd, heads, rows, hd, ld, 64, 1, 64);
  std::lock_guard<std::mutex> lk(g_head_maps_mu);
  if (g_head_maps.size() > 4096) g_head_maps.clear();
  g_head_maps.emplace(key, m);
  return m;
}

void check_shape(int B, int T, int nh, int hd) {
  if (B <= 0 || T <= 0 || nh <= 0) throw std::runtime_error("attention: empty problem");
  if (hd % 8 != 0 || hd > 64) throw std::runtime_error("attention: head_dim must be a multiple of 8 and <= 64");
}

constexpr int kFwdSmem = kFwdGroups * kFwdGroupBytes + 1024;
constexpr int kDqSmem = kDqGroups * kDqGroupBytes + 1024;
constexpr int kDkvSmem = kDkvGroups * kDkvGroupBytes + 1024;
constexpr int kFwdThreads = 5 * kFwdGroups * 32, kDqThreads = (kBwdRowWarps + 1) * kDqGroups * 32, kDkvThreads = (kBwdRowWarps + 1) * kDkvGroups * 32;

void* g_attn_trace = nullptr;
int g_attn_occupancy[3] = {0, 0, 0};  // resident CTAs per SM reported for fwd / dq / dkv

}  // namespace

void attention_set_trace(void* buf) { g_attn_trace = buf; }
int attention_occupancy(int which) { return which >= 0 && which < 3 ? g_attn_occupancy[which] : 0; }

void attention_fwd(const AttnDesc& d, cudaStream_t stream) {
  check_shape(d.B, d.T, d.nh, d.hd);
  const long long rows = (long long)d.B * d.T;
  CUtensorMap map = head_map(d.qkv, d.ld_qkv, rows, d.hd, 3 * d.nh);
  static bool configured = false;
  if (!configured) {
    check(cudaFuncSetAttribute(attn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kFwdSmem), "cudaFuncSetAttribute(attn_fwd)");
    // several CTAs per SM are the latency-hiding mechanism of these kernels: ask for the largest shared-memory carve-out
    check(cudaFuncSetAttribute(attn_fwd_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared), "carveout(attn_fwd)");
    int occ = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, attn_fwd_kernel, kFwdThreads, kFwdSmem);
    g_attn_occupancy[0] = occ;
    if (getenv("RB_ATTN_DEBUG") != nullptr) {
      cudaFuncAttributes fa;
      cudaFuncGetAttributes(&fa, attn_fwd_kernel);
      int o0 = 0, o1 = 0;
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o0, attn_fwd_kernel, kFwdThreads, 0);
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o1, attn_fwd_kernel, kFwdThreads, 32768);
      int smem_sm = 0, smem_optin = 0, regs_sm = 0;
      cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, 0);
      cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, 0);
      cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, 0);
      printf("attn_fwd: regs %d static smem %zu maxdyn %d local %zu | occ(dyn=%d)=%d occ(0)=%d occ(32K)=%d | smem/SM %d optin %d regs/SM %d\n",
             fa.numRegs, fa.sharedSizeBytes, fa.maxDynamicSharedSizeBytes, fa.localSizeBytes, kFwdSmem, occ, o0, o1, smem_sm, smem_optin, regs_sm);
    }
    configured = true;
  }
  FwdArgs p;
  p.trace = reinterpret_cast<long long*>(g_attn_trace);
  p.out = reinterpret_cast<bf16*>(d.out); p.ld_out = d.ld_out; p.lse = d.lse;
  p.B = d.B; p.T = d.T; p.nh = d.nh; p.hd = d.hd;
  p.scale_log2 = d.scale * 1.4426950408889634f;
  const long long items = (long long)((d.T + BQ - 1) / BQ) * d.nh * d.B;
  dim3 grid((unsigned)((items + kFwdGroups - 1) / kFwdGroups));
  launch_k(attn_fwd_kernel, grid, kFwdThreads, kFwdSmem, stream, map, p);
  RB_CHECK_LAUNCH("attn_fwd_kernel");
}

void attention_bwd(const AttnBwdDesc& d, cudaStream_t stream) {
  check_shape(d.B, d.T, d.nh, d.hd);
  const long long rows = (long long)d.B * d.T;
  CUtensorMap map_qkv = head_map(d.qkv, d.ld_qkv, rows, d.hd, 3 * d.nh);
  CUtensorMap map_do = head_map(d.dout, d.ld_dout, rows, d.hd, d.nh);
  static bool configured = false;
  if (!configured) {
    check(cudaFuncSetAttribute(attn_bwd_dq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kDqSmem), "cudaFuncSetAttribute(attn_dq)");
    check(cudaFuncSetAttribute(attn_bwd_dkv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kDkvSmem), "cudaFuncSetAttribute(attn_dkv)");
    check(cudaFuncSetAttribute(attn_bwd_dq_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared), "carveout(attn_dq)");
    check(cudaFuncSetAttribute(attn_bwd_dkv_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared), "carveout(attn_dkv)");
    int occ = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, attn_bwd_dq_kernel, kDqThreads, kDqSmem);
    g_attn_occupancy[1] = occ;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, attn_bwd_dkv_kernel, kDkvThreads, kDkvSmem);
    g_attn_occupancy[2] = occ;
    configured = true;
  }
  {
    const long long total = rows * d.nh;
    const int grid = (int)std::min<long long>((total + 255) / 256, (long long)num_sms() * 8);
    launch_k(attn_delta_kernel, grid, 256, 0, stream, reinterpret_cast<const bf16*>(d.out), d.ld_out, reinterpret_cast<const bf16*>(d.dout),
                                                d.ld_dout, d.delta, d.B, d.T, d.nh, d.hd);
    RB_CHECK_LAUNCH("attn_delta_kernel");
  }
  BwdArgs p;
  p.lse = d.lse; p.delta = d.delta; p.dqkv = reinterpret_cast<bf16*>(d.dqkv); p.ld_dqkv = d.ld_dqkv;
  p.B = d.B; p.T = d.T; p.nh = d.nh; p.hd = d.hd;
  p.scale = d.scale; p.scale_log2 = d.scale * 1.4426950408889634f;
  const long long items = (long long)((d.T + BQ - 1) / BQ) * d.nh * d.B;
  p.store_ds = d.ds_workspace != nullptr ? 1 : 0;
  CUtensorMap map_ds = map_do;
  if (p.store_ds) {
    // dSᵀ workspace [B*nh][Tp keys][Tp queries] bf16, Tp = T rounded up to 64 (16-byte pitch for any T); tiles of 64 queries x 128 keys
    const long long Tp = attention_ds_pitch(d.T);
    map_ds = make_map_3d_bf16(d.ds_workspace, d.T, d.T, (long long)d.B * d.nh, Tp, Tp * Tp, 64, 128, 1);
  }
  launch_k(attn_bwd_dkv_kernel, dim3((unsigned)((items + kDkvGroups - 1) / kDkvGroups)), kDkvThreads, kDkvSmem, stream, map_qkv, map_do, map_ds, p);
  RB_CHECK_LAUNCH("attn_bwd_dkv_kernel");
  if (p.store_ds) {
    static bool cfg2 = false;
    if (!cfg2) {
      check(cudaFuncSetAttribute(attn_bwd_dq2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kDq2Smem), "attr(attn_bwd_dq2)");
      cfg2 = true;
    }
    launch_k(attn_bwd_dq2_kernel, dim3((unsigned)items), 160, kDq2Smem, stream, map_qkv, map_ds, p);
    RB_CHECK_LAUNCH("attn_bwd_dq2_kernel");
  } else {
    launch_k(attn_bwd_dq_kernel, dim3((unsigned)((items + kDqGroups - 1) / kDqGroups)), kDqThreads, kDqSmem, stream, map_qkv, map_do, p);
    RB_CHECK_LAUNCH("attn_bwd_dq_kernel");
  }
}

long long attention_ds_pitch(int T) { return ((long long)T + 63) / 64 * 64; }
long long attention_ds_workspace_elems(int B, int T, int nh) {
  const long long Tp = attention_ds_pitch(T);
  return (long long)B * nh * Tp * Tp;
}

}  // namespace rb

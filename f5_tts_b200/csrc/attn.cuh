// Non-causal flash-attention forward on tcgen05 for dim_head = 64 (reference: model/modules.py:471-556,
// F.scaled_dot_product_attention(q, k, v, attn_mask=None | key mask), scale 1/sqrt(64)).
//
// One CTA = one (sample, head, 256-query block) = TWO 128-row query tiles that ping-pong on the tensor core:
// while softmax warpgroup 0 works on S0 = Q0 K_j^T, the tensor core already computes S1 = Q1 K_j^T and the
// pending P V products, so MMA and the exp-heavy softmax overlap inside a CTA.
// q/k/v are read in place from the fused QKV projection output [Be*seq, 3*inner] (fp16) through ONE 3-D TMA tensor
// map (cols, seq rows, sample): no head-split transpose ever touches HBM, and rows past the end of a sample are
// zero-filled by TMA instead of leaking the next sample.
//   S_w = Q_w K^T  : tcgen05.mma 128x128x16 x4 (both operands K-major in shared memory), fp32 in TMEM
//   softmax        : 2 x 128 threads, one query row each (tcgen05.ld 32x32b: a thread owns a full row -> no shuffles);
//                    the whole 128-key row lives in registers (single pass); online max (3-input FMNMX3) / sum in fp32;
//                    lazy rescaling: O is only rescaled when some row's max grew by > 2^8.
//                    Exponentials: the MUFU.EX2 unit retires 16 lanes / clk / SM, which is HALF the tensor-core pace of
//                    this kernel, so kPolyOf8 of every 8 element pairs are computed on the FMA pipe instead
//                    (Cody-Waite split x = n + f, degree-3 polynomial for 2^f, exponent add for 2^n), all in packed
//                    fp32x2 arithmetic (FFMA2 / FADD2: one issue slot per two elements).
//   O_w += P_w V   : P never touches shared memory: it is written fp16-packed into TMEM (tcgen05.st, 64 columns per
//                    query tile) and consumed from there as the A operand of tcgen05.mma (TS form); V is consumed
//                    MN-major straight from its TMA layout.  That removes the 64 KB P store + 64 KB P read per key tile
//                    from the shared-memory port, which was as loaded as the MUFU unit.
// TMEM columns: S0 [0,128) S1 [128,256) O0 [256,320) O1 [320,384) P0 [384,448) P1 [448,512).
// Warp roles (384 threads = three warpgroups): warp 0 TMA producer, warp 1 MMA issuer / TMEM allocator, warps 2-3 idle;
// warps 4..7 softmax WG0, warps 8..11 softmax WG1 (warp w touches TMEM lane quarter w % 4).  The softmax threads hold a
// 128-score row AND its 64 packed probabilities in registers, so the register file is re-split with setmaxnreg: the
// producer warpgroup drops to 64 registers per thread, the two softmax warpgroups grow to 216 (no spills; 128 x 64 + 256 x 216 stays inside the 384 x 168 registers the CTA was launched with — setmaxnreg.inc can only draw on the CTA's own pool).
#pragma once
#include "common.cuh"
#include "kparams.h"

// register split of the CTA's pool (384 threads x 168 registers): 128 x PRODUCER + 256 x SOFTMAX must not exceed it
#ifndef F5_ATTN_REGS_PRODUCER
#define F5_ATTN_REGS_PRODUCER 64
#endif
#ifndef F5_ATTN_REGS_SOFTMAX
#define F5_ATTN_REGS_SOFTMAX 216
#endif
static_assert(128 * F5_ATTN_REGS_PRODUCER + 256 * F5_ATTN_REGS_SOFTMAX <= 384 * 168, "setmaxnreg split exceeds the CTA's pool");

namespace f5 {

__device__ __forceinline__ float ex2_approx(float x) {  // one MUFU.EX2; inputs are <= ~8, -inf -> 0
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void named_bar_arrive(int id, int nthreads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- packed fp32x2 helpers (sm_100: FFMA2 / FADD2 / FMUL2 issue once for two lanes of a register pair) ----
__device__ __forceinline__ uint64_t f2_pack(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t f2_sub(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t f2_add_rm(uint64_t a, uint64_t b) {  // round toward -inf
  uint64_t d;
  asm("add.rm.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

// 2^x for two lanes on the FMA pipe.  x <= ~8.  n = floor(x) by adding 1.5 * 2^23 with round-down (the integer lands in
// the low mantissa bits), f = x - n in [0, 1), 2^f by a degree-3 polynomial (max relative error 8.8e-5: below the fp16
// rounding P gets anyway), 2^n by adding n to the exponent field.  Coefficients: minimax fit of 2^f on [0, 1).
__device__ __forceinline__ void ex2_poly2(uint64_t x2, float& e0, float& e1) {
  float x0, x1;
  f2_unpack(x2, x0, x1);
  x0 = fmaxf(x0, -125.0f);  // also maps -inf (masked / first tile) to 2^-125 ~ 0
  x1 = fmaxf(x1, -125.0f);
  const uint64_t x = f2_pack(x0, x1);
  const uint64_t magic = f2_pack(12582912.0f, 12582912.0f);
  const uint64_t t = f2_add_rm(x, magic);
  const uint64_t f = f2_sub(x, f2_sub(t, magic));
  uint64_t p = f2_fma(f, f2_pack(0.077119089663028717f, 0.077119089663028717f),
                      f2_pack(0.227564394474029541f, 0.227564394474029541f));
  p = f2_fma(p, f, f2_pack(0.695146143436431885f, 0.695146143436431885f));
  p = f2_fma(p, f, f2_pack(1.0f, 1.0f));
  float p0, p1, t0, t1;
  f2_unpack(p, p0, p1);
  f2_unpack(t, t0, t1);
  e0 = __uint_as_float(__float_as_uint(p0) + (__float_as_uint(t0) << 23));  // exponent += n (two's complement wraps)
  e1 = __uint_as_float(__float_as_uint(p1) + (__float_as_uint(t1) << 23));
}

constexpr int kPolyOf8 = 3;  // element pairs (of every 8) whose 2^x runs on the FMA pipe instead of MUFU

// 32 scores -> 16 packed fp16 pairs of exp2(s * sc - ms).  Keys past the end of the sample carry a score of -inf (set by
// the caller on the last tile), so there is ONE code path; a 32-key chunk that lies entirely past the end costs nothing.
// POLY = pairs of every 8 computed with the polynomial (evenly interleaved with the MUFU ones).
template <int POLY>
__device__ __forceinline__ void exp_pack32(const uint32_t (&r)[32], int col0, int kv_rem, uint64_t sc2, uint64_t nms2,
                                           uint64_t& sum2, uint32_t* pk) {
  if (col0 >= kv_rem) {  // warp-uniform: every key of this chunk is past the end of the sample -> P = 0
#pragma unroll
    for (int i = 0; i < 16; ++i) pk[i] = 0u;
    return;
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const uint64_t x2 = f2_fma(f2_pack(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1])), sc2, nms2);
    float e0, e1;
    const int pi = i & 7;
    if (((pi + 1) * POLY) / 8 != (pi * POLY) / 8) {  // compile-time pattern
      ex2_poly2(x2, e0, e1);
    } else {
      float x0, x1;
      f2_unpack(x2, x0, x1);
      e0 = ex2_approx(x0);
      e1 = ex2_approx(x1);
    }
    sum2 = f2_add(sum2, f2_pack(e0, e1));
    pk[i] = pack_half2(e0, e1);
  }
}

__device__ __forceinline__ float row_max128(const uint32_t (&r0)[32], const uint32_t (&r1)[32], const uint32_t (&r2)[32],
                                            const uint32_t (&r3)[32]) {
  float ma = -INFINITY, mb = -INFINITY;
#pragma unroll
  for (int i = 0; i < 32; i += 2) {
    ma = fmax3(ma, __uint_as_float(r0[i]), __uint_as_float(r0[i + 1]));
    mb = fmax3(mb, __uint_as_float(r1[i]), __uint_as_float(r1[i + 1]));
    ma = fmax3(ma, __uint_as_float(r2[i]), __uint_as_float(r2[i + 1]));
    mb = fmax3(mb, __uint_as_float(r3[i]), __uint_as_float(r3[i + 1]));
  }
  return fmaxf(ma, mb);
}

__device__ __forceinline__ float row_max32(const uint32_t (&r)[32]) {
  float ma = -INFINITY, mb = -INFINITY;
#pragma unroll
  for (int i = 0; i < 32; i += 4) {
    ma = fmax3(ma, __uint_as_float(r[i]), __uint_as_float(r[i + 1]));
    mb = fmax3(mb, __uint_as_float(r[i + 2]), __uint_as_float(r[i + 3]));
  }
  return fmaxf(ma, mb);
}

// scores of keys at or past kv_rem -> -inf (last key tile of a sample only)
__device__ __forceinline__ void mask_tail32(uint32_t (&r)[32], int col0, int kv_rem) {
#pragma unroll
  for (int i = 0; i < 32; ++i)
    if (col0 + i >= kv_rem) r[i] = 0xff800000u;
}

template <int POLY>
__global__ void __launch_bounds__(kAttnThreads, 1)
attn_fwd_tcgen05_kernel(const __grid_constant__ CUtensorMap tmQKV, const AttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  uint8_t* sQ = smem;                              // 2 tiles
  uint8_t* sK = sQ + 2 * kAttnTile;                // kAttnStages tiles
  uint8_t* sV = sK + kAttnStages * kAttnTile;      // kAttnStages tiles
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + kAttnStages * kAttnTile);
  uint64_t* q_full = bars;                         // [1]
  uint64_t* k_full = q_full + 1;                   // [stages]
  uint64_t* k_empty = k_full + kAttnStages;        // [stages]
  uint64_t* v_full = k_empty + kAttnStages;        // [stages]
  uint64_t* v_empty = v_full + kAttnStages;        // [stages]
  uint64_t* s_full = v_empty + kAttnStages;        // [2]
  uint64_t* p_full = s_full + 2;                   // [2]
  uint64_t* o_full = p_full + 2;                   // [2]
  uint64_t* s_free = o_full + 2;                   // [2] softmax has pulled S into registers
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_free + 2);

  const int warp = threadIdx.x >> 5;
  const int qb = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int q0 = qb * 2 * kAttnBQ;
  // key-masked (variable-length) mode: query blocks that lie wholly past the end of their sample are padding rows whose
  // output nobody reads — the CTA leaves at once (kv_len was written long before the preceding kernel).
  if (p.kv_len != nullptr && q0 >= p.kv_len[b]) return;
  const int col_q = h * 64, col_k = p.inner + h * 64, col_v = 2 * p.inner + h * 64;

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmQKV);
    mbar_init(q_full, 1);
    for (int s = 0; s < kAttnStages; ++s) {
      mbar_init(&k_full[s], 1);
      mbar_init(&k_empty[s], 1);
      mbar_init(&v_full[s], 1);
      mbar_init(&v_empty[s], 1);
    }
    for (int w = 0; w < 2; ++w) {
      mbar_init(&s_full[w], 1);
      mbar_init(&p_full[w], 128);
      mbar_init(&o_full[w], 1);
      mbar_init(&s_free[w], 128);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  pdl_launch_dependents();
  // kv_len[b] >= 1 here: a sample with kv_len[b] < 1 (a caller error) left above without writing any output
  const int kv_len = p.kv_len ? max(1, min(p.kv_len[b], p.seq)) : p.seq;
  const int n_kv = (kv_len + kAttnBKV - 1) / kAttnBKV;

  if (warp < 4) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(F5_ATTN_REGS_PRODUCER));
  if (warp == 0) {
    if (elect_one()) {
      mbar_expect_tx(q_full, 2 * kAttnTile);
      tma_load_3d(sQ, &tmQKV, q_full, col_q, q0, b);
      tma_load_3d(sQ + kAttnTile, &tmQKV, q_full, col_q, q0 + kAttnBQ, b);
      for (int j = 0; j < n_kv; ++j) {
        const int s = j % kAttnStages;
        const uint32_t ph = (j / kAttnStages) & 1;
        mbar_wait(&k_empty[s], ph ^ 1);
        mbar_expect_tx(&k_full[s], kAttnTile);
        tma_load_3d(sK + s * kAttnTile, &tmQKV, &k_full[s], col_k, j * kAttnBKV, b);
        mbar_wait(&v_empty[s], ph ^ 1);
        mbar_expect_tx(&v_full[s], kAttnTile);
        tma_load_3d(sV + s * kAttnTile, &tmQKV, &v_full[s], col_v, j * kAttnBKV, b);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc_s = make_idesc_f16(128, 128, 0, 0);  // S = Q K^T : both K-major
      constexpr uint32_t idesc_o = make_idesc_f16(128, 64, 0, 1);   // O = P V   : P from TMEM, V is MN-major
      auto issue_s = [&](int w, int ks) {
        const uint64_t qdesc = make_smem_desc_sw128(smem_u32(sQ + w * kAttnTile));
        const uint64_t kdesc = make_smem_desc_sw128(smem_u32(sK + ks * kAttnTile));
#pragma unroll
        for (int k = 0; k < 4; ++k)
          tc_mma_ss(tmem_base + w * 128, qdesc + uint64_t(2 * k), kdesc + uint64_t(2 * k), idesc_s, k != 0);
        tc_commit(&s_full[w]);
      };
      mbar_wait(q_full, 0);
      mbar_wait(&k_full[0], 0);
      tc_fence_after();
      issue_s(0, 0);
      issue_s(1, 0);
      tc_commit(&k_empty[0]);
      for (int j = 0; j < n_kv; ++j) {
        // S of the NEXT tile is issued as soon as the softmax warps have pulled the current S into registers
        // (s_free), i.e. long before their exponentials / P are done: the Q K^T latency leaves the softmax chain.
        if (j + 1 < n_kv) {
          const int sk = (j + 1) % kAttnStages;
          mbar_wait(&k_full[sk], ((j + 1) / kAttnStages) & 1);
          for (int w = 0; w < 2; ++w) {
            mbar_wait(&s_free[w], j & 1);
            tc_fence_after();
            issue_s(w, sk);
          }
          tc_commit(&k_empty[sk]);
        }
        const int sv = j % kAttnStages;
        // 16-key MMA steps that hold at least one valid key (keys past the end have P = 0 and zero-filled V rows)
        const int kv_rem = kv_len - j * kAttnBKV;
        const int nkk = kv_rem >= kAttnBKV ? 8 : (kv_rem + 15) >> 4;
        mbar_wait(&v_full[sv], (j / kAttnStages) & 1);
        for (int w = 0; w < 2; ++w) {
          mbar_wait(&p_full[w], j & 1);
          tc_fence_after();
          for (int kk = 0; kk < nkk; ++kk) {
            // A = P_w[:, 16 kk .. 16 kk + 15]: 8 TMEM columns of packed fp16 pairs; B = 16 key rows of V (2 KB apart)
            const uint64_t vdesc = make_smem_desc_sw128(smem_u32(sV + sv * kAttnTile + kk * 16 * 128));
            tc_mma_ts(tmem_base + 256 + w * 64, tmem_base + 384 + w * 64 + kk * 8, vdesc, idesc_o, (j | kk) != 0);
          }
          tc_commit(&o_full[w]);
        }
        tc_commit(&v_empty[sv]);
      }
    }
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(F5_ATTN_REGS_SOFTMAX));
    const int w = (warp - 4) >> 2;  // softmax warpgroup 0 / 1
    const int q = warp & 3;         // TMEM lane quarter
    const int row = q * 32 + int(lane_id());
    const uint32_t lane_off = uint32_t(q * 32) << 16;
    const uint32_t tmem_S = tmem_base + w * 128 + lane_off;
    const uint32_t tmem_O = tmem_base + 256 + w * 64 + lane_off;
    const uint32_t tmem_P = tmem_base + 384 + w * 64 + lane_off;
    float m_run = -INFINITY, l_run = 0.0f;
#ifdef F5_TRACE
    long long* ts = p.dbg_ts ? p.dbg_ts + ((long long)(blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 16 + w * 8 : nullptr;
    long long c_s = 0, c_turn = 0, c_exp = 0, c_o = 0, c_p = 0, c0 = 0, c_begin = 0, c_ld = 0, c_max = 0;
    if (ts) c_begin = clock64();
#endif
    // Ping-pong turnstile (named barriers 3 + w, 256 threads): the two warpgroups take turns in the exp2-heavy
    // section, so one warpgroup's MUFU work overlaps the other's max / TMEM traffic instead of both running in lockstep.
    if (p.turnstile && w == 1) named_bar_arrive(3, 256);  // WG0 goes first
    for (int j = 0; j < n_kv; ++j) {
      const int kv_rem = kv_len - j * kAttnBKV;  // valid keys in this tile (>= 1)
#ifdef F5_TRACE
      if (ts) c0 = clock64();
#endif
      mbar_wait(&s_full[w], j & 1);
      tc_fence_after();
#ifdef F5_TRACE
      if (ts) { const long long c1 = clock64(); c_s += c1 - c0; c0 = c1; }
#endif
      uint32_t r0[32], r1[32], r2[32], r3[32];
      tmem_ld32(tmem_S + 0, r0);
      tmem_ld32(tmem_S + 32, r1);
      tmem_ld32(tmem_S + 64, r2);
      tmem_ld32(tmem_S + 96, r3);
      tmem_ld_wait();
#ifdef F5_TRACE
      if (ts) { const long long c1 = clock64(); c_ld += c1 - c0; c0 = c1; }
#endif
      tc_fence_before();
      mbar_arrive(&s_free[w]);  // S_w is in registers: the tensor core may overwrite it with the next tile's scores
      float mx;
      if (kv_rem < kAttnBKV) {
        // warp-uniform, last tile of the sample: only the 32-key chunk that straddles the end is masked element by
        // element; chunks that lie wholly past the end are left out of the max and cost no exponentials below
        // (the full masking pass was 256 instructions — a third of a tile's issue slots — on one tile in eight)
        if (kv_rem < 32) mask_tail32(r0, 0, kv_rem);
        else if (kv_rem < 64) mask_tail32(r1, 32, kv_rem);
        else if (kv_rem < 96) mask_tail32(r2, 64, kv_rem);
        else mask_tail32(r3, 96, kv_rem);
        mx = row_max32(r0);
        if (kv_rem > 32) mx = fmaxf(mx, row_max32(r1));
        if (kv_rem > 64) mx = fmaxf(mx, row_max32(r2));
        if (kv_rem > 96) mx = fmaxf(mx, row_max32(r3));
      } else {
        mx = row_max128(r0, r1, r2, r3);
      }
      const float m_new = fmaxf(m_run, mx * p.scale_log2);
      // lazy rescale (warp-uniform decision because tcgen05.ld/st are warp-collective)
      const bool grow = (m_new - m_run) > 8.0f;  // also true on the first tile (m_run = -inf)
      const bool do_rescale = __any_sync(0xffffffffu, grow);
      float alpha = 1.0f;
      if (do_rescale) {
        alpha = ex2_approx(m_run - m_new);  // first tile: exp2(-inf) = 0
        m_run = m_new;
      }
#ifdef F5_TRACE
      if (ts) { const long long c1 = clock64(); c_max += c1 - c0; c0 = c1; }
#endif
      if (p.turnstile) named_bar_sync(3 + w, 256);  // only the exp2 loop is serialised between the warpgroups
#ifdef F5_TRACE
      if (ts) { const long long c1 = clock64(); c_turn += c1 - c0; c0 = c1; }
#endif
      // exponentials -> packed fp16 (kept in registers until the P columns are free)
      const uint64_t sc2 = f2_pack(p.scale_log2, p.scale_log2);
      const uint64_t nms2 = f2_pack(-m_run, -m_run);
      uint64_t sum2 = f2_pack(0.0f, 0.0f);
      uint32_t pa[32], pb[32];  // keys 0..63 / 64..127 as fp16 pairs = TMEM columns 0..31 / 32..63 of P_w
      exp_pack32<POLY>(r0, 0, kv_rem, sc2, nms2, sum2, pa);
      exp_pack32<POLY>(r1, 32, kv_rem, sc2, nms2, sum2, pa + 16);
      exp_pack32<POLY>(r2, 64, kv_rem, sc2, nms2, sum2, pb);
      exp_pack32<POLY>(r3, 96, kv_rem, sc2, nms2, sum2, pb + 16);
      float ls0, ls1;
      f2_unpack(sum2, ls0, ls1);
      l_run = l_run * alpha + (ls0 + ls1);
      if (p.turnstile) named_bar_arrive(3 + (w ^ 1), 256);  // hand the exp section to the other warpgroup
#ifdef F5_TRACE
      if (ts) { const long long c1 = clock64(); c_exp += c1 - c0; c0 = c1; }
#endif
      if (j > 0) {
        mbar_wait(&o_full[w], (j - 1) & 1);  // P V of the previous tile retired: the P columns and O are ours
        tc_fence_after();
      }
#ifdef F5_TRACE
      if (ts) { const long long c1 = clock64(); c_o += c1 - c0; c0 = c1; }
#endif
      // P -> TMEM (A operand of the P V product): lane = query row, column c holds keys 2c, 2c + 1
      tmem_st32(tmem_P, pa);
      tmem_st32(tmem_P + 32, pb);
      if (do_rescale && j > 0) {
#pragma unroll 1
        for (int c = 0; c < 2; ++c) {
          uint32_t r[32];
          tmem_ld32(tmem_O + uint32_t(c * 32), r);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * alpha);
          tmem_st32(tmem_O + uint32_t(c * 32), r);
        }
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(&p_full[w]);
#ifdef F5_TRACE
      if (ts) c_p += clock64() - c0;
#endif
    }
#ifdef F5_TRACE
    if (ts && row == 0) {
      ts[0] = c_s; ts[1] = c_turn; ts[2] = c_exp; ts[3] = c_o; ts[4] = c_p; ts[5] = clock64() - c_begin; ts[6] = c_max; ts[7] = c_ld;
    }
#endif
    // epilogue: O / l -> fp16
    mbar_wait(&o_full[w], (n_kv - 1) & 1);
    tc_fence_after();
    const float inv_l = 1.0f / l_run;
    const int qrow = q0 + w * kAttnBQ + row;
#pragma unroll 1
    for (int c = 0; c < 2; ++c) {
      uint32_t r[32];
      tmem_ld32(tmem_O + uint32_t(c * 32), r);
      tmem_ld_wait();
      if (qrow < p.seq) {
        __half* o = p.out + ((long long)b * p.seq + qrow) * p.inner + h * 64 + c * 32;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint4 wv;
          wv.x = pack_half2(__uint_as_float(r[8 * g + 0]) * inv_l, __uint_as_float(r[8 * g + 1]) * inv_l);
          wv.y = pack_half2(__uint_as_float(r[8 * g + 2]) * inv_l, __uint_as_float(r[8 * g + 3]) * inv_l);
          wv.z = pack_half2(__uint_as_float(r[8 * g + 4]) * inv_l, __uint_as_float(r[8 * g + 5]) * inv_l);
          wv.w = pack_half2(__uint_as_float(r[8 * g + 6]) * inv_l, __uint_as_float(r[8 * g + 7]) * inv_l);
          reinterpret_cast<uint4*>(o)[g] = wv;
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

}  // namespace f5

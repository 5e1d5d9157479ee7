// Persistent, warp-specialised tcgen05 GEMM / grouped-conv-as-GEMM for sm_100a.
//
//   C[m, n] = epilogue( sum_k A[m, k] * W[n, k] )        A, W fp16, K-major; fp32 accumulation in TMEM.
//
// grid = min(#tiles, #SMs); every CTA walks tiles t = blockIdx.x, +gridDim.x, ... (n fastest, so CTAs that run
// together share the A row-panel in L2 and sweep W once).  Warp roles (320 threads):
//   warp 0        TMA producer (one elected lane): STAGES-deep ring of {A 128x64, W BNx64} fp16 tiles, SWIZZLE_128B
//   warp 1        TMEM allocator + single-thread tcgen05.mma issuer; accumulators double-buffered in TMEM
//                 (2 x BN columns) so the epilogue of tile i overlaps the main loop of tile i+1
//   warps 2..9    epilogue, two column groups of four warps: tcgen05.ld (one accumulator row per thread) -> fused bias /
//                 activation / RoPE / gate / mask -> 128-byte row chunks staged in shared memory (128B swizzle, conflict
//                 free) -> ONE elected thread per group issues a bulk TMA store (fp16 outputs) or a TMA reduce-add (fp32
//                 residual: x += ..., the residual is never read by the SM).  Per-thread scattered global stores were
//                 measured 2.4x slower than the whole main loop.  Warp w owns TMEM lane quarter (w % 4); the second
//                 warp per quarter exists because ONE epilogue warp per scheduler is latency-bound.
// Pipelines: smem full/empty mbarriers (TMA <-> MMA), TMEM acc_full/acc_empty mbarriers (MMA <-> epilogue).
// Tails in M, N and K come from TMA out-of-bounds zero fill plus guarded stores.
//
// CONV mode computes the reference's grouped Conv1d(k=31, groups=16, padding=15) (model/modules.py:175-201)
// as 31 accumulated 128x64x64 GEMMs: tap t multiplies the activation tile shifted by (t - 15) rows — the shift is
// just the TMA row coordinate, and rows outside [0, seq) of the SAME sample are zero-filled by the 3-D tensor map,
// which is exactly the conv's zero padding.
#pragma once
#include "common.cuh"
#include "kparams.h"

namespace f5 {

// Diagnostic kernel modes (skip loads / MMAs / epilogue: WRONG results, timing decomposition only) exist in the
// instrumented build (make TRACE=1) and nowhere else.
#ifdef F5_TRACE
#define F5_DBG(p, mode) ((p).dbg_mode == (mode))
#else
#define F5_DBG(p, mode) false
#endif

constexpr uint32_t kEpiChunkBytes = kBM * 128;  // 128 rows x 128 B (64 fp16 or 32 fp32 columns)
constexpr int kEpiBufs = 2;                     // one staging buffer per epilogue column group

// Epilogue warps per TMEM lane quarter.  ONE warp per scheduler is latency-bound, so activation epilogues (GELU / Mish:
// ~2x the instructions) get a second column group (measured FF1: 14.1 -> 12.4 us at M = 1876, 1025 -> 1196 TFLOP/s at
// M = 15008); the plain / RoPE / reduce-add epilogues were not faster with eight warps (register cap 168, single TMEM
// buffer) and keep four.
__host__ __device__ constexpr int gemm_epi_groups(int /*epi*/, int act) { return act != ACT_NONE ? 2 : 1; }
__host__ __device__ constexpr int gemm_threads(int epi, int act) { return 64 + 128 * gemm_epi_groups(epi, act); }

template <int BN, int STAGES, bool PAIR = false>
constexpr size_t gemm_smem_bytes() {
  return size_t(STAGES) * (kBM * kBK * 2 + (PAIR ? BN / 2 : BN) * kBK * 2) + kEpiBufs * kEpiChunkBytes /*epilogue staging*/ +
         1024 /*align slack*/ + 256 /*barriers*/ + 2048 /*bias + gate staging*/;
}

// fused epilogue for one 32-column chunk of one accumulator row
template <int EPI, int ACT>
__device__ __forceinline__ void epilogue_chunk(const GemmParams& p, const uint32_t (&r)[32], int nc, long long grow,
                                               int pos, bool valid, const float* gate) {
  float v[32];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.bias != nullptr) {
      if (nc + 4 * i + 3 < p.n_out) b = __ldg(reinterpret_cast<const float4*>(p.bias + nc) + i);
      else {
        if (nc + 4 * i + 0 < p.n_out) b.x = __ldg(p.bias + nc + 4 * i + 0);
        if (nc + 4 * i + 1 < p.n_out) b.y = __ldg(p.bias + nc + 4 * i + 1);
        if (nc + 4 * i + 2 < p.n_out) b.z = __ldg(p.bias + nc + 4 * i + 2);
      }
    }
    v[4 * i + 0] = __uint_as_float(r[4 * i + 0]) + b.x;
    v[4 * i + 1] = __uint_as_float(r[4 * i + 1]) + b.y;
    v[4 * i + 2] = __uint_as_float(r[4 * i + 2]) + b.z;
    v[4 * i + 3] = __uint_as_float(r[4 * i + 3]) + b.w;
  }
  if (EPI == EPI_QKV_ROPE) {
    const int sec = nc / p.inner;
    const int head = (nc % p.inner) / 64;
    if (sec < 2 && head < p.pe_heads) {
      const int pair0 = (nc % 64) / 2;
      const float4* cs = reinterpret_cast<const float4*>(p.rope_cos + (long long)pos * 32 + pair0);
      const float4* sn = reinterpret_cast<const float4*>(p.rope_sin + (long long)pos * 32 + pair0);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 c4 = __ldg(cs + i), s4 = __ldg(sn + i);
        const float cc[4] = {c4.x, c4.y, c4.z, c4.w}, ss[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float x0 = v[8 * i + 2 * j], x1 = v[8 * i + 2 * j + 1];
          v[8 * i + 2 * j] = x0 * cc[j] - x1 * ss[j];
          v[8 * i + 2 * j + 1] = x1 * cc[j] + x0 * ss[j];
        }
      }
    }
  }
  if (ACT != ACT_NONE) {
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      if (ACT == ACT_GELU_TANH) v[i] = gelu_tanh(v[i]);
      if (ACT == ACT_GELU_ERF) v[i] = gelu_erf(v[i]);
      if (ACT == ACT_MISH) v[i] = mish(v[i]);
    }
  }
  const bool full_chunk = (nc + 32 <= p.n_out);
  if (EPI == EPI_F16 || EPI == EPI_QKV_ROPE) {
    __half* o = reinterpret_cast<__half*>(p.out) + grow * p.ldo + nc;
    if (full_chunk && (p.ldo % 8 == 0)) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        uint4 w;
        w.x = valid ? pack_half2(v[8 * i + 0], v[8 * i + 1]) : 0u;
        w.y = valid ? pack_half2(v[8 * i + 2], v[8 * i + 3]) : 0u;
        w.z = valid ? pack_half2(v[8 * i + 4], v[8 * i + 5]) : 0u;
        w.w = valid ? pack_half2(v[8 * i + 6], v[8 * i + 7]) : 0u;
        reinterpret_cast<uint4*>(o)[i] = w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i)  // static indices only: a dynamic index would push v[] into local memory
        if (nc + i < p.n_out) o[i] = __float2half_rn(valid ? v[i] : 0.0f);
    }
  } else if (EPI == EPI_F32) {
    float* o = reinterpret_cast<float*>(p.out) + grow * p.ldo + nc;
    if (full_chunk && (p.ldo % 4 == 0)) {
#pragma unroll
      for (int i = 0; i < 8; ++i)
        reinterpret_cast<float4*>(o)[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (nc + i < p.n_out) o[i] = v[i];
    }
    if (p.out16b != nullptr) {
      __half* o2 = p.out16b + grow * p.ldo + nc;
      if (full_chunk && (p.ldo % 8 == 0)) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          uint4 w;
          w.x = valid ? pack_half2(v[8 * i + 0], v[8 * i + 1]) : 0u;
          w.y = valid ? pack_half2(v[8 * i + 2], v[8 * i + 3]) : 0u;
          w.z = valid ? pack_half2(v[8 * i + 4], v[8 * i + 5]) : 0u;
          w.w = valid ? pack_half2(v[8 * i + 6], v[8 * i + 7]) : 0u;
          reinterpret_cast<uint4*>(o2)[i] = w;
        }
      } else {
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          if (nc + i + 1 < p.n_out) *reinterpret_cast<uint32_t*>(o2 + i) = valid ? pack_half2(v[i], v[i + 1]) : 0u;
          else if (nc + i < p.n_out) o2[i] = __float2half_rn(valid ? v[i] : 0.0f);  // odd n_out: column n_out is not ours
        }
      }
    }
  } else if (EPI == EPI_RESID) {
    float* o = p.resid + grow * p.ldo + nc;
    if (!valid) return;
    if (full_chunk && (p.ldo % 4 == 0)) {
      float4 x[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = reinterpret_cast<const float4*>(o)[i];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float4 g = make_float4(1.f, 1.f, 1.f, 1.f);
        if (gate != nullptr) g = __ldg(reinterpret_cast<const float4*>(gate + nc) + i);
        x[i].x += g.x * v[4 * i];
        x[i].y += g.y * v[4 * i + 1];
        x[i].z += g.z * v[4 * i + 2];
        x[i].w += g.w * v[4 * i + 3];
        reinterpret_cast<float4*>(o)[i] = x[i];
      }
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (nc + i < p.n_out) o[i] += (gate ? gate[nc + i] : 1.0f) * v[i];
    }
  }
}

// Packed / variable-length execution (SURVEY.md §8f-1; reference masked mode modules.py:513-540): with skip_pad, a tile
// whose rows ALL lie past the end of their sample is never loaded, multiplied or stored.  Every warp role evaluates the
// same predicate, so the smem ring, the TMEM double buffer and the tile order stay in step.  m0 = first row of the
// (pair-)tile, tm = its height; CONV: rows are per sample (bz), plain: rows are the flattened [samples x seq] axis.
template <bool CONV>
__device__ __forceinline__ bool tile_is_padding(const GemmParams& p, int m0, int tm, int bz) {
  if (!p.skip_pad) return false;
  if (CONV) return m0 >= p.row_len[bz];
  const int last = min(m0 + tm, p.rows) - 1;
  const int b0 = m0 / p.seq;
  if (b0 != last / p.seq) return false;  // the tile reaches into the next sample, whose first rows are valid
  return m0 - b0 * p.seq >= p.row_len[b0];
}

// PAIR = true: cta_group::2.  Two CTAs of a cluster (same TPC) compute one 256 x BN tile: each CTA stages its own 128
// rows of A and HALF of the W tile (BN/2 rows), the leader CTA issues tcgen05.mma.cta_group::2 (M = 256) for both, and
// each CTA's accumulator half lands in its own TMEM.  Shared-memory traffic per MMA cycle drops by 1/4 (BN = 256) —
// the measured limiter of the single-CTA kernel (operand writes by TMA + reads by the tensor core > 128 B/clk).
template <int BN, int STAGES, int EPI, int ACT, bool CONV, bool PAIR = false>
__global__ void __launch_bounds__(gemm_threads(EPI, ACT), 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmC, const GemmParams p) {
  static_assert(!(PAIR && CONV), "the conv schedule is single-CTA");
  constexpr int BNL = PAIR ? BN / 2 : BN;  // W rows staged by this CTA
  constexpr int TM = PAIR ? 2 * kBM : kBM;  // rows of one (pair-)tile
  constexpr uint32_t A_BYTES = kBM * kBK * 2;
  constexpr uint32_t B_BYTES = BNL * kBK * 2;
  constexpr uint32_t TMEM_COLS = (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;  // double-buffered accumulator
  static_assert(BN == 64 || BN == 128 || BN == 192 || BN == 256, "BN");
  static_assert(!(PAIR && BN == 64), "pair tiles are 128, 192 or 256 wide");

  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * A_BYTES;
  uint8_t* sC = smem + STAGES * (A_BYTES + B_BYTES);  // kEpiBufs x 16 KB epilogue staging (1024-aligned)
  uint64_t* full = reinterpret_cast<uint64_t*>(sC + kEpiBufs * kEpiChunkBytes);
  uint64_t* empty = full + STAGES;
  uint64_t* acc_full = empty + STAGES;  // [2]
  uint64_t* acc_empty = acc_full + 2;   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  float* sBias = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full) + 256);  // [256] bias of the current tile
  float* sGate = sBias + 256;                                                         // [256] gate of the current tile

  const int warp = threadIdx.x >> 5;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0;       // 0 = leader CTA of the pair
  const int cta_id = PAIR ? int(blockIdx.x >> 1) : int(blockIdx.x);
  const int cta_step = PAIR ? int(gridDim.x >> 1) : int(gridDim.x);
#ifdef F5_TRACE
  long long* ts = p.dbg_ts ? p.dbg_ts + (long long)blockIdx.x * 16 : nullptr;
#endif
#ifdef F5_TRACE
  if (ts && threadIdx.x == 0) {
    unsigned long long g;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
    ts[0] = (long long)g;
    ts[1] = clock64();
  }
#endif
  const int tiles_n = (p.n_out + BN - 1) / BN;
  const int tiles_m = (p.rows + TM - 1) / TM;
  const int num_tiles = tiles_n * tiles_m * p.batches;

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (EPI != EPI_F32) tma_prefetch_desc(&tmC);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&acc_full[b], 1);
      mbar_init(&acc_empty[b], (PAIR ? 2 : 1) * 128 * gemm_epi_groups(EPI, ACT));  // PAIR: both CTAs' epilogue threads arrive on the leader's barrier
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    if (PAIR) tmem_alloc_pair(tmem_slot, TMEM_COLS);
    else tmem_alloc(tmem_slot, TMEM_COLS);
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all();  // peer barriers are initialised before any remote arrive / multicast commit
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // Programmatic dependent launch: everything above overlapped the predecessor's tail.  The producer thread goes one
  // step further (below): W tiles are weights, not produced by the predecessor, so their TMA loads are issued BEFORE
  // the dependency wait and the DRAM latency of the first STAGES k-blocks hides under the predecessor too.
  if (warp != 0) pdl_wait();  // predecessor kernel finished: its outputs (our A operand, residual, ...) are visible
  pdl_launch_dependents();    // let the next kernel's prologue overlap our tail
#ifdef F5_TRACE
  if (ts && threadIdx.x == 0) ts[2] = clock64();  // setup done
#endif

  if (warp == 0) {
    if (elect_one()) {
      // ===== TMA producer =====
      uint32_t it = 0;  // running k-block counter across tiles -> stage / phase
      // W tile of k-block kb of the tile at column n0 -> stage s (barrier already armed)
      auto load_w = [&](int s, int kb, int n0) {
        if (PAIR) tma_load_2d_pair(sB + s * B_BYTES, &tmB, mapa_u32(&full[s], 0), kb * kBK, n0 + int(rank) * BNL);
        else if (CONV) tma_load_2d(sB + s * B_BYTES, &tmB, &full[s], 0, kb * p.n_out + n0);  // [tap][out_channel][in 64]
        else tma_load_2d(sB + s * B_BYTES, &tmB, &full[s], kb * kBK, n0);
      };
      auto arm = [&](int s) {
        // PAIR: both CTAs load; every byte is credited to the LEADER's full barrier, which the MMA issuer waits on
        if (PAIR) {
          if (rank == 0) mbar_expect_tx(&full[s], 2 * (A_BYTES + B_BYTES));
        } else {
          mbar_expect_tx(&full[s], A_BYTES + B_BYTES);
        }
      };
      // weights of the first tile's first k-blocks: in flight before the dependency wait (slots are free at start)
      uint32_t pre = 0;
      if (cta_id < num_tiles && !F5_DBG(p, 1) && p.w_prefetch) {
        pre = uint32_t(p.num_kb < STAGES ? p.num_kb : STAGES);
        for (uint32_t kb = 0; kb < pre; ++kb) {
          arm(int(kb));
          load_w(int(kb), int(kb), (cta_id % tiles_n) * BN);
        }
      }
      pdl_wait();
      for (int t = cta_id; t < num_tiles; t += cta_step) {
        const int n0 = (t % tiles_n) * BN;
        const int m0 = ((t / tiles_n) % tiles_m) * TM + int(rank) * kBM;
        const int bz = t / (tiles_n * tiles_m);
        if (tile_is_padding<CONV>(p, ((t / tiles_n) % tiles_m) * TM, TM, bz)) continue;
        for (int kb = 0; kb < p.num_kb; ++kb, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1;
          if (it >= pre) {
            mbar_wait(&empty[s], ph ^ 1);
            if (F5_DBG(p, 1)) {
              mbar_arrive(&full[s]);
              continue;
            }
            arm(s);
            load_w(s, kb, n0);
          }
          if (PAIR) tma_load_3d_pair(sA + s * A_BYTES, &tmA, mapa_u32(&full[s], 0), kb * kBK, m0, bz);
          else if (CONV) tma_load_3d(sA + s * A_BYTES, &tmA, &full[s], n0, m0 + kb - p.conv_pad, bz);  // tap shift
          else tma_load_3d(sA + s * A_BYTES, &tmA, &full[s], kb * kBK, m0, bz);
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0 && elect_one()) {
      // ===== MMA issuer (leader CTA only when PAIR) =====
      constexpr uint32_t idesc = make_idesc_f16(TM, BN, 0, 0);
      uint32_t it = 0, tl = 0;
      for (int t = cta_id; t < num_tiles; t += cta_step) {
        if (tile_is_padding<CONV>(p, ((t / tiles_n) % tiles_m) * TM, TM, t / (tiles_n * tiles_m))) continue;
        const uint32_t buf = tl & 1;
        mbar_wait(&acc_empty[buf], ((tl >> 1) & 1) ^ 1);  // epilogue drained this accumulator
        tc_fence_after();
        const uint32_t tmem_acc = tmem_base + buf * BN;
        for (int kb = 0; kb < p.num_kb; ++kb, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1;
          mbar_wait(&full[s], ph);
#ifdef F5_TRACE
          if (ts && it == 0) ts[3] = clock64();  // first operands landed
#endif
          tc_fence_after();
          const uint64_t adesc = make_smem_desc_sw128(smem_u32(sA + s * A_BYTES));
          const uint64_t bdesc = make_smem_desc_sw128(smem_u32(sB + s * B_BYTES));
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k) {
            if (F5_DBG(p, 2)) break;
            // +32 bytes (16 fp16) along K inside the 128B swizzle atom = +2 in the (addr >> 4) field
            if (PAIR) tc_mma_ss_pair(tmem_acc, adesc + uint64_t(k * 2), bdesc + uint64_t(k * 2), idesc, (kb | k) != 0);
            else tc_mma_ss(tmem_acc, adesc + uint64_t(k * 2), bdesc + uint64_t(k * 2), idesc, (kb | k) != 0);
          }
          if (PAIR) tc_commit_pair(&empty[s]);  // frees the slot in BOTH CTAs once these MMAs retire
          else tc_commit(&empty[s]);
        }
        if (PAIR) tc_commit_pair(&acc_full[buf]);
        else tc_commit(&acc_full[buf]);
        ++tl;
      }
#ifdef F5_TRACE
      if (ts) ts[4] = clock64();  // all MMAs issued
#endif
    }
  } else {
    // ===== epilogue: warps 2.. (4 * EG warps).  Warp w reads TMEM lane quarter w % 4 (rows); with EG = 2 column group
    // eg = (w - 2) / 4 takes every other 128-byte chunk of the tile, so two warps per scheduler hide each other's
    // latencies (a lone warp needs ~860 clk per 32-column piece for ~200 issue slots).
    constexpr int EG = gemm_epi_groups(EPI, ACT);
    constexpr int ETH = 128 * EG;  // epilogue threads
    const int q = warp & 3;
    const int eg = (EG == 2) ? (warp - 2) >> 2 : 0;
    const int et = int(threadIdx.x) - 64;                 // 0 .. ETH-1
    const bool issuer = (et == eg * 128);                 // owns this group's bulk stores
    const int bar_a = 1 + 2 * eg, bar_b = 2 + 2 * eg;     // named barriers of this column group (128 threads)
    // Staging buffers: two column groups own one buffer each; a single group (EG = 1) uses BOTH as a ring, so the bulk
    // store of chunk c reads its buffer while chunk c + 1 is already being written into the other one.
    uint32_t cc = 0;                                      // running chunk counter of this group (EG = 1 ring index)
    const float* gate = nullptr;
    if (EPI == EPI_RESID && p.gate != nullptr)
      gate = p.gate + (p.step_ptr ? (long long)(*p.step_ptr) : 0) * p.gate_step_stride;
    uint32_t tl = 0;
#ifdef F5_TRACE
    long long t_accwait = 0;
#endif
    for (int t = cta_id; t < num_tiles; t += cta_step) {
      const int n0 = (t % tiles_n) * BN;
      const int m0 = ((t / tiles_n) % tiles_m) * TM + int(rank) * kBM;
      const int bz = t / (tiles_n * tiles_m);
      if (tile_is_padding<CONV>(p, ((t / tiles_n) % tiles_m) * TM, TM, bz)) continue;
      const uint32_t buf = tl & 1;
      const int row_in_batch = m0 + q * 32 + int(lane_id());
      const bool row_ok = row_in_batch < p.rows;
      const long long grow = (long long)bz * p.rows + row_in_batch;
      bool valid = row_ok;
      int pos = 0;
      if (p.seq > 0) {
        pos = int(grow % p.seq);
        if (p.row_len != nullptr && row_ok) valid = pos < p.row_len[grow / p.seq];
      }
      // ---- prefetch everything the epilogue reads from global memory while the main loop of this tile runs ----
      float4 rope_c[8], rope_s[8];
      if (EPI != EPI_F32) {
        named_bar_sync(5, ETH);  // every thread is done with the previous tile's sBias / sGate
#pragma unroll
        for (int c = et; c < BN; c += ETH) {
          const int n = n0 + c;
          sBias[c] = (p.bias != nullptr && n < p.n_out) ? __ldg(p.bias + n) : 0.0f;
          if (EPI == EPI_RESID) sGate[c] = (gate != nullptr && n < p.n_out) ? __ldg(gate + n) : 1.0f;
        }
        if (EPI == EPI_QKV_ROPE) {
          const float4* cs = reinterpret_cast<const float4*>(p.rope_cos + (long long)pos * 32);
          const float4* sn = reinterpret_cast<const float4*>(p.rope_sin + (long long)pos * 32);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            rope_c[i] = __ldg(cs + i);
            rope_s[i] = __ldg(sn + i);
          }
        }
      }
#ifdef F5_TRACE
      long long ta0 = 0;
#endif
#ifdef F5_TRACE
      if (ts) ta0 = clock64();
#endif
      mbar_wait(&acc_full[buf], (tl >> 1) & 1);
#ifdef F5_TRACE
      if (ts) t_accwait += clock64() - ta0;
#endif
#ifdef F5_TRACE
      if (ts && tl == 0 && threadIdx.x == 64) ts[5] = clock64();  // first accumulator complete
#endif
      tc_fence_after();
      const uint32_t tmem_acc = tmem_base + buf * BN + (uint32_t(q * 32) << 16);
      if (EPI == EPI_F32) {
        // direct stores (used once per step for the input projection: fp32 + masked fp16 copy)
#pragma unroll 1
        for (int c = eg; c < BN / 32; c += EG) {
          uint32_t r[32];
          tmem_ld32(tmem_acc + uint32_t(c * 32), r);
          tmem_ld_wait();
          const int nc = n0 + c * 32;
          if (row_ok && nc < p.n_out && !F5_DBG(p, 3)) epilogue_chunk<EPI, ACT>(p, r, nc, grow, pos, valid, gate);
        }
      } else {
        // staged: 32-column pieces -> 128-byte row chunks in swizzled smem -> bulk TMA store / reduce-add.
        // All global reads the epilogue needs (bias, gate, rotary rows) were issued BEFORE the accumulator wait, TMEM
        // loads are double-buffered, and a chunk's values wait in registers until the group's staging buffer has been
        // read by the previous bulk store, so no DRAM / L2 / TMEM / TMA latency sits on the per-chunk path.
        constexpr int PIECES = BN / 32;
        constexpr int PPC = (EPI == EPI_RESID) ? 1 : 2;  // pieces per 128-byte chunk
        constexpr int NCH = PIECES / PPC;                // chunks per tile
        constexpr int NCHG = (NCH + EG - 1) / EG;        // chunks per column group (upper bound)
        constexpr bool DB = true;                        // TMEM loads double-buffered
        named_bar_sync(6, ETH);                          // sBias / sGate of this tile are published
        const int erow = q * 32 + int(lane_id());
        uint32_t ra[32], rb[32];
        if (eg < NCH) tmem_ld32(tmem_acc + uint32_t(eg * PPC * 32), ra);
#pragma unroll
        for (int i = 0; i < NCHG; ++i) {
          const int ch = eg + EG * i;
          if (ch < NCH) {
            uint32_t st[32];  // RESID: 32 fp32 values ; fp16: 2 x 16 packed pairs
#pragma unroll
            for (int sub = 0; sub < PPC; ++sub) {
              const int k = i * PPC + sub;  // running piece counter of this group (compile time)
              uint32_t(&rc)[32] = (DB && (k & 1)) ? rb : ra;
              uint32_t(&rn)[32] = (DB && !(k & 1)) ? rb : ra;
              const int pc = ch * PPC + sub;
              const int pc_next = (sub + 1 < PPC) ? pc + 1 : (ch + EG) * PPC;
              const bool has_next = (sub + 1 < PPC) || (ch + EG < NCH);
              tmem_ld_wait();
              if (DB && has_next) tmem_ld32(tmem_acc + uint32_t(pc_next * 32), rn);
              const int ct = pc * 32;  // column inside the tile
              float v[32];
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float4 bb = *reinterpret_cast<const float4*>(sBias + ct + 4 * j);
                v[4 * j + 0] = __uint_as_float(rc[4 * j + 0]) + bb.x;
                v[4 * j + 1] = __uint_as_float(rc[4 * j + 1]) + bb.y;
                v[4 * j + 2] = __uint_as_float(rc[4 * j + 2]) + bb.z;
                v[4 * j + 3] = __uint_as_float(rc[4 * j + 3]) + bb.w;
              }
              if (!DB && has_next) tmem_ld32(tmem_acc + uint32_t(pc_next * 32), ra);  // rc == ra has been consumed into v
              if (EPI == EPI_QKV_ROPE) {
                const int nc = n0 + ct;
                const int sec = nc / p.inner, head = (nc % p.inner) / 64;
                if (sec < 2 && head < p.pe_heads) {
                  // pairs 0..15 of the head for its first 32 columns, pairs 16..31 for the second
#pragma unroll
                  for (int j = 0; j < 4; ++j) {
                    const float4 c4 = rope_c[(nc % 64) ? 4 + j : j], s4 = rope_s[(nc % 64) ? 4 + j : j];
                    const float cc[4] = {c4.x, c4.y, c4.z, c4.w}, ss[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                      const float x0 = v[8 * j + 2 * u], x1 = v[8 * j + 2 * u + 1];
                      v[8 * j + 2 * u] = x0 * cc[u] - x1 * ss[u];
                      v[8 * j + 2 * u + 1] = x1 * cc[u] + x0 * ss[u];
                    }
                  }
                }
              }
              if (ACT != ACT_NONE) {
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                  if (ACT == ACT_GELU_TANH) v[j] = gelu_tanh(v[j]);
                  if (ACT == ACT_GELU_ERF) v[j] = gelu_erf(v[j]);
                  if (ACT == ACT_MISH) v[j] = mish(v[j]);
                }
              }
              if (EPI == EPI_RESID) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const float4 g = *reinterpret_cast<const float4*>(sGate + ct + 4 * j);
                  st[4 * j + 0] = __float_as_uint(valid ? g.x * v[4 * j] : 0.f);
                  st[4 * j + 1] = __float_as_uint(valid ? g.y * v[4 * j + 1] : 0.f);
                  st[4 * j + 2] = __float_as_uint(valid ? g.z * v[4 * j + 2] : 0.f);
                  st[4 * j + 3] = __float_as_uint(valid ? g.w * v[4 * j + 3] : 0.f);
                }
              } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) st[sub * 16 + j] = valid ? pack_half2(v[2 * j], v[2 * j + 1]) : 0u;
              }
            }
            uint8_t* sbuf = sC + (EG == 2 ? uint32_t(eg) : (cc & 1u)) * kEpiChunkBytes;
            ++cc;
            if (issuer) {  // the bulk store that last read THIS buffer has finished reading it
              if (EG == 2) tma_store_wait_read<0>();
              else tma_store_wait_read<1>();
            }
            named_bar_sync(bar_a, 128);
            uint8_t* srow = sbuf + erow * 128;
#pragma unroll
            for (int j = 0; j < 8; ++j)
              *reinterpret_cast<uint4*>(srow + ((j ^ (erow & 7)) << 4)) =
                  make_uint4(st[4 * j], st[4 * j + 1], st[4 * j + 2], st[4 * j + 3]);
            fence_proxy_async_smem();
            named_bar_sync(bar_b, 128);
            if (issuer && !F5_DBG(p, 3)) {
              const int c0 = n0 + ch * (32 * PPC);
              if (c0 < p.n_out) {
                if (EPI == EPI_RESID) tma_reduce_add_3d(&tmC, sbuf, c0, m0, bz);
                else tma_store_3d(&tmC, sbuf, c0, m0, bz);
              }
              tma_store_commit();
            }
          }
        }
      }
      tc_fence_before();
      if (PAIR) mbar_arrive_cluster(mapa_u32(&acc_empty[buf], 0));  // the leader's MMA issuer owns the accumulator ring
      else mbar_arrive(&acc_empty[buf]);
      ++tl;
    }
#ifdef F5_TRACE
    if (ts && threadIdx.x == 64) ts[12] = clock64();
#endif
    if (EPI != EPI_F32 && issuer) {
      tma_store_wait_read<0>();  // smem must outlive the last bulk store
    }
#ifdef F5_TRACE
    if (ts && threadIdx.x == 64) {
      ts[6] = clock64();  // epilogue done
      ts[11] = t_accwait;
    }
#endif
  }

  tc_fence_before();
  if (PAIR) cluster_sync_all();  // the peer may still be consuming our smem / signalling our barriers
  else __syncthreads();
#ifdef F5_TRACE
  if (ts && threadIdx.x == 0) ts[7] = clock64();
#endif
  if (warp == 1) {
    if (PAIR) tmem_dealloc_pair(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

}  // namespace f5

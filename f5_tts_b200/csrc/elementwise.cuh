// Bandwidth-bound kernels of the ODE-sampling path: row normalisations (+AdaLN modulation), depthwise conv + LN,
// text embedding gather, GRN, input packing, CFG + ODE update, small fp32 linears, rotary tables.
// All are warp-per-row / grid-stride kernels with 128-bit vectorised, coalesced global accesses.
#pragma once
#include "common.cuh"
#include "ew_params.h"

namespace f5 {

// ---------------------------------------------------------------------------------------------------------
// Row norm + modulation: x fp32 [rows, D] -> out fp16 [rows, D].  One warp per row, row kept in registers.
//   MODE 0: LayerNorm(eps, no affine) * (1 + scale[c]) + shift[c]     (modules.py:312-326, 333-347, 753)
//   MODE 1: LayerNorm(eps) * w[c] + b[c]                               (ConvNeXt / Vocos norms)
//   MODE 2: x / max(||x||, 1e-12) * sqrt(D) * g[c]                     (x_transformers RMSNorm, unett.py:154)
// scale/shift live in the per-step modulation table: ptr + (*step_ptr) * step_stride.
// ---------------------------------------------------------------------------------------------------------

template <int MODE>
__global__ void __launch_bounds__(256) row_norm_kernel(const NormParams p) {
  pdl_launch_dependents();
  const int row = blockIdx.x * int(blockDim.x >> 5) + (threadIdx.x >> 5);  // one warp per row
  const int lane = lane_id();
  const int nv = p.D >> 7;  // float4 per lane (D multiple of 128, <= 1024)
  float4 v[8], ga[8], gb[8];
  float s = 0.f;
  // Scale / shift of this step: inside the engine they were written long before the producer of x (modulation table,
  // step counter of the previous NFE step), so they are fetched BEFORE the programmatic-launch dependency wait — the
  // block is already resident while the residual GEMM is still running, and only the x rows are left to read after it.
  auto load_params = [&]() {
    const long long so = p.step_ptr ? (long long)(*p.step_ptr) * p.step_stride : 0;
    const float4* A = reinterpret_cast<const float4*>(p.a + so);
    const float4* B = (MODE == 2) ? nullptr : reinterpret_cast<const float4*>(p.b + so);
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (i < nv) {
        ga[i] = __ldg(A + i * 32 + lane);
        if (MODE != 2) gb[i] = __ldg(B + i * 32 + lane);
      }
  };
  if (p.params_static && row < p.rows) load_params();
  pdl_wait();
  if (row >= p.rows) return;
  const float4* xr = reinterpret_cast<const float4*>(p.x + (long long)row * p.D);
  // issue every remaining global load up front: one exposed L2 latency
#pragma unroll
  for (int i = 0; i < 8; ++i)
    if (i < nv) v[i] = xr[i * 32 + lane];
  if (!p.params_static) load_params();
#pragma unroll
  for (int i = 0; i < 8; ++i)
    if (i < nv) s += v[i].x + v[i].y + v[i].z + v[i].w;
  float mean = 0.f, rstd;
  if (MODE != 2) {
    mean = warp_sum(s) / float(p.D);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (i < nv) {
        float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
        q += a * a + b * b + c * c + d * d;
      }
    rstd = rsqrtf(warp_sum(q) / float(p.D) + p.eps);
  } else {
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (i < nv) q += v[i].x * v[i].x + v[i].y * v[i].y + v[i].z * v[i].z + v[i].w * v[i].w;
    rstd = sqrtf(float(p.D)) / fmaxf(sqrtf(warp_sum(q)), 1e-12f);
  }
  uint2* o = reinterpret_cast<uint2*>(p.out + (long long)row * p.D);
#pragma unroll
  for (int i = 0; i < 8; ++i)
    if (i < nv) {
      const float4 a = ga[i];
      float4 r;
      if (MODE == 0) {
        const float4 b = gb[i];
        r.x = (v[i].x - mean) * rstd * (1.f + a.x) + b.x;
        r.y = (v[i].y - mean) * rstd * (1.f + a.y) + b.y;
        r.z = (v[i].z - mean) * rstd * (1.f + a.z) + b.z;
        r.w = (v[i].w - mean) * rstd * (1.f + a.w) + b.w;
      } else if (MODE == 1) {
        const float4 b = gb[i];
        r.x = (v[i].x - mean) * rstd * a.x + b.x;
        r.y = (v[i].y - mean) * rstd * a.y + b.y;
        r.z = (v[i].z - mean) * rstd * a.z + b.z;
        r.w = (v[i].w - mean) * rstd * a.w + b.w;
      } else {
        r.x = v[i].x * rstd * a.x;
        r.y = v[i].y * rstd * a.y;
        r.z = v[i].z * rstd * a.z;
        r.w = v[i].w * rstd * a.w;
      }
      o[i * 32 + lane] = make_uint2(pack_half2(r.x, r.y), pack_half2(r.z, r.w));
    }
}

// ---------------------------------------------------------------------------------------------------------
// Depthwise Conv1d(k=7, pad=3, groups=C) along the sequence + bias, then LayerNorm(affine) -> fp16.
// ConvNeXt-V2 text blocks (modules.py:261-268) and Vocos blocks.  x fp32 [B, N, C]; one warp per (b, n) row.
// ---------------------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(256) dwconv7_ln_kernel(const DwConvLnParams p) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= p.B * p.N) return;
  const int lane = lane_id();
  const int b = row / p.N, n = row % p.N;
  const int per = p.C >> 5;  // channels per lane (C multiple of 32, <= 512 -> per <= 16)
  float acc[16];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i)
    if (i < per) {
      const int c = i * 32 + lane;
      float a = __ldg(p.wb + c);
#pragma unroll
      for (int t = 0; t < 7; ++t) {
        const int nn = n + t - 3;
        if (nn >= 0 && nn < p.N) a += __ldg(p.w + c * 7 + t) * p.x[((long long)b * p.N + nn) * p.C + c];
      }
      acc[i] = a;
      s += a;
    }
  const float mean = warp_sum(s) / float(p.C);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i)
    if (i < per) q += (acc[i] - mean) * (acc[i] - mean);
  const float rstd = rsqrtf(warp_sum(q) / float(p.C) + p.eps);
#pragma unroll
  for (int i = 0; i < 16; ++i)
    if (i < per) {
      const int c = i * 32 + lane;
      p.out[(long long)row * p.C + c] = __float2half_rn((acc[i] - mean) * rstd * __ldg(p.ln_w + c) + __ldg(p.ln_b + c));
    }
}

// ---------------------------------------------------------------------------------------------------------
// Text embedding gather (backbones/dit.py:86-121, unett.py:55-70): ids (+1, crop/pad to N, per-sample valid
// length), optional drop (all-zero ids), + absolute sin/cos position table.  Writes fp32 [2B, N, Td]
// (first B = cond variant, last B = uncond variant) and the filler mask (text == 0 BEFORE drop) [B, N].
// ---------------------------------------------------------------------------------------------------------

__global__ void text_gather_kernel(const TextGatherParams p) {
  const int row = blockIdx.x;  // over 2B*N
  const int variant = row / (p.B * p.N);
  const int r = row % (p.B * p.N);
  const int b = r / p.N, n = r % p.N;
  const bool valid = p.valid_len == nullptr || n < p.valid_len[b];
  long long id = 0;
  if (n < p.nt && valid) id = p.ids[(long long)b * p.nt + n] + 1;
  id = id < 0 ? 0 : (id >= p.num_embeds ? p.num_embeds - 1 : id);  // never read outside the table
  if (variant == 0 && threadIdx.x == 0) p.filler[r] = (id == 0) ? 1 : 0;
  if (variant == 1) id = 0;
  const int half = p.Td / 2;
  for (int c = threadIdx.x; c < p.Td; c += blockDim.x) {
    float v = valid ? p.table[id * p.Td + c] : 0.f;
    if (p.add_pos && valid) {
      const int i = c < half ? c : c - half;
      const float freq = 1.0f / powf(10000.0f, float(2 * i) / float(p.Td));
      const float ang = float(n) * freq;
      v += (c < half) ? cosf(ang) : sinf(ang);
    }
    p.out[(long long)row * p.Td + c] = v;
  }
}

// rows where filler[b, n] != 0 are zeroed (text_mask_padding, dit.py:123-127); x fp32 [2B, N, C]
__global__ void mask_rows_kernel(float* x, const uint8_t* filler, int BN, int rows, int C) {
  const int row = blockIdx.x;
  if (row >= rows) return;
  if (filler[row % BN] == 0) return;
  for (int c = threadIdx.x; c < C; c += blockDim.x) x[(long long)row * C + c] = 0.f;
}

// rows at or past the valid length of their sample are zeroed: x [variants * B, N, C], valid_len [B]
template <typename T>
__global__ void mask_rows_len_kernel(T* x, const int* valid_len, int B, int N, int rows, int C) {
  const int row = blockIdx.x;
  if (row >= rows) return;
  const int b = (row / N) % B, n = row % N;
  if (n < valid_len[b]) return;
  for (int c = threadIdx.x; c < C; c += blockDim.x) x[(long long)row * C + c] = T(0.f);
}

// ---------------------------------------------------------------------------------------------------------
// GRN (modules.py:236-245): Gx[b,c] = ||g[b,:,c]||_2 over the SEQUENCE; Nx = Gx / (mean_c Gx + 1e-6);
// g <- gamma * (g * Nx) + beta + g.   g fp16 [B, N, C].
// ---------------------------------------------------------------------------------------------------------
__global__ void grn_sumsq_kernel(const __half* g, float* partial, int N, int C, int rows_per_block) {
  // grid (ceil(C/256), nblk = ceil(N/rows_per_block), B); thread = channel.  partial[b][blk][c], no atomics:
  // the reduction order is fixed, so results are bit-reproducible run to run.
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.z;
  if (c >= C) return;
  const int n0 = blockIdx.y * rows_per_block;
  const int n1 = min(N, n0 + rows_per_block);
  float s = 0.f;
  for (int n = n0; n < n1; ++n) {
    const float v = __half2float(g[((long long)b * N + n) * C + c]);
    s += v * v;
  }
  partial[((long long)b * gridDim.y + blockIdx.y) * C + c] = s;
}

__global__ void grn_finalize_kernel(const float* partial, int nblk, float* nx, int C) {
  // one block per sample: Gx[c] = sqrt(sum_blk partial), Nx = Gx / (mean_c Gx + 1e-6)
  __shared__ float red[32];
  extern __shared__ float gx[];
  const int b = blockIdx.x;
  float s = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float t = 0.f;
    for (int k = 0; k < nblk; ++k) t += partial[((long long)b * nblk + k) * C + c];
    const float r = sqrtf(t);
    gx[c] = r;
    s += r;
  }
  s = warp_sum(s);
  if (lane_id() == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0) red[0] = t / float(C);
  }
  __syncthreads();
  const float mean = red[0];
  for (int c = threadIdx.x; c < C; c += blockDim.x) nx[(long long)b * C + c] = gx[c] / (mean + 1e-6f);
}

__global__ void grn_apply_kernel(__half* g, const float* nx, const float* gamma, const float* beta, int N, int C,
                                 long long total) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = int(i % C);
    const int b = int(i / ((long long)N * C));
    const float v = __half2float(g[i]);
    g[i] = __float2half_rn(gamma[c] * (v * nx[(long long)b * C + c]) + beta[c] + v);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Input packing (backbones/dit.py:151-163): xin[Be*N, Kpad] fp16 = [ x | cond or 0 | text_emb | 0-pad ].
// Static part once per sample(); the x columns are rewritten after every evaluation by the update kernel.
// ---------------------------------------------------------------------------------------------------------

__global__ void pack_input_kernel(const PackParams p) {
  const int row = blockIdx.x;  // Be*N
  const int half = row / (p.B * p.N);
  const int r = row % (p.B * p.N);
  __half* o = p.xin + (long long)row * p.Kpad;
  for (int c = threadIdx.x; c < p.Kpad; c += blockDim.x) {
    float v = 0.f;
    if (c < p.mel) v = p.y[(long long)r * p.mel + c];
    else if (c < 2 * p.mel) v = half == 0 ? p.step_cond[(long long)r * p.mel + (c - p.mel)] : 0.f;
    else if (c < 2 * p.mel + p.Td) v = p.text[((long long)half * p.B * p.N + r) * p.Td + (c - 2 * p.mel)];
    o[c] = __float2half_rn(v);
  }
}

// ---------------------------------------------------------------------------------------------------------
// CFG + ODE update (cfm.py:190-191 + torchdiffeq fixed-grid Euler / midpoint, cfm.py:218), one launch per backbone
// evaluation e = *step_ptr with st = stages[e] (ew_params.h: OdeStage):
//   x = y + st.coef * (pred + (pred - null) * cfg);  xin[:, :mel] <- fp16(x) for both halves;
//   st.commit >= 0: y <- x, trajectory[st.commit] = x;
//   the last thread block to finish advances the device counter so one captured graph serves every evaluation.
// v: [Be*N, mel] fp32 (pred rows first, null rows second).
// ---------------------------------------------------------------------------------------------------------

__global__ void cfg_update_kernel(const UpdateParams p) {
  pdl_wait();
  pdl_launch_dependents();
  const int e = *p.step_ptr;
  const OdeStage st = p.stages[e];
  const SampleIo io = *p.io;
  const long long total = (long long)p.BN * p.mel;
  const long long null_off = (long long)p.B * p.seq_tok * p.mel;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / p.mel;
    const int c = int(i % p.mel);
    const long long b = r / p.N;
    const int n = int(r % p.N);
    const long long vi = ((b * p.seq_tok) + n + p.tok_off) * p.mel + c;
    const float pr = p.v[vi];
    float g = pr;
    if (p.packed) {
      const float nu = p.v[null_off + vi];
      g = pr + (pr - nu) * io.cfg;
    }
    const float x = io.y[i] + st.coef * g;
    if (st.commit >= 0) {
      io.y[i] = x;
      if (io.traj) io.traj[(long long)st.commit * total + i] = x;
    }
    const __half h = __float2half_rn(x);
    p.xin[r * p.Kpad + c] = h;
    if (p.packed) p.xin[(r + p.BN) * p.Kpad + c] = h;
  }
  // the last CTA to finish advances the device counter (every CTA has read entry e by then)
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    int* done = p.step_ptr + 1;
    if (atomicAdd(done, 1) == int(gridDim.x) - 1) {
      *done = 0;
      *p.step_ptr = e + 1;
    }
  }
}

__global__ void advance_step_kernel(int* step_ptr) {
  pdl_wait();
  pdl_launch_dependents();
  *step_ptr += 1;
}

// ---------------------------------------------------------------------------------------------------------
// Small fp32 linear for the per-sample() conditioning MLPs (modules.py:852-862): out[s, n] = act(in[s,:] . W[n,:] + b)
// W fp16 [Nout, K]; one warp per output column, S <= 64 rows.
// ---------------------------------------------------------------------------------------------------------
template <int ACT>  // 0 none, 1 silu
__global__ void small_linear_kernel(const float* in, const __half* W, const float* bias, float* out, int S, int K,
                                    int Nout) {
  const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (n >= Nout) return;
  const int lane = lane_id();
  const __half* wrow = W + (long long)n * K;
  if (K <= 1024 && (K & 31) == 0) {
    // the weight row is read ONCE into registers (lane l holds k = l, l + 32, ...) and reused for all S input rows —
    // the loop below keeps the accumulation order of the generic path (k ascending per lane, then the warp tree)
    float w[32];
    const int nk = K >> 5;
#pragma unroll
    for (int i = 0; i < 32; ++i) w[i] = i < nk ? __half2float(wrow[lane + 32 * i]) : 0.f;
    const float bv = bias ? bias[n] : 0.f;
    for (int s = 0; s < S; ++s) {
      const float* x = in + (long long)s * K + lane;
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (i < nk) acc += x[32 * i] * w[i];
      acc = warp_sum(acc);
      if (lane == 0) {
        acc += bv;
        out[(long long)s * Nout + n] = ACT == 1 ? silu(acc) : acc;
      }
    }
    return;
  }
  for (int s = 0; s < S; ++s) {
    float acc = 0.f;
    for (int k = lane; k < K; k += 32) acc += in[(long long)s * K + k] * __half2float(wrow[k]);
    acc = warp_sum(acc);
    if (lane == 0) {
      acc += bias ? bias[n] : 0.f;
      out[(long long)s * Nout + n] = ACT == 1 ? silu(acc) : acc;
    }
  }
}

// sinusoidal time features (modules.py:157-169): feat[s, :] = cat(sin, cos)(1000 * t[s] * exp(-ln(1e4)/(half-1) * i))
__global__ void time_features_kernel(const float* t, float* feat, int S, int dim) {
  const int s = blockIdx.x;
  const int half = dim / 2;
  const float k = logf(10000.0f) / float(half - 1);
  for (int i = threadIdx.x; i < half; i += blockDim.x) {
    const float arg = 1000.0f * t[s] * expf(-k * float(i));
    feat[(long long)s * dim + i] = sinf(arg);
    feat[(long long)s * dim + half + i] = cosf(arg);
  }
}

__global__ void silu_to_half_kernel(const float* in, __half* out, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = __float2half_rn(silu(in[i]));
}

__global__ void float_to_half_kernel(const float* in, __half* out, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = __float2half_rn(in[i]);
}

// rotary tables (x_transformers RotaryEmbedding, dit.py:207,352): cos/sin[pos, i] of pos * 10000^(-2i/dh)
__global__ void rope_table_kernel(float* cs, float* sn, int seq, int half) {
  const int pos = blockIdx.x;
  for (int i = threadIdx.x; i < half; i += blockDim.x) {
    const float inv = 1.0f / powf(10000.0f, float(2 * i) / float(2 * half));
    const float ang = float(pos) * inv;
    cs[pos * half + i] = cosf(ang);
    sn[pos * half + i] = sinf(ang);
  }
}

// UNetT (unett.py:271-273): h[b, 0, :] = t_emb[step], h[b, 1:, :] = src[b, :, :]   (fp32)
__global__ void prepend_time_token_kernel(float* dst, const float* src, const float* t_emb, const int* step_ptr,
                                          int N, int D, long long rows_out) {
  pdl_wait();
  pdl_launch_dependents();
  const long long row = blockIdx.x;
  if (row >= rows_out) return;
  const long long b = row / (N + 1);
  const int n = int(row % (N + 1));
  const float* s = (n == 0) ? t_emb + (long long)(*step_ptr) * D : src + (b * N + (n - 1)) * D;
  for (int c = threadIdx.x; c < D; c += blockDim.x) dst[row * D + c] = s[c];
}

// UNetT skip connection (unett.py:293-295): cat[m, :] = fp16([x[m, :], skip[m, :]])
__global__ void concat_half_kernel(const float* x, const float* skip, __half* out, long long rows, int D) {
  pdl_wait();
  pdl_launch_dependents();
  const long long total = rows * 2 * D;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long m = i / (2 * D);
    const int c = int(i % (2 * D));
    out[i] = __float2half_rn(c < D ? x[m * D + c] : skip[m * D + (c - D)]);
  }
}

// LayerNorm(affine) with fp32 output (Vocos: the normalised embedding IS the residual stream)
__global__ void ln_affine_f32_kernel(const float* x, float* out, int rows, int D, float eps, const float* w,
                                     const float* b) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = lane_id();
  float s = 0.f;
  for (int c = lane; c < D; c += 32) s += x[(long long)row * D + c];
  const float mean = warp_sum(s) / float(D);
  float q = 0.f;
  for (int c = lane; c < D; c += 32) {
    const float d = x[(long long)row * D + c] - mean;
    q += d * d;
  }
  const float rstd = rsqrtf(warp_sum(q) / float(D) + eps);
  for (int c = lane; c < D; c += 32) out[(long long)row * D + c] = (x[(long long)row * D + c] - mean) * rstd * w[c] + b[c];
}

}  // namespace f5

/*
 * f5tts_b200 — C ABI of the B200-native F5-TTS / E2-TTS ODE-sampling hot path.
 *
 * Plain C symbols, raw device pointers + explicit sizes, a CUDA stream, `int` return (0 = ok, < 0 = error;
 * f5_last_error() returns the message for the calling thread).  No ownership transfer: every buffer, including
 * the scratch workspace, belongs to the caller.  The only library-owned object is the opaque f5_engine, which
 * stores architecture constants and POINTERS to the caller's re-packed weights (see f5_weights).  Calls on
 * distinct (stream, workspace) pairs may run concurrently (the reference samples from a ThreadPoolExecutor,
 * infer/utils_infer.py:540-541).
 *
 * Each entry point names the reference interface it replaces (paths relative to /root/reference/src/f5_tts).
 * The reference has no native FFI on this path (it is pure PyTorch); the binding a maintainer adds is the ctypes
 * stub shown in INTEGRATION.md / f5_tts_b200/_lib.py.
 *
 * Requires an sm_100a device (tcgen05 / TMEM / TMA).  There is no CPU or non-Blackwell fallback.
 */
#ifndef F5TTS_B200_H
#define F5TTS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* f5_stream_t; /* cudaStream_t */

int f5_version(void);
const char* f5_last_error(void);
/* diagnostics only: per-CTA clock trace of the last GEMM when the process runs with F5_GEMM_TRACE=1 */
int f5_debug_gemm_trace(long long* host_out, int n_ctas);
int f5_debug_attn_trace(long long* host_out, int n_ctas); /* F5_ATTN_TRACE=1 */
/* number of kernels this library has launched in this process (bench.py reports it as gpu_launches) */
unsigned long long f5_launch_count(void);

/* ------------------------------------------------------------------------------------------------------------
 * Kernel-level entry points (used by the parity tests and by the Python operator mirrors)
 * ------------------------------------------------------------------------------------------------------------ */

enum { F5_ACT_NONE = 0, F5_ACT_GELU_TANH = 1, F5_ACT_GELU_ERF = 2, F5_ACT_MISH = 3 };
enum { F5_EPI_F16 = 0, F5_EPI_F32 = 1, F5_EPI_RESID = 2, F5_EPI_QKV_ROPE = 3 };

/* Fused linear: C = epilogue(A[M,K] . W[N,K]^T) — replaces nn.Linear (aten::addmm) call sites
 * model/modules.py:317,338,360-361,398-400 and, with conv != 0, the grouped Conv1d(k=taps, groups=D/64,
 * padding=taps/2) of ConvPositionEmbedding (model/modules.py:175-201).
 *   A fp16 [batches*rows, lda]; W fp16 [N, ldw] (conv: [taps][N][64]); fp32 accumulation. */
typedef struct {
  int rows;      /* valid rows per batch entry (plain GEMM: M, batches = 1) */
  int batches;
  int n_out;
  int k;         /* reduction length (plain) ; ignored for conv */
  int lda, ldw;  /* elements */
  int bn;        /* output tile width: 64 | 128 | 192 | 256 (0 = the planner picks width and cta_pair) */
  int epi, act;
  int conv_taps; /* 0 = plain GEMM */
  int cta_pair;  /* 1 = 2-CTA (cta_group::2) 256 x bn tiles; bn must be 128 or 256; plain GEMM, not EPI_F32 */
  const float* bias;
  void* out;               /* fp16 (F16 / QKV_ROPE, ldo % 8 == 0) or fp32 (F32, 16-byte aligned) [batches*rows, ldo] */
  void* out16b;            /* optional fp16 masked copy for F32 (rows past row_len are 0), same ldo: needs a 16-byte
                              aligned pointer and ldo % 8 == 0 */
  float* resid;            /* RESID: in/out fp32, ldo % 4 == 0 */
  int ldo;                 /* output row stride in elements (>= n_out); columns n_out .. ldo-1 are never written */
  const float* gate;       /* RESID: per-column gate (NULL = 1) */
  const int* step_ptr;     /* device step counter used to index gate (NULL = 0) */
  long long gate_step_stride;
  const int* row_len;      /* per-sample valid rows (NULL = all) */
  int seq;                 /* rows per sample */
  const float* rope_cos;   /* [seq, 32] */
  const float* rope_sin;
  int inner, pe_heads;
  int weights_static;      /* 1 = W was NOT written by the kernel preceding this call on the stream (model weights):
                              its first tiles are fetched ahead of the programmatic-dependent-launch wait */
  /* Packed / variable-length execution: 1 = output tiles whose rows all lie past row_len of their sample are skipped
   * entirely (not loaded, multiplied or stored: their output rows keep whatever the buffer held).  Needs row_len and
   * seq.  The reference's counterpart is its masked mode (flash_attn_varlen / attn_mask, modules.py:513-540). */
  int skip_padded_tiles;
} f5_gemm_args;
int f5_gemm(const void* A, const void* W, const f5_gemm_args* args, f5_stream_t stream);
/* Tile shape f5_gemm would run `args` with (after bn = 0 resolution): *bn tile width, *cta_pair 0/1. */
int f5_gemm_tile(const f5_gemm_args* args, int* bn, int* cta_pair);

/* Non-causal attention over the fused QKV buffer — replaces F.scaled_dot_product_attention at
 * model/modules.py:519 (attn_mask=None, or the key mask of modules.py:513-517 via kv_len).
 *   qkv fp16 [batches*seq, 3*heads*64]; out fp16 [batches*seq, heads*64]. dim_head must be 64.
 *   kv_len (device int32 [batches] or NULL = seq): sample b attends to its first kv_len[b] keys; 1 <= kv_len[b] is
 *   required.  With kv_len, the 256-row query blocks of sample b that start at or past kv_len[b] are not written (those
 *   rows of out keep what the buffer held; kv_len[b] = 0 leaves the whole sample unwritten). */
int f5_attention(const void* qkv, void* out, int batches, int seq, int heads, const int* kv_len, float scale,
                 f5_stream_t stream);

/* Row normalisation + modulation -> fp16 (model/modules.py:312-326,333-347,753; x_transformers RMSNorm unett.py:154)
 *   mode 0: LN(eps) * (1 + a[c]) + b[c]   mode 1: LN(eps) * a[c] + b[c]   mode 2: x/||x|| * sqrt(D) * a[c] */
int f5_row_norm(const float* x, void* out_f16, int rows, int D, int mode, float eps, const float* a, const float* b,
                f5_stream_t stream);

/* Vocos mel front-end — replaces MelSpec.forward / get_vocos_mel_spectrogram (model/modules.py:80-151).
 *   wav fp32 [B, nw]; fb fp32 [513, n_mels]; out fp32 [B, n_mels, T] (or [B, T, n_mels] if out_btc), T = 1 + nw/256 */
int f5_mel_spectrogram(const float* wav, int B, int nw, const float* fb, int n_mels, float* out, int out_btc,
                       f5_stream_t stream);

/* Vocos back-end — replaces vocos.Vocos.decode as used at infer/utils_infer.py:511 (VocosBackbone + ISTFTHead). */
typedef struct {
  const void* embed_w;   /* fp16 [512, 704]  im2col-packed Conv1d(100,512,7) weight, K padded 700 -> 704 */
  const float* embed_b;
  const float* norm_w; const float* norm_b;
  const float* dw_w[8]; const float* dw_b[8];        /* [512, 7], [512] */
  const float* ln_w[8]; const float* ln_b[8];
  const void* pw1_w[8]; const float* pw1_b[8];       /* fp16 [1536, 512] */
  const void* pw2_w[8]; const float* pw2_b[8];       /* fp16 [512, 1536] */
  const float* gamma[8];
  const float* final_w; const float* final_b;
  const void* head_w; const float* head_b;           /* fp16 [1026, 512] */
  int dim, inter, layers, n_mels;
} f5_vocos_weights;
size_t f5_vocos_workspace_bytes(int B, int T);
/* mel fp32 [B, 100, T] -> wav fp32 [B, 256*(T-1)] */
int f5_vocos_decode(const f5_vocos_weights* w, const float* mel, int B, int T, void* workspace, size_t ws_bytes,
                    float* wav, f5_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Engine: the whole CFM.sample NFE loop (model/cfm.py:160-223) for a DiT (backbones/dit.py:319-370) or UNetT
 * (backbones/unett.py:244-307) backbone.
 * ------------------------------------------------------------------------------------------------------------ */
typedef struct {
  int backbone;          /* 0 = DiT, 1 = UNetT */
  int dim, depth, heads, dim_head, ff_inner, mel_dim, text_dim, text_num_embeds, conv_layers;
  int text_mask_padding; /* yaml arch.text_mask_padding */
  int pe_attn_head;      /* -1 = all heads */
  int attn_mask_enabled;
} f5_arch;

typedef struct {
  const void* w_qkv; const float* b_qkv;   /* fp16 [3*inner, D] (to_q | to_k | to_v), fp32 [3*inner] */
  const void* w_out; const float* b_out;   /* fp16 [D, inner] */
  const void* w_ff1; const float* b_ff1;   /* fp16 [F, D] */
  const void* w_ff2; const float* b_ff2;   /* fp16 [D, F] */
  const void* w_skip;                      /* UNetT later half: fp16 [D, 2D], else NULL */
  const float* g_attn; const float* g_ff;  /* UNetT RMSNorm gains */
} f5_layer_weights;

typedef struct {
  const void* time_w0; const float* time_b0;  /* fp16 [D, 256] */
  const void* time_w1; const float* time_b1;  /* fp16 [D, D] */
  const float* text_table;                    /* fp32 [V+1, Td] */
  struct {
    const float* dw_w; const float* dw_b; const float* ln_w; const float* ln_b;
    const void* pw1_w; const float* pw1_b;    /* fp16 [2Td, Td] */
    const float* grn_gamma; const float* grn_beta;
    const void* pw2_w; const float* pw2_b;    /* fp16 [Td, 2Td] */
  } text_blocks[8];
  const void* proj_w; const float* proj_b;    /* fp16 [D, Kpad] input_embed.proj, K zero-padded to a multiple of 64 */
  int proj_kpad;
  const void* conv_w[2]; const float* conv_b[2]; /* fp16 [31][D][64] re-packed grouped conv, fp32 [D] */
  const void* mod_w; const float* mod_b;      /* DiT: fp16 [depth*6D + 2D, D] all AdaLN linears stacked; fp32 bias */
  const f5_layer_weights* layers;             /* [depth] */
  const float* g_out;                         /* UNetT norm_out.g */
  const void* out_w; const float* out_b;      /* fp16 [mel, D] proj_out */
} f5_weights;

typedef struct f5_engine f5_engine;
int f5_engine_create(const f5_arch* arch, const f5_weights* weights, f5_engine** out);
void f5_engine_destroy(f5_engine* e);

/* ODE solver of the NFE loop: torchdiffeq's fixed-grid methods on the caller's grid (odeint_kwargs, cfm.py:39-42,218).
 * Euler evaluates the backbone once per grid step, midpoint twice (at t_k and at t_k + dt/2). */
enum { F5_ODE_EULER = 0, F5_ODE_MIDPOINT = 1 };

typedef struct {
  int B, N, nt, steps;       /* steps: grid steps (t has steps+1 points) */
  const long long* text;     /* device int64 [B, nt], padded with -1 (model/utils.py:99-106) */
  const float* step_cond;    /* device fp32 [B, N, mel]  (cfm.py:151-153) */
  float* y;                  /* device fp32 [B, N, mel]  in: y0 (cfm.py:196-201), out: trajectory[-1] */
  const int* duration;       /* device int32 [B] per-sample lengths = `mask` of cfm.py:155-158, or NULL (B == 1) */
  const float* t;            /* HOST fp32 [steps+1] time grid after EPSS / sway (cfm.py:211-216) */
  float cfg_strength;        /* < 1e-5 -> single un-packed forward (cfm.py:166-177) */
  float* trajectory;         /* device fp32 [steps+1, B, N, mel] or NULL */
  int use_graph;             /* capture one NFE step into a CUDA graph and replay it */
  float* v_out;              /* optional device fp32 [Be, N, mel]: raw backbone output of the LAST evaluation (the value
                                transformer(x, cond, text, time, mask, cfg_infer=...) returns, dit.py:367-370); for
                                midpoint that is the evaluation at t[steps-1] + dt/2 */
  int exact_varlen;          /* with duration != NULL: 1 = every sample is computed exactly as if it were ALONE in the batch
                                with N = duration[b] — text blocks, conv position embedding and attention see nothing past
                                the sample's end, padded tiles are skipped.  This is what a loop of B = 1 sample() calls
                                computes (the reference's per-chunk loop, infer/utils_infer.py:540-541), in one batch.
                                0 = the reference's batched semantics (padded rows computed; attended unless
                                arch.attn_mask_enabled) */
  int ode_method;            /* F5_ODE_EULER or F5_ODE_MIDPOINT; any other value is rejected (since f5_version() 101) */
} f5_sample_args;
/* `evals` below is the number of backbone evaluations of the call: steps for Euler, 2 * steps for midpoint. */
size_t f5_sample_workspace_bytes(const f5_engine* e, int B, int N, int evals, float cfg_strength);
int f5_sample(f5_engine* e, const f5_sample_args* args, void* workspace, size_t ws_bytes, f5_stream_t stream);

/* algorithmic FLOPs of one f5_sample call (SURVEY.md §8d formula) — used by bench.py for the roofline */
double f5_sample_flops(const f5_engine* e, int B, int N, int evals, float cfg_strength);

#ifdef __cplusplus
}
#endif
#endif /* F5TTS_B200_H */

// Engine: the CFM.sample NFE loop (model/cfm.py:160-223) over a DiT (backbones/dit.py:319-370) or UNetT
// (backbones/unett.py:244-307) backbone, expressed as a fixed kernel schedule over a caller-owned workspace.
//
// Per sample() call (hoisted out of the NFE loop because it is step- or batch-invariant):
//   * text embeddings, cond + uncond variants (dit.py:284-314 caches them the same way)
//   * time embedding of every backbone evaluation and — DiT — the AdaLN modulation vectors of every (evaluation,
//     block) as one [evals, depth*6D + 2D] table: 22 weight-streaming GEMVs per evaluation become one GEMM per call
//     (evals = steps for Euler, 2 * steps for midpoint: every table is indexed by evaluation, not by grid step)
//   * rotary cos/sin table, static columns of the packed input projection operand
// Per backbone evaluation: input projection -> grouped conv position embedding x2 (tensor-core implicit GEMM) -> depth x
// {norm+modulate, fused QKV+RoPE GEMM, flash attention, out-proj (+gate, +mask, +residual), norm+modulate,
//  FF1+GELU, FF2 (+gate, +residual)} -> final norm -> proj_out -> fused CFG + ODE update (Euler step, midpoint half
// step or midpoint full step, read from the per-evaluation OdeStage table).
// Every kernel reads the evaluation index from a device counter, so one captured CUDA graph serves all evaluations.
#include <climits>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <vector>

#include "internal.h"

namespace f5 {

static inline size_t al256(size_t x) { return (x + 255) & ~size_t(255); }

struct Bump {
  uint8_t* base;
  size_t off = 0;
  explicit Bump(void* p) : base(reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(p) + 255) & ~uintptr_t(255))) {}
  template <typename T>
  T* take(size_t count) {
    T* r = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += al256(count * sizeof(T));
    return r;
  }
};

struct Layout {
  // sizes
  int B, Be, N, seq, evals, packed;  // evals: backbone evaluations of the call (ode_evals)
  long long M, M1;
  // common
  int* step_ptr;
  SampleIo* io;     // caller tensors + cfg scale of THIS call, read by the step kernels through the workspace
  OdeStage* stages;  // [evals]
  float* t_dev;      // [evals] time of every evaluation
  float *rope_cos, *rope_sin;
  int* row_len;     // [Be] or unused
  int* kv_len;      // [Be] or unused
  int* frame_len;   // [Be] valid mel frames per sample (row_len without the UNetT time token)
  int* valid_len;   // [B]
  float *tfeat, *th1, *temb;
  __half* temb_silu;
  float* mod;
  // text
  float* tx;
  uint8_t* filler;
  __half *ta, *tg;
  float *sumsq, *nx;
  // step buffers
  __half* xin;
  float* h0;
  __half *h0h, *c1;
  float* x;                  // UNetT residual [M1, D]; DiT: alias of h0
  std::vector<float*> skips;
  __half* cat;
  __half *a, *qkv, *ao, *g;
  float* v;
  size_t bytes;
};

}  // namespace f5

using namespace f5;

// One instantiated step graph.  The graph touches only the workspace: the caller's tensors (y, trajectory) and the CFG
// scale reach the kernels through the SampleIo block the prologue writes into the workspace, so the cache key is the
// workspace address plus the shape parameters the layout / kernel plans depend on — a fresh `y` or `trajectory`
// allocation per call no longer forces a re-capture.  Entries are reference-counted: a launch in flight on one thread
// keeps its graph alive while another thread evicts it.
struct GraphHolder {
  cudaGraphExec_t exec = nullptr;
  int nodes = 0;  // kernel/memcpy nodes per replay (for the launch counter)
  ~GraphHolder() {
    if (exec) cudaGraphExecDestroy(exec);
  }
};
struct GraphKey {
  const void* ws;
  // evals, not (steps, method): the layout and every kernel plan depend on the evaluation count only, and the solver's
  // rule lives in the OdeStage table the prologue uploads per call — so an Euler call with 2S steps and a midpoint call
  // with S steps share one graph.
  int B, N, evals, packed, masked;  // masked: 0 = no lengths, 1 = lengths (reference batched semantics), 2 = exact_varlen
  bool operator==(const GraphKey& o) const {
    return ws == o.ws && B == o.B && N == o.N && evals == o.evals && packed == o.packed && masked == o.masked;
  }
};
struct GraphEntry {
  GraphKey key;
  std::shared_ptr<GraphHolder> g;
};

struct f5_engine {
  f5_arch arch;
  f5_weights w;
  std::vector<f5_layer_weights> layers;
  int inner, modW, kin;
  std::mutex mu;
  std::vector<GraphEntry> graphs;
};

static int ode_evals(int steps, int ode_method) { return ode_method == F5_ODE_MIDPOINT ? 2 * steps : steps; }

static void plan_layout(const f5_engine* e, Layout& L, void* ws, int B, int N, int evals, float cfg) {
  const f5_arch& A = e->arch;
  Bump bp(ws);
  L.B = B;
  L.N = N;
  L.evals = evals;
  L.packed = cfg < 1e-5f ? 0 : 1;
  L.Be = L.packed ? 2 * B : B;
  L.seq = A.backbone == 1 ? N + 1 : N;
  L.M = (long long)L.Be * N;
  L.M1 = (long long)L.Be * L.seq;
  const int D = A.dim, Td = A.text_dim, F = A.ff_inner;
  L.step_ptr = bp.take<int>(64);
  L.io = bp.take<SampleIo>(1);
  L.stages = bp.take<OdeStage>(evals);
  L.t_dev = bp.take<float>(evals);
  L.rope_cos = bp.take<float>((size_t)L.seq * 32);
  L.rope_sin = bp.take<float>((size_t)L.seq * 32);
  L.row_len = bp.take<int>(L.Be);
  L.kv_len = bp.take<int>(L.Be);
  L.frame_len = bp.take<int>(L.Be);
  L.valid_len = bp.take<int>(B);
  L.tfeat = bp.take<float>((size_t)evals * 256);
  L.th1 = bp.take<float>((size_t)evals * D);
  L.temb = bp.take<float>((size_t)evals * D);
  L.temb_silu = bp.take<__half>((size_t)evals * D);
  L.mod = bp.take<float>((size_t)evals * (e->modW > 0 ? e->modW : 1));
  L.tx = bp.take<float>((size_t)2 * B * N * Td);
  L.filler = bp.take<uint8_t>((size_t)B * N);
  L.ta = bp.take<__half>((size_t)2 * B * N * Td);
  L.tg = bp.take<__half>((size_t)2 * B * N * 2 * Td);
  L.sumsq = bp.take<float>((size_t)2 * B * ((N + kGrnRows - 1) / kGrnRows) * 2 * Td);
  L.nx = bp.take<float>((size_t)2 * B * 2 * Td);
  L.xin = bp.take<__half>((size_t)L.M * e->kin);
  L.h0 = bp.take<float>((size_t)L.M * D);
  L.h0h = bp.take<__half>((size_t)L.M * D);
  L.c1 = bp.take<__half>((size_t)L.M * D);
  L.skips.clear();
  if (A.backbone == 1) {
    L.x = bp.take<float>((size_t)L.M1 * D);
    for (int i = 0; i < A.depth / 2; ++i) L.skips.push_back(bp.take<float>((size_t)L.M1 * D));
    L.cat = bp.take<__half>((size_t)L.M1 * 2 * D);
  } else {
    L.x = L.h0;
    L.cat = nullptr;
  }
  L.a = bp.take<__half>((size_t)L.M1 * D);
  L.qkv = bp.take<__half>((size_t)L.M1 * 3 * e->inner);
  L.ao = bp.take<__half>((size_t)L.M1 * e->inner);
  L.g = bp.take<__half>((size_t)L.M1 * F);
  L.v = bp.take<float>((size_t)L.M1 * A.mel_dim);
  L.bytes = bp.off + 512;
}

extern "C" {

int f5_engine_create(const f5_arch* arch, const f5_weights* weights, f5_engine** out) {
  if (!arch || !weights || !out) {
    set_error("engine_create: null argument");
    return -1;
  }
  if (arch->dim_head != 64) {
    set_error("engine_create: dim_head must be 64 (got %d)", arch->dim_head);
    return -1;
  }
  if (arch->dim % 128 || arch->dim > 1024 || (arch->ff_inner % 64)) {
    set_error("engine_create: dim must be a multiple of 128 and <= 1024, ff_inner a multiple of 64 (dim=%d ff=%d)",
              arch->dim, arch->ff_inner);
    return -1;
  }
  if (arch->dim / 16 != 64) {
    set_error("engine_create: ConvPositionEmbedding(groups=16) is built for 64 channels per group, i.e. dim == 1024");
    return -1;
  }
  if (arch->conv_layers > 8 || (arch->conv_layers > 0 && (arch->text_dim % 64 || arch->text_dim > 512))) {
    set_error("engine_create: text conv blocks need text_dim %% 64 == 0, <= 512, at most 8 layers");
    return -1;
  }
  if (int rc = configure_kernels()) return rc;
  f5_engine* e = new f5_engine();
  e->arch = *arch;
  e->w = *weights;
  e->layers.assign(weights->layers, weights->layers + arch->depth);
  e->w.layers = e->layers.data();
  e->inner = arch->heads * arch->dim_head;
  e->modW = arch->backbone == 0 ? arch->depth * 6 * arch->dim + 2 * arch->dim : 0;
  e->kin = weights->proj_kpad;
  if (e->kin % 64 || e->kin < 2 * arch->mel_dim + arch->text_dim) {
    set_error("engine_create: proj_kpad must be a multiple of 64 covering 2*mel + text_dim");
    delete e;
    return -1;
  }
  *out = e;
  return 0;
}

void f5_engine_destroy(f5_engine* e) {
  if (!e) return;
  delete e;  // graph holders destroy their executables
}

size_t f5_sample_workspace_bytes(const f5_engine* e, int B, int N, int evals, float cfg_strength) {
  Layout L;
  plan_layout(e, L, nullptr, B, N, evals, cfg_strength);
  return L.bytes;
}

double f5_sample_flops(const f5_engine* e, int B, int N, int evals, float cfg_strength) {
  const f5_arch& A = e->arch;
  const double D = A.dim, mel = A.mel_dim, Td = A.text_dim, F = A.ff_inner, Ld = A.depth;
  const double Be = cfg_strength < 1e-5f ? B : 2.0 * B;
  double per;  // one sample-forward
  if (A.backbone == 0) {
    const double n = N;
    per = Ld * (8.0 * n * D * D + 4.0 * n * D * F + 4.0 * n * n * D) + 2.0 * n * (2 * mel + Td) * D +
          2.0 * (2.0 * n * D * (D / 16.0) * 31.0) + 2.0 * n * D * mel;
  } else {
    const double n1 = N + 1.0, n = N;
    per = Ld * (8.0 * n1 * D * D + 4.0 * n1 * D * F + 4.0 * n1 * n1 * D) + (Ld / 2.0) * 4.0 * n1 * D * D +
          2.0 * n * (2 * mel + Td) * D + 2.0 * (2.0 * n * D * (D / 16.0) * 31.0) + 2.0 * n1 * D * mel;
  }
  double total = evals * Be * per;
  // text embedding, once per sample and CFG branch: conv_layers x (2 pointwise GEMMs)
  total += 2.0 * B * A.conv_layers * (2.0 * 2.0 * N * Td * 2.0 * Td);
  // conditioning: time MLP + AdaLN table, once per call
  total += evals * (2.0 * 256 * D + 2.0 * D * D + 2.0 * D * (double)e->modW);
  return total;
}

}  // extern "C"

// -------------------------------------------------------------------------------------------------------------
namespace {

struct StepPlans {
  GemmPlan proj, conv1, conv2, out_proj;
  std::vector<GemmPlan> qkv, oproj, ff1, ff2, skip;
  std::vector<AttnPlan> attn;  // identical per layer, kept once
};

#define RC(x)                \
  do {                       \
    int _rc = (x);           \
    if (_rc) return _rc;     \
  } while (0)

f5_gemm_args base_args(long long rows, int n_out, int k, int lda, int ldw, int bn, int epi, int act) {
  f5_gemm_args a{};
  a.weights_static = 1;  // every W the engine multiplies by is a packed model weight
  a.rows = (int)rows;
  a.batches = 1;
  a.n_out = n_out;
  a.k = k;
  a.lda = lda;
  a.ldw = ldw;
  a.bn = bn;
  a.epi = epi;
  a.act = act;
  return a;
}

constexpr int kAutoTile = 0;  // bn = 0: the GEMM planner picks the tile shape per problem (gemm.cu: pick_tile)

int build_step_plans(f5_engine* e, const Layout& L, const f5_sample_args* sa, StepPlans& P) {
  const f5_arch& A = e->arch;
  const f5_weights& W = e->w;
  const int D = A.dim, F = A.ff_inner, inner = e->inner;
  const bool dit = A.backbone == 0;
  const bool masked = sa->duration != nullptr;
  const bool strict = masked && sa->exact_varlen;  // every sample exactly as if alone in the batch (f5_sample_args)
  const bool mask_in = (dit && masked) || strict;  // input projection / conv position embedding see per-sample lengths
  const int pe_heads = A.pe_attn_head < 0 ? A.heads : A.pe_attn_head;
  const long long modS = e->modW;

  {  // input projection: h0 = xin . proj_w^T + b ; h0h = fp16(mask(h0))
    f5_gemm_args a = base_args(L.M, D, e->kin, e->kin, e->kin, 128, F5_EPI_F32, F5_ACT_NONE);
    a.bias = W.proj_b;
    a.out = L.h0;
    a.out16b = L.h0h;
    a.ldo = D;
    a.seq = L.N;
    a.row_len = mask_in ? L.frame_len : nullptr;
    a.skip_padded_tiles = (mask_in && (A.attn_mask_enabled || strict)) ? 1 : 0;
    RC(gemm_plan(&P.proj, L.xin, W.proj_w, &a));
  }
  for (int c = 0; c < 2; ++c) {  // grouped conv position embedding
    f5_gemm_args a{};
    a.weights_static = 1;
    a.rows = L.N;
    a.batches = L.Be;
    a.n_out = D;
    a.lda = D;
    a.conv_taps = 31;
    a.act = F5_ACT_MISH;
    a.bias = W.conv_b[c];
    a.ldo = D;
    a.seq = L.N;
    a.row_len = mask_in ? L.frame_len : nullptr;
    a.skip_padded_tiles = (mask_in && (A.attn_mask_enabled || strict)) ? 1 : 0;
    if (c == 0) {
      a.epi = F5_EPI_F16;
      a.out = L.c1;
      RC(gemm_plan(&P.conv1, L.h0h, W.conv_w[0], &a));
    } else {
      a.epi = F5_EPI_RESID;
      a.resid = L.h0;
      RC(gemm_plan(&P.conv2, L.c1, W.conv_w[1], &a));
    }
  }
  P.qkv.resize(A.depth);
  P.oproj.resize(A.depth);
  P.ff1.resize(A.depth);
  P.ff2.resize(A.depth);
  P.skip.resize(A.depth);
  const int* rl = masked ? L.row_len : nullptr;
  // Variable-length execution (SURVEY.md §8f-1): in the reference's key-masked mode (attn_mask_enabled, modules.py:
  // 513-518) padded rows influence nothing, so every GEMM / conv / attention tile that holds only padding is skipped.
  // In the default "faithful" mode padded keys ARE attended (SURVEY.md §0.5) and every row must be computed.
  const int skip = (masked && (A.attn_mask_enabled || strict)) ? 1 : 0;
  auto varlen = [&](f5_gemm_args& a) {
    if (!skip) return;
    a.row_len = L.row_len;
    a.seq = L.seq;
    a.skip_padded_tiles = 1;
  };
  for (int i = 0; i < A.depth; ++i) {
    const f5_layer_weights& lw = W.layers[i];
    if (!dit && lw.w_skip) {
      f5_gemm_args a = base_args(L.M1, D, 2 * D, 2 * D, 2 * D, 128, F5_EPI_F32, F5_ACT_NONE);
      a.out = L.x;
      a.ldo = D;
      RC(gemm_plan(&P.skip[i], L.cat, lw.w_skip, &a));  // (EPI_F32 direct-store path: not tile-skipped)
    }
    {
      f5_gemm_args a = base_args(L.M1, 3 * inner, D, D, D, kAutoTile, F5_EPI_QKV_ROPE, F5_ACT_NONE);
      a.bias = lw.b_qkv;
      a.out = L.qkv;
      a.ldo = 3 * inner;
      a.seq = L.seq;
      a.rope_cos = L.rope_cos;
      a.rope_sin = L.rope_sin;
      a.inner = inner;
      a.pe_heads = pe_heads;
      varlen(a);
      RC(gemm_plan(&P.qkv[i], L.a, lw.w_qkv, &a));
    }
    {
      f5_gemm_args a = base_args(L.M1, D, inner, inner, inner, kAutoTile, F5_EPI_RESID, F5_ACT_NONE);
      a.bias = lw.b_out;
      a.resid = L.x;
      a.ldo = D;
      a.seq = L.seq;
      a.row_len = rl;
      if (dit) {
        a.gate = L.mod + (size_t)i * 6 * D + 2 * D;
        a.step_ptr = L.step_ptr;
        a.gate_step_stride = modS;
      }
      varlen(a);
      RC(gemm_plan(&P.oproj[i], L.ao, lw.w_out, &a));
    }
    {
      f5_gemm_args a = base_args(L.M1, F, D, D, D, kAutoTile, F5_EPI_F16, F5_ACT_GELU_TANH);
      a.bias = lw.b_ff1;
      a.out = L.g;
      a.ldo = F;
      varlen(a);
      RC(gemm_plan(&P.ff1[i], L.a, lw.w_ff1, &a));
    }
    {
      f5_gemm_args a = base_args(L.M1, D, F, F, F, kAutoTile, F5_EPI_RESID, F5_ACT_NONE);
      a.bias = lw.b_ff2;
      a.resid = L.x;
      a.ldo = D;
      if (dit) {
        a.gate = L.mod + (size_t)i * 6 * D + 5 * D;
        a.step_ptr = L.step_ptr;
        a.gate_step_stride = modS;
      }
      varlen(a);
      RC(gemm_plan(&P.ff2[i], L.g, lw.w_ff2, &a));
    }
  }
  {
    f5_gemm_args a = base_args(L.M1, A.mel_dim, D, D, D, 128, F5_EPI_F32, F5_ACT_NONE);
    a.bias = W.out_b;
    a.out = L.v;
    a.ldo = A.mel_dim;
    RC(gemm_plan(&P.out_proj, L.a, W.out_w, &a));
  }
  P.attn.resize(1);
  RC(attn_plan(&P.attn[0], L.qkv, L.ao, L.Be, L.seq, A.heads, skip ? L.kv_len : nullptr,
               1.0f / sqrtf((float)A.dim_head)));
  return 0;
}

// Instrumented build (make TRACE=1) only: F5_DIAG_SKIP="norm,attn,qkv,out,ff1,ff2,conv" removes kernels from the step
// schedule (timing decomposition; results are wrong).  The production library has no such switch.
#ifdef F5_TRACE
static bool diag_skip(const char* what) {
  static const char* v = getenv("F5_DIAG_SKIP");
  return v != nullptr && strstr(v, what) != nullptr;
}
#else
static constexpr bool diag_skip(const char*) { return false; }
#endif

int norm_mod(const f5_engine* e, const Layout& L, const float* x, long long rows, int mode, const float* a,
             const float* b, bool step_indexed, cudaStream_t s) {
  NormParams p{};
  p.x = x;
  p.out = L.a;
  p.rows = (int)rows;
  p.D = e->arch.dim;
  p.eps = 1e-6f;
  p.a = a;
  p.b = b;
  p.step_ptr = step_indexed ? L.step_ptr : nullptr;
  p.step_stride = step_indexed ? e->modW : 0;
  p.params_static = 1;  // modulation table / gains: complete long before the GEMM that produces x
  if (diag_skip("norm")) return 0;
  return run_row_norm(mode, p, s);
}

int run_step(f5_engine* e, const Layout& L, const f5_sample_args* sa, const StepPlans& P, cudaStream_t s) {
  const f5_arch& A = e->arch;
  const int D = A.dim;
  const bool dit = A.backbone == 0;
  RC(gemm_run(P.proj, s));
  if (!diag_skip("conv")) {
    RC(gemm_run(P.conv1, s));
    RC(gemm_run(P.conv2, s));
  }
  if (!dit) RC(run_prepend_time_token(L.x, L.h0, L.temb, L.step_ptr, L.N, D, L.M1, s));
  const int half = A.depth / 2;
  for (int i = 0; i < A.depth; ++i) {
    const f5_layer_weights& lw = e->w.layers[i];
    if (dit) {
      const float* m = L.mod + (size_t)i * 6 * D;
      RC(norm_mod(e, L, L.x, L.M1, 0, m + D, m, true, s));  // scale_msa, shift_msa
    } else {
      if (i < half) {
        RC(check_cuda(cudaMemcpyAsync(L.skips[i], L.x, sizeof(float) * L.M1 * D, cudaMemcpyDeviceToDevice, s),
                      "skip copy"));
      } else {
        RC(run_concat_half(L.x, L.skips[A.depth - 1 - i], L.cat, L.M1, D, s));
        RC(gemm_run(P.skip[i], s));
      }
      RC(norm_mod(e, L, L.x, L.M1, 2, lw.g_attn, nullptr, false, s));
    }
    if (!diag_skip("qkv")) RC(gemm_run(P.qkv[i], s));
    if (!diag_skip("attn")) RC(attn_run(P.attn[0], s));
    if (!diag_skip("out")) RC(gemm_run(P.oproj[i], s));
    if (dit) {
      const float* m = L.mod + (size_t)i * 6 * D;
      RC(norm_mod(e, L, L.x, L.M1, 0, m + 4 * D, m + 3 * D, true, s));  // scale_mlp, shift_mlp
    } else {
      RC(norm_mod(e, L, L.x, L.M1, 2, lw.g_ff, nullptr, false, s));
    }
    if (!diag_skip("ff1")) RC(gemm_run(P.ff1[i], s));
    if (!diag_skip("ff2")) RC(gemm_run(P.ff2[i], s));
  }
  if (dit) {
    const float* m = L.mod + (size_t)A.depth * 6 * D;
    RC(norm_mod(e, L, L.x, L.M1, 0, m, m + D, true, s));  // AdaLayerNorm_Final: scale, shift (modules.py:342-347)
  } else {
    RC(norm_mod(e, L, L.x, L.M1, 2, e->w.g_out, nullptr, false, s));
  }
  RC(gemm_run(P.out_proj, s));
  UpdateParams ep{};
  ep.io = L.io;
  ep.v = L.v;
  ep.xin = L.xin;
  ep.stages = L.stages;
  ep.step_ptr = L.step_ptr;
  ep.BN = L.B * L.N;
  ep.mel = A.mel_dim;
  ep.Kpad = e->kin;
  ep.packed = L.packed;
  ep.N = L.N;
  ep.seq_tok = L.seq;
  ep.tok_off = dit ? 0 : 1;
  ep.B = L.B;
  return run_cfg_update(ep, s);
}

int run_prologue(f5_engine* e, const Layout& L, const f5_sample_args* sa, cudaStream_t s) {
  const f5_arch& A = e->arch;
  const f5_weights& W = e->w;
  const int D = A.dim, Td = A.text_dim, B = L.B, N = L.N, E = L.evals;
  const bool dit = A.backbone == 0;
  const bool masked = sa->duration != nullptr;
  const bool strict = masked && sa->exact_varlen;
  // per-evaluation update rule and time, in fp32 as torchdiffeq forms them on the grid's dtype:
  // Euler evaluates at t_k; midpoint at t_k and at t_k + dt/2 with dt = t_{k+1} - t_k
  std::vector<OdeStage> stage(E);
  std::vector<float> te(E);
  for (int k = 0; k < sa->steps; ++k) {
    const float dt = sa->t[k + 1] - sa->t[k];
    if (sa->ode_method == F5_ODE_MIDPOINT) {
      const float half = 0.5f * dt;
      stage[2 * k] = OdeStage{half, -1};
      stage[2 * k + 1] = OdeStage{dt, k + 1};
      te[2 * k] = sa->t[k];
      te[2 * k + 1] = sa->t[k] + half;
    } else {
      stage[k] = OdeStage{dt, k + 1};
      te[k] = sa->t[k];
    }
  }
  // small host -> device control data (pageable source: cudaMemcpyAsync stages it before returning)
  RC(check_cuda(cudaMemcpyAsync(L.stages, stage.data(), sizeof(OdeStage) * E, cudaMemcpyHostToDevice, s), "stages h2d"));
  RC(check_cuda(cudaMemcpyAsync(L.t_dev, te.data(), sizeof(float) * E, cudaMemcpyHostToDevice, s), "t h2d"));
  RC(check_cuda(cudaMemsetAsync(L.step_ptr, 0, sizeof(int) * 64, s), "step memset"));
  SampleIo io{sa->y, sa->trajectory, sa->cfg_strength};
  RC(check_cuda(cudaMemcpyAsync(L.io, &io, sizeof(io), cudaMemcpyHostToDevice, s), "io h2d"));
  if (masked) {
    // row_len[Be] = duration (+1 for the UNetT time token, unett.py:274-275); kv_len likewise
    std::vector<int> hd(B);
    RC(check_cuda(cudaMemcpyAsync(hd.data(), sa->duration, sizeof(int) * B, cudaMemcpyDeviceToHost, s), "dur d2h"));
    RC(check_cuda(cudaStreamSynchronize(s), "dur sync"));
    std::vector<int> rl(L.Be);
    for (int i = 0; i < L.Be; ++i) rl[i] = hd[i % B] + (dit ? 0 : 1);
    RC(check_cuda(cudaMemcpyAsync(L.row_len, rl.data(), sizeof(int) * L.Be, cudaMemcpyHostToDevice, s), "row_len"));
    RC(check_cuda(cudaMemcpyAsync(L.kv_len, rl.data(), sizeof(int) * L.Be, cudaMemcpyHostToDevice, s), "kv_len"));
    RC(check_cuda(cudaMemcpyAsync(L.valid_len, hd.data(), sizeof(int) * B, cudaMemcpyHostToDevice, s), "valid_len"));
    std::vector<int> fl(L.Be);
    for (int i = 0; i < L.Be; ++i) fl[i] = hd[i % B];
    RC(check_cuda(cudaMemcpyAsync(L.frame_len, fl.data(), sizeof(int) * L.Be, cudaMemcpyHostToDevice, s), "frame_len"));
    RC(check_cuda(cudaStreamSynchronize(s), "len sync"));
    if (A.attn_mask_enabled || sa->exact_varlen) {
      // tile skipping leaves padded rows of these buffers unwritten for the whole call: the conv inputs must read as
      // zero there (= the conv's padding), and q/k/v rows next to a sample's end are multiplied by P = 0 (must be finite)
      RC(check_cuda(cudaMemsetAsync(L.h0h, 0, sizeof(__half) * L.M * D, s), "h0h clear"));
      RC(check_cuda(cudaMemsetAsync(L.c1, 0, sizeof(__half) * L.M * D, s), "c1 clear"));
      RC(check_cuda(cudaMemsetAsync(L.qkv, 0, sizeof(__half) * L.M1 * 3 * e->inner, s), "qkv clear"));
    }
  }
  RC(run_rope_table(L.rope_cos, L.rope_sin, L.seq, 32, s));
  // time embedding for every backbone evaluation (modules.py:852-862)
  RC(run_time_features(L.t_dev, L.tfeat, E, 256, s));
  RC(run_small_linear(1, L.tfeat, reinterpret_cast<const __half*>(W.time_w0), W.time_b0, L.th1, E, 256, D, s));
  RC(run_small_linear(0, L.th1, reinterpret_cast<const __half*>(W.time_w1), W.time_b1, L.temb, E, D, D, s));
  if (dit) {
    RC(run_silu_to_half(L.temb, L.temb_silu, (long long)E * D, s));
    f5_gemm_args a = base_args(E, e->modW, D, D, D, 128, F5_EPI_F32, F5_ACT_NONE);
    a.bias = W.mod_b;
    a.out = L.mod;
    a.ldo = e->modW;
    GemmPlan pl;
    RC(gemm_plan(&pl, L.temb_silu, W.mod_w, &a));
    RC(gemm_run(pl, s));
  }
  // text embedding, both CFG variants (dit.py:86-139 / unett.py:55-84)
  TextGatherParams tp{};
  tp.ids = sa->text;
  tp.B = B;
  tp.nt = sa->nt;
  tp.N = N;
  tp.Td = Td;
  tp.valid_len = (dit && masked) ? L.valid_len : nullptr;
  tp.table = W.text_table;
  tp.num_embeds = A.text_num_embeds + 1;
  tp.add_pos = A.conv_layers > 0;
  tp.out = L.tx;
  tp.filler = L.filler;
  RC(run_text_gather(tp, s));
  const int R2 = 2 * B * N;
  for (int i = 0; i < A.conv_layers; ++i) {
    if (A.text_mask_padding) RC(run_mask_rows(L.tx, L.filler, B * N, R2, Td, s));
    DwConvLnParams dp{};
    dp.x = L.tx;
    dp.out = L.ta;
    dp.B = 2 * B;
    dp.N = N;
    dp.C = Td;
    dp.w = W.text_blocks[i].dw_w;
    dp.wb = W.text_blocks[i].dw_b;
    dp.ln_w = W.text_blocks[i].ln_w;
    dp.ln_b = W.text_blocks[i].ln_b;
    dp.eps = 1e-6f;
    RC(run_dwconv7_ln(dp, s));
    f5_gemm_args g1 = base_args(R2, 2 * Td, Td, Td, Td, 128, F5_EPI_F16, F5_ACT_GELU_ERF);
    g1.bias = W.text_blocks[i].pw1_b;
    g1.out = L.tg;
    g1.ldo = 2 * Td;
    RC(f5_gemm(L.ta, W.text_blocks[i].pw1_w, &g1, s));
    // exact_varlen: the sequence ends at the sample's own length — rows past it take no part in GRN's norm over the
    // sequence (modules.py:243) and are cleared again after the block (= the zero padding a B = 1 call would see)
    if (strict) RC(run_mask_rows_len_half(L.tg, L.valid_len, B, N, R2, 2 * Td, s));
    RC(run_grn(L.tg, L.sumsq, L.nx, W.text_blocks[i].grn_gamma, W.text_blocks[i].grn_beta, 2 * B, N, 2 * Td, s));
    f5_gemm_args g2 = base_args(R2, Td, 2 * Td, 2 * Td, 2 * Td, 64, F5_EPI_RESID, F5_ACT_NONE);
    g2.bias = W.text_blocks[i].pw2_b;
    g2.resid = L.tx;
    g2.ldo = Td;
    RC(f5_gemm(L.tg, W.text_blocks[i].pw2_w, &g2, s));
    if (strict) RC(run_mask_rows_len(L.tx, L.valid_len, B, N, R2, Td, s));
  }
  if (A.conv_layers > 0 && A.text_mask_padding) RC(run_mask_rows(L.tx, L.filler, B * N, R2, Td, s));
  PackParams pp{};
  pp.xin = L.xin;
  pp.B = B;
  pp.N = N;
  pp.mel = A.mel_dim;
  pp.Td = Td;
  pp.Kpad = e->kin;
  pp.packed = L.packed;
  pp.y = sa->y;
  pp.step_cond = sa->step_cond;
  pp.text = L.tx;
  RC(run_pack_input(pp, s));
  if (sa->trajectory)
    RC(check_cuda(cudaMemcpyAsync(sa->trajectory, sa->y, sizeof(float) * B * N * A.mel_dim, cudaMemcpyDeviceToDevice, s),
                  "trajectory[0]"));
  return 0;
}

int copy_v_out(const f5_engine* e, const Layout& L, const f5_sample_args* sa, cudaStream_t s) {
  if (!sa->v_out) return 0;
  const int mel = e->arch.mel_dim;
  const int off = e->arch.backbone == 0 ? 0 : 1;
  for (int b = 0; b < L.Be; ++b)
    RC(check_cuda(cudaMemcpyAsync(sa->v_out + (size_t)b * L.N * mel, L.v + ((size_t)b * L.seq + off) * mel,
                                  sizeof(float) * L.N * mel, cudaMemcpyDeviceToDevice, s),
                  "v_out copy"));
  return 0;
}

}  // namespace

extern "C" int f5_sample(f5_engine* e, const f5_sample_args* sa, void* workspace, size_t ws_bytes, f5_stream_t stream) {
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (!e || !sa || !workspace) {
    set_error("f5_sample: null argument");
    return -1;
  }
  if (sa->B <= 0 || sa->N <= 0 || sa->steps <= 0 || sa->nt <= 0) {
    set_error("f5_sample: empty problem (B=%d N=%d steps=%d nt=%d)", sa->B, sa->N, sa->steps, sa->nt);
    return -1;
  }
  if (sa->ode_method != F5_ODE_EULER && sa->ode_method != F5_ODE_MIDPOINT) {
    set_error("f5_sample: ode_method must be F5_ODE_EULER (0) or F5_ODE_MIDPOINT (1) (got %d)", sa->ode_method);
    return -1;
  }
  if (sa->ode_method == F5_ODE_MIDPOINT && sa->steps > INT_MAX / 2) {
    set_error("f5_sample: steps=%d: 2 * steps midpoint evaluations overflow int", sa->steps);
    return -1;
  }
  const int evals = ode_evals(sa->steps, sa->ode_method);
  Layout L;
  plan_layout(e, L, workspace, sa->B, sa->N, evals, sa->cfg_strength);
  if (ws_bytes < L.bytes) {
    set_error("f5_sample: workspace too small (%zu < %zu)", ws_bytes, L.bytes);
    return -1;
  }
  RC(run_prologue(e, L, sa, s));
  if (sa->use_graph) {
    const GraphKey key{workspace, sa->B, sa->N, evals, L.packed,
                       sa->duration == nullptr ? 0 : (sa->exact_varlen ? 2 : 1)};
    std::shared_ptr<GraphHolder> g;
    {
      std::lock_guard<std::mutex> lk(e->mu);
      for (auto& en : e->graphs)
        if (en.key == key) g = en.g;
    }
    if (!g) {
      // Capture outside the engine mutex (thread-local capture mode: concurrent sample() calls capture independently)
      // on a private stream — the caller's stream may be the legacy default stream, which cannot capture.
      StepPlans P;
      RC(build_step_plans(e, L, sa, P));
      cudaStream_t cs;
      RC(check_cuda(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking), "capture stream"));
      if (int brc = check_cuda(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal), "begin capture")) {
        cudaStreamDestroy(cs);
        return brc;
      }
      const unsigned long long before = f5_launch_count();
      const int rc = run_step(e, L, sa, P, cs);
      cudaGraph_t graph = nullptr;
      const cudaError_t ce = cudaStreamEndCapture(cs, &graph);
      cudaStreamDestroy(cs);
      count_launch(-(int)(f5_launch_count() - before));  // captured, not launched
      if (rc || ce != cudaSuccess) {
        if (graph) cudaGraphDestroy(graph);
        return rc ? rc : check_cuda(ce, "end capture");
      }
      g = std::make_shared<GraphHolder>();
      size_t nn = 0;
      cudaGraphGetNodes(graph, nullptr, &nn);
      g->nodes = (int)nn;
      const cudaError_t ie = cudaGraphInstantiate(&g->exec, graph, 0);
      cudaGraphDestroy(graph);
      if (ie != cudaSuccess) {
        g->exec = nullptr;
        return check_cuda(ie, "graph instantiate");
      }
      std::lock_guard<std::mutex> lk(e->mu);
      if (e->graphs.size() >= 16) e->graphs.erase(e->graphs.begin());  // holder is freed when its last user is done
      e->graphs.push_back(GraphEntry{key, g});
    }
    for (int k = 0; k < evals; ++k) RC(check_cuda(cudaGraphLaunch(g->exec, s), "graph launch"));
    count_launch(g->nodes * evals);
    return copy_v_out(e, L, sa, s);
  }
  StepPlans P;
  RC(build_step_plans(e, L, sa, P));
  for (int k = 0; k < evals; ++k) RC(run_step(e, L, sa, P, s));
  return copy_v_out(e, L, sa, s);
}

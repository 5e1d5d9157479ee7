// Launch wrappers + C entry points for the bandwidth-bound kernels, the mel front-end and the Vocos back-end.
#include "elementwise.cuh"
#include "fft.cuh"
#include "internal.h"

#include <cstdlib>
#include <map>
#include <memory>
#include <mutex>
#include <utility>
#include <vector>

namespace f5 {

// ---- per-device constant tables of the FFT kernels (twiddles, Hann window) and per-filterbank band indices ----------
namespace {
std::mutex g_fft_mu;
std::map<int, FftTables> g_fft_tables;                                  // device ordinal -> tables
std::map<std::pair<int, const void*>, std::pair<short*, short*>> g_bands;  // (device, fb pointer) -> (lo, hi) [n_mels]
}  // namespace

static int fft_tables(FftTables* out, cudaStream_t s) {
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lk(g_fft_mu);
  auto it = g_fft_tables.find(dev);
  if (it == g_fft_tables.end()) {
    float2* tw = nullptr;
    float* hann = nullptr;
    if (int rc = check_cuda(cudaMalloc(&tw, sizeof(float2) * kNfft / 2), "fft tables")) return rc;
    if (int rc = check_cuda(cudaMalloc(&hann, sizeof(float) * kNfft), "fft tables")) return rc;
    fft_tables_kernel<<<kNfft / 256, 256, 0, s>>>(tw, hann);  // same stream as the first user: ordered before it
    if (int rc = check_launch("fft_tables_kernel")) return rc;
    // later users may sit on other streams: the tables must be complete before this call returns
    if (int rc = check_cuda(cudaStreamSynchronize(s), "fft tables sync")) return rc;
    it = g_fft_tables.emplace(dev, FftTables{tw, hann}).first;
  }
  *out = it->second;
  return 0;
}

// First / last non-zero bin of every mel filter of the caller's dense [513, n_mels] filterbank (one D2H read per
// filterbank tensor; the Python side keeps one per device).
static int mel_bands(const float* fb, int n_mels, const short** lo, const short** hi, cudaStream_t s) {
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lk(g_fft_mu);
  const auto key = std::make_pair(dev, static_cast<const void*>(fb));
  auto it = g_bands.find(key);
  if (it == g_bands.end()) {
    std::vector<float> h((size_t)kBins * n_mels);
    if (int rc = check_cuda(cudaMemcpyAsync(h.data(), fb, sizeof(float) * h.size(), cudaMemcpyDeviceToHost, s), "fb d2h")) return rc;
    if (int rc = check_cuda(cudaStreamSynchronize(s), "fb sync")) return rc;
    std::vector<short> l(n_mels, 1), u(n_mels, 0);  // empty band: lo > hi
    for (int m = 0; m < n_mels; ++m) {
      int first = -1, last = -1;
      for (int f = 0; f < kBins; ++f)
        if (h[(size_t)f * n_mels + m] != 0.0f) {
          if (first < 0) first = f;
          last = f;
        }
      if (first >= 0) l[m] = (short)first, u[m] = (short)last;
    }
    short *dl = nullptr, *du = nullptr;
    if (int rc = check_cuda(cudaMalloc(&dl, sizeof(short) * n_mels), "band index")) return rc;
    if (int rc = check_cuda(cudaMalloc(&du, sizeof(short) * n_mels), "band index")) return rc;
    cudaMemcpyAsync(dl, l.data(), sizeof(short) * n_mels, cudaMemcpyHostToDevice, s);
    cudaMemcpyAsync(du, u.data(), sizeof(short) * n_mels, cudaMemcpyHostToDevice, s);
    if (int rc = check_cuda(cudaStreamSynchronize(s), "band index sync")) return rc;
    if (g_bands.size() >= 64) {  // filterbanks are per-process constants; a churning caller must not leak without bound
      for (auto& kv : g_bands) {
        cudaFree(kv.second.first);
        cudaFree(kv.second.second);
      }
      g_bands.clear();
    }
    it = g_bands.emplace(key, std::make_pair(dl, du)).first;
  }
  *lo = it->second.first;
  *hi = it->second.second;
  return 0;
}

static inline int grid_for(long long n, int block, int cap = 148 * 16) {
  long long g = (n + block - 1) / block;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

int run_row_norm(int mode, const NormParams& p, cudaStream_t s) {
  if (p.D % 128 || p.D > 1024) {
    set_error("row_norm: D must be a multiple of 128 and <= 1024 (got %d)", p.D);
    return -1;
  }
  // warps (= rows) per block: small blocks fit next to a still-running GEMM CTA (register file), so more of them are
  // resident with their modulation rows prefetched when the producer finishes
  // cfg2 on B200: 55.17 / 54.91 / 54.83 ms per utterance with 8 / 4 / 2 warps per block
  constexpr int wpb = 4;
  PdlLaunch L(dim3((p.rows + wpb - 1) / wpb), dim3(32 * wpb), 0, s);
  cudaError_t ce;
  if (mode == 0) ce = cudaLaunchKernelEx(&L.cfg, row_norm_kernel<0>, p);
  else if (mode == 1) ce = cudaLaunchKernelEx(&L.cfg, row_norm_kernel<1>, p);
  else if (mode == 2) ce = cudaLaunchKernelEx(&L.cfg, row_norm_kernel<2>, p);
  else {
    set_error("row_norm: bad mode %d", mode);
    return -1;
  }
  if (int rc = check_cuda(ce, "row_norm launch")) return rc;
  count_launch();
  return check_launch("row_norm_kernel");
}

int run_dwconv7_ln(const DwConvLnParams& p, cudaStream_t s) {
  if (p.C % 32 || p.C > 512) {
    set_error("dwconv7_ln: C must be a multiple of 32 and <= 512 (got %d)", p.C);
    return -1;
  }
  dwconv7_ln_kernel<<<(p.B * p.N + 7) / 8, 256, 0, s>>>(p);
  count_launch();
  return check_launch("dwconv7_ln_kernel");
}

int run_text_gather(const TextGatherParams& p, cudaStream_t s) {
  text_gather_kernel<<<2 * p.B * p.N, 128, 0, s>>>(p);
  count_launch();
  return check_launch("text_gather_kernel");
}

int run_mask_rows(float* x, const uint8_t* filler, int BN, int rows, int C, cudaStream_t s) {
  mask_rows_kernel<<<rows, 128, 0, s>>>(x, filler, BN, rows, C);
  count_launch();
  return check_launch("mask_rows_kernel");
}

int run_mask_rows_len(float* x, const int* valid_len, int B, int N, int rows, int C, cudaStream_t s) {
  mask_rows_len_kernel<float><<<rows, 128, 0, s>>>(x, valid_len, B, N, rows, C);
  count_launch();
  return check_launch("mask_rows_len_kernel<float>");
}
int run_mask_rows_len_half(__half* x, const int* valid_len, int B, int N, int rows, int C, cudaStream_t s) {
  mask_rows_len_kernel<__half><<<rows, 128, 0, s>>>(x, valid_len, B, N, rows, C);
  count_launch();
  return check_launch("mask_rows_len_kernel<half>");
}

int run_grn(__half* g, float* partial, float* nx, const float* gamma, const float* beta, int B, int N, int C,
            cudaStream_t s) {
  // `partial` must hold B * ceil(N / kGrnRows) * C floats
  const int nblk = (N + kGrnRows - 1) / kGrnRows;
  grn_sumsq_kernel<<<dim3((C + 255) / 256, nblk, B), 256, 0, s>>>(g, partial, N, C, kGrnRows);
  grn_finalize_kernel<<<B, 256, sizeof(float) * C, s>>>(partial, nblk, nx, C);
  const long long total = (long long)B * N * C;
  grn_apply_kernel<<<grid_for(total, 256), 256, 0, s>>>(g, nx, gamma, beta, N, C, total);
  count_launch(3);
  return check_launch("grn kernels");
}

int run_pack_input(const PackParams& p, cudaStream_t s) {
  const int Be = p.packed ? 2 * p.B : p.B;
  pack_input_kernel<<<Be * p.N, 128, 0, s>>>(p);
  count_launch();
  return check_launch("pack_input_kernel");
}

int run_cfg_update(const UpdateParams& p, cudaStream_t s) {
  const long long total = (long long)p.BN * p.mel;
  PdlLaunch L1(dim3(grid_for(total, 256, 148 * 4)), dim3(256), 0, s);
  if (int rc = check_cuda(cudaLaunchKernelEx(&L1.cfg, cfg_update_kernel, p), "cfg_update launch")) return rc;
  count_launch(1);
  return check_launch("cfg_update_kernel");
}

int run_small_linear(int act, const float* in, const __half* W, const float* bias, float* out, int S, int K, int Nout,
                     cudaStream_t s) {
  dim3 grid((Nout + 7) / 8);
  if (act == 1) small_linear_kernel<1><<<grid, 256, 0, s>>>(in, W, bias, out, S, K, Nout);
  else small_linear_kernel<0><<<grid, 256, 0, s>>>(in, W, bias, out, S, K, Nout);
  count_launch();
  return check_launch("small_linear_kernel");
}

int run_time_features(const float* t, float* feat, int S, int dim, cudaStream_t s) {
  time_features_kernel<<<S, 128, 0, s>>>(t, feat, S, dim);
  count_launch();
  return check_launch("time_features_kernel");
}

int run_silu_to_half(const float* in, __half* out, long long n, cudaStream_t s) {
  silu_to_half_kernel<<<grid_for(n, 256), 256, 0, s>>>(in, out, n);
  count_launch();
  return check_launch("silu_to_half_kernel");
}

int run_rope_table(float* cs, float* sn, int seq, int half, cudaStream_t s) {
  rope_table_kernel<<<seq, 32, 0, s>>>(cs, sn, seq, half);
  count_launch();
  return check_launch("rope_table_kernel");
}

int run_prepend_time_token(float* dst, const float* src, const float* t_emb, const int* step_ptr, int N, int D,
                           long long rows_out, cudaStream_t s) {
  PdlLaunch L(dim3((unsigned)rows_out), dim3(256), 0, s);
  if (int rc = check_cuda(cudaLaunchKernelEx(&L.cfg, prepend_time_token_kernel, dst, src, t_emb, step_ptr, N, D, rows_out),
                          "prepend_time_token launch"))
    return rc;
  count_launch();
  return check_launch("prepend_time_token_kernel");
}

int run_concat_half(const float* x, const float* skip, __half* out, long long rows, int D, cudaStream_t s) {
  PdlLaunch L(dim3(grid_for(rows * 2 * D, 256)), dim3(256), 0, s);
  if (int rc = check_cuda(cudaLaunchKernelEx(&L.cfg, concat_half_kernel, x, skip, out, rows, D), "concat_half launch")) return rc;
  count_launch();
  return check_launch("concat_half_kernel");
}

}  // namespace f5

using namespace f5;

extern "C" {

int f5_row_norm(const float* x, void* out_f16, int rows, int D, int mode, float eps, const float* a, const float* b,
                f5_stream_t stream) {
  NormParams p{};
  p.x = x;
  p.out = reinterpret_cast<__half*>(out_f16);
  p.rows = rows;
  p.D = D;
  p.eps = eps;
  p.a = a;
  p.b = b;
  return run_row_norm(mode, p, reinterpret_cast<cudaStream_t>(stream));
}

int f5_mel_spectrogram(const float* wav, int B, int nw, const float* fb, int n_mels, float* out, int out_btc,
                       f5_stream_t stream) {
  if (B <= 0 || nw <= kNfft / 2) {
    set_error("mel_spectrogram: need B > 0 and nw > %d (reflect padding), got B=%d nw=%d", kNfft / 2, B, nw);
    return -1;
  }
  const int T = 1 + nw / kHop;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  FftTables tab;
  if (int rc = fft_tables(&tab, s)) return rc;
  const short *lo = nullptr, *hi = nullptr;
  if (int rc = mel_bands(fb, n_mels, &lo, &hi, s)) return rc;
  mel_stft_kernel<<<dim3(T, B), 256, 0, s>>>(wav, nw, T, fb, n_mels, lo, hi, tab, out, out_btc);
  count_launch();
  return check_launch("mel_stft_kernel");
}

static inline size_t al256(size_t x) { return (x + 255) & ~size_t(255); }

size_t f5_vocos_workspace_bytes(int B, int T) {
  const size_t R = (size_t)B * T;
  size_t n = 0;
  n += al256(R * 704 * 2);   // im2col
  n += al256(R * 512 * 4);   // x residual fp32
  n += al256(R * 512 * 4);   // embed out fp32 (pre-norm)
  n += al256(R * 512 * 2);   // a fp16
  n += al256(R * 1536 * 2);  // g fp16
  n += al256(R * 1026 * 4);  // head fp32
  n += al256(R * 1024 * 4);  // frames
  return n + 1024;
}

}  // extern "C"

namespace {

// All kernels of one decode, enqueued on `s` (graph capture or direct).
int vocos_enqueue(const f5_vocos_weights* w, const float* mel, int B, int T, void* workspace, float* wav, FftTables tab,
                  cudaStream_t s) {
  f5_stream_t stream = reinterpret_cast<f5_stream_t>(s);
  const int R = B * T;
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  auto take = [&](size_t bytes) {
    uint8_t* p = base;
    base += al256(bytes);
    return p;
  };
  __half* A0 = reinterpret_cast<__half*>(take((size_t)R * 704 * 2));
  float* x = reinterpret_cast<float*>(take((size_t)R * 512 * 4));
  float* e = reinterpret_cast<float*>(take((size_t)R * 512 * 4));
  __half* a = reinterpret_cast<__half*>(take((size_t)R * 512 * 2));
  __half* g = reinterpret_cast<__half*>(take((size_t)R * 1536 * 2));
  float* head = reinterpret_cast<float*>(take((size_t)R * 1026 * 4));
  float* frames = reinterpret_cast<float*>(take((size_t)R * 1024 * 4));

  int rc;
  vocos_im2col_kernel<<<R, 256, 0, s>>>(mel, B, 100, T, A0, 704);
  count_launch();
  f5_gemm_args ga{};
  ga.weights_static = 1;
  ga.rows = R; ga.batches = 1; ga.n_out = 512; ga.k = 704; ga.lda = 704; ga.ldw = 704; ga.bn = 64;
  ga.epi = F5_EPI_F32; ga.act = F5_ACT_NONE; ga.bias = w->embed_b; ga.out = e; ga.ldo = 512;
  if ((rc = f5_gemm(A0, w->embed_w, &ga, stream))) return rc;
  // x = LayerNorm(embed(mel)) is the residual stream (fp32)
  ln_affine_f32_kernel<<<(R + 7) / 8, 256, 0, s>>>(e, x, R, 512, 1e-6f, w->norm_w, w->norm_b);
  count_launch();
  if ((rc = check_launch("ln_affine_f32_kernel"))) return rc;
  for (int i = 0; i < w->layers; ++i) {
    DwConvLnParams dp{};
    dp.x = x; dp.out = a; dp.B = B; dp.N = T; dp.C = 512; dp.w = w->dw_w[i]; dp.wb = w->dw_b[i];
    dp.ln_w = w->ln_w[i]; dp.ln_b = w->ln_b[i]; dp.eps = 1e-6f;
    if ((rc = run_dwconv7_ln(dp, s))) return rc;
    f5_gemm_args g1{};
    g1.weights_static = 1;
    g1.rows = R; g1.batches = 1; g1.n_out = 1536; g1.k = 512; g1.lda = 512; g1.ldw = 512; g1.bn = 128;
    g1.epi = F5_EPI_F16; g1.act = F5_ACT_GELU_ERF; g1.bias = w->pw1_b[i]; g1.out = g; g1.ldo = 1536;
    if ((rc = f5_gemm(a, w->pw1_w[i], &g1, stream))) return rc;
    f5_gemm_args g2{};
    g2.weights_static = 1;
    g2.rows = R; g2.batches = 1; g2.n_out = 512; g2.k = 1536; g2.lda = 1536; g2.ldw = 1536; g2.bn = 64;
    g2.epi = F5_EPI_RESID; g2.act = F5_ACT_NONE; g2.bias = w->pw2_b[i]; g2.resid = x; g2.ldo = 512;
    g2.gate = w->gamma[i];
    if ((rc = f5_gemm(g, w->pw2_w[i], &g2, stream))) return rc;
  }
  {
    NormParams np{};
    np.x = x; np.out = a; np.rows = R; np.D = 512; np.eps = 1e-6f; np.a = w->final_w; np.b = w->final_b;
    if ((rc = run_row_norm(1, np, s))) return rc;
  }
  f5_gemm_args gh{};
  gh.weights_static = 1;
  gh.rows = R; gh.batches = 1; gh.n_out = 1026; gh.k = 512; gh.lda = 512; gh.ldw = 512; gh.bn = 128;
  gh.epi = F5_EPI_F32; gh.act = F5_ACT_NONE; gh.bias = w->head_b; gh.out = head; gh.ldo = 1026;
  if ((rc = f5_gemm(a, w->head_w, &gh, stream))) return rc;
  istft_frames_kernel<<<R, 256, 0, s>>>(head, 1026, frames, tab);
  const long long total = (long long)B * kHop * (T - 1);
  istft_ola_kernel<<<grid_for(total, 256), 256, 0, s>>>(frames, T, wav, B, tab);
  count_launch(2);
  return check_launch("vocos istft kernels");
}

// One captured decode per (weights, workspace, B, T).  Only two kernels touch caller tensors — the im2col reads `mel`, the
// overlap-add writes `wav` — and their node parameters are patched before every launch, so fresh input / output
// allocations do not invalidate the graph.
struct VocosGraph {
  const void* w0;
  const void* ws;
  int B, T;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  cudaGraphNode_t n_in = nullptr, n_out = nullptr;
  int nodes = 0;
  ~VocosGraph() {
    if (exec) cudaGraphExecDestroy(exec);
    if (graph) cudaGraphDestroy(graph);
  }
};
std::mutex g_vocos_mu;
std::vector<std::shared_ptr<VocosGraph>> g_vocos_graphs;

}  // namespace

extern "C" {

int f5_vocos_decode(const f5_vocos_weights* w, const float* mel, int B, int T, void* workspace, size_t ws_bytes,
                    float* wav, f5_stream_t stream) {
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (w->dim != 512 || w->inter != 1536 || w->n_mels != 100 || w->layers > 8) {
    set_error("vocos_decode: only the charactr/vocos-mel-24khz shape (512/1536, 100 mels, <= 8 layers) is built");
    return -1;
  }
  if (B <= 0 || T < 2) {
    set_error("vocos_decode: need B > 0 and at least 2 frames");
    return -1;
  }
  if (ws_bytes < f5_vocos_workspace_bytes(B, T)) {
    set_error("vocos_decode: workspace too small");
    return -1;
  }
  int rc;
  if ((rc = configure_kernels())) return rc;
  FftTables tab;
  if ((rc = fft_tables(&tab, s))) return rc;
  std::shared_ptr<VocosGraph> g;
  {
    std::lock_guard<std::mutex> lk(g_vocos_mu);
    for (auto& e : g_vocos_graphs)
      if (e->w0 == w->embed_w && e->ws == workspace && e->B == B && e->T == T) g = e;
  }
  if (!g) {
    cudaStream_t cs;
    if ((rc = check_cuda(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking), "capture stream"))) return rc;
    if ((rc = check_cuda(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal), "begin capture"))) {
      cudaStreamDestroy(cs);
      return rc;
    }
    const unsigned long long before = f5_launch_count();
    rc = vocos_enqueue(w, mel, B, T, workspace, wav, tab, cs);
    g = std::make_shared<VocosGraph>();
    const cudaError_t ce = cudaStreamEndCapture(cs, &g->graph);
    cudaStreamDestroy(cs);
    g->nodes = (int)(f5_launch_count() - before);
    count_launch(-g->nodes);  // captured, not launched
    if (rc) return rc;
    if ((rc = check_cuda(ce, "end capture"))) return rc;
    size_t nn = 0;
    cudaGraphGetNodes(g->graph, nullptr, &nn);
    std::vector<cudaGraphNode_t> nodes(nn);
    cudaGraphGetNodes(g->graph, nodes.data(), &nn);
    for (auto nd : nodes) {
      cudaGraphNodeType ty;
      if (cudaGraphNodeGetType(nd, &ty) != cudaSuccess || ty != cudaGraphNodeTypeKernel) continue;
      cudaKernelNodeParams kp{};
      if (cudaGraphKernelNodeGetParams(nd, &kp) != cudaSuccess) continue;
      if (kp.func == reinterpret_cast<void*>(vocos_im2col_kernel)) g->n_in = nd;
      if (kp.func == reinterpret_cast<void*>(istft_ola_kernel)) g->n_out = nd;
    }
    if (!g->n_in || !g->n_out) {
      set_error("vocos_decode: could not locate the I/O kernel nodes of the captured graph");
      return -7;
    }
    if ((rc = check_cuda(cudaGraphInstantiate(&g->exec, g->graph, 0), "graph instantiate"))) return rc;
    g->w0 = w->embed_w;
    g->ws = workspace;
    g->B = B;
    g->T = T;
    std::lock_guard<std::mutex> lk(g_vocos_mu);
    if (g_vocos_graphs.size() >= 32) g_vocos_graphs.erase(g_vocos_graphs.begin());
    g_vocos_graphs.push_back(g);
  }
  // patch the two nodes that see caller tensors (same grid / block / other arguments as captured)
  {
    cudaKernelNodeParams kp{};
    if ((rc = check_cuda(cudaGraphKernelNodeGetParams(g->n_in, &kp), "node params"))) return rc;
    const float* mel_arg = mel;
    void** args = kp.kernelParams;
    void* patched[6] = {(void*)&mel_arg, args[1], args[2], args[3], args[4], args[5]};
    kp.kernelParams = patched;
    if ((rc = check_cuda(cudaGraphExecKernelNodeSetParams(g->exec, g->n_in, &kp), "patch im2col node"))) return rc;
  }
  {
    cudaKernelNodeParams kp{};
    if ((rc = check_cuda(cudaGraphKernelNodeGetParams(g->n_out, &kp), "node params"))) return rc;
    float* wav_arg = wav;
    void** args = kp.kernelParams;
    void* patched[5] = {args[0], args[1], (void*)&wav_arg, args[3], args[4]};
    kp.kernelParams = patched;
    if ((rc = check_cuda(cudaGraphExecKernelNodeSetParams(g->exec, g->n_out, &kp), "patch overlap-add node"))) return rc;
  }
  if ((rc = check_cuda(cudaGraphLaunch(g->exec, s), "vocos graph launch"))) return rc;
  count_launch(g->nodes);
  return 0;
}

}  // extern "C"

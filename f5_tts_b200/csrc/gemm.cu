// Host side of the tcgen05 GEMM: tensor-map encoding, instantiation table, launch, C entry point f5_gemm.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <atomic>
#include <mutex>

#include "gemm.cuh"
#include "internal.h"

namespace f5 {

static thread_local char g_err[512] = "";
static long long* g_trace = nullptr;
static std::atomic<unsigned long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add((unsigned long long)(long long)n, std::memory_order_relaxed); }
int check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return 0;
  set_error("%s: %s", what, cudaGetErrorString(e));
  return -2;
}
int check_launch(const char* what) { return check_cuda(cudaGetLastError(), what); }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

int encode_tmap_f16(CUtensorMap* m, const void* ptr, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1,
                    uint64_t stride2, uint32_t b0, uint32_t b1, int rank) {
  return encode_tmap(m, 0, ptr, d0, d1, d2, stride1, stride2, b0, b1, rank);
}

int encode_tmap(CUtensorMap* m, int is_f32, const void* ptr, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1,
                uint64_t stride2, uint32_t b0, uint32_t b1, int rank) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled unavailable (no CUDA driver / not a TMA-capable device)");
    return -3;
  }
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || (stride1 & 15) || (rank == 3 && (stride2 & 15))) {
    set_error("tensor map: pointer/strides must be 16-byte aligned (ptr=%p s1=%llu s2=%llu)", ptr,
              (unsigned long long)stride1, (unsigned long long)stride2);
    return -4;
  }
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {stride1, stride2};
  cuuint32_t box[3] = {b0, b1, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(m, is_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, (cuuint32_t)rank, const_cast<void*>(ptr), dims, strides, box,
                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed: %d (dims %llu,%llu,%llu box %u,%u)", (int)r, (unsigned long long)d0,
              (unsigned long long)d1, (unsigned long long)d2, b0, b1);
    return -5;
  }
  return 0;
}

int configure_kernels();
int num_sms();

template <int BN, int STAGES, int EPI, int ACT, bool CONV, bool PAIR = false>
static int launch_inst(const GemmPlan& pl, cudaStream_t s) {
  auto kern = gemm_tcgen05_kernel<BN, STAGES, EPI, ACT, CONV, PAIR>;
  constexpr size_t smem = gemm_smem_bytes<BN, STAGES, PAIR>();
  if (int rc = configure_kernels()) return rc;
  PdlLaunch L(pl.grid, dim3(gemm_threads(EPI, ACT)), smem, s, PAIR ? 2 : 1);
  if (int rc = check_cuda(cudaLaunchKernelEx(&L.cfg, kern, pl.tmA, pl.tmB, pl.tmC, pl.p), "gemm launch")) return rc;
  count_launch();
  return check_launch("gemm_tcgen05_kernel launch");
}

template <int BN, int STAGES, int EPI, int ACT, bool CONV, bool PAIR = false>
static int configure_inst() {
  auto kern = gemm_tcgen05_kernel<BN, STAGES, EPI, ACT, CONV, PAIR>;
  constexpr size_t smem = gemm_smem_bytes<BN, STAGES, PAIR>();
  if (int rc = check_cuda(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                          "cudaFuncSetAttribute(gemm smem)"))
    return rc;
  cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
  return 0;
}

#define F5_GEMM_CASE(BN_, ST_, EPI_, ACT_, CONV_)                                                                   \
  if (!pl.pair && pl.bn == BN_ && pl.epi == EPI_ && pl.act == ACT_ && (pl.conv != 0) == CONV_)        \
    return launch_inst<BN_, ST_, EPI_, ACT_, CONV_>(pl, s);
#define F5_GEMM_PAIR_CASE(BN_, ST_, EPI_, ACT_)                                                  \
  if (pl.pair && pl.bn == BN_ && pl.epi == EPI_ && pl.act == ACT_ && !pl.conv)     \
    return launch_inst<BN_, ST_, EPI_, ACT_, false, true>(pl, s);
// cudaFuncSetAttribute is per device: the configured flag and the SM count are tracked per device ordinal, so one
// process may drive engines on several GPUs (ADVICE r1).
namespace {
constexpr int kMaxDevices = 64;
struct DeviceState {
  bool configured = false;
  int sms = 0;
};
DeviceState g_dev[kMaxDevices];
std::mutex g_dev_mu;
int current_device() {
  int d = 0;
  cudaGetDevice(&d);
  return (d >= 0 && d < kMaxDevices) ? d : 0;
}
}  // namespace

int configure_kernels() {
  const int dev = current_device();
  std::lock_guard<std::mutex> lk(g_dev_mu);
  if (g_dev[dev].configured) return 0;
  if (int rc = configure_inst<64, 7, EPI_F16, ACT_NONE, false>()) return rc;
  if (int rc = configure_inst<64, 7, EPI_F16, ACT_GELU_TANH, false>()) return rc;
  if (int rc = configure_inst<64, 7, EPI_F16, ACT_GELU_ERF, false>()) return rc;
  if (int rc = configure_inst<64, 7, EPI_F32, ACT_NONE, false>()) return rc;
  if (int rc = configure_inst<64, 7, EPI_RESID, ACT_NONE, false>()) return rc;
  if (int rc = configure_inst<128, 5, EPI_F16, ACT_NONE, false>()) return rc;
  if (int rc = configure_inst<128, 5, EPI_F16, ACT_GELU_TANH, false>()) return rc;
  if (int rc = configure_inst<128, 5, EPI_F16, ACT_GELU_ERF, false>()) return rc;
  if (int rc = configure_inst<128, 5, EPI_F32, ACT_NONE, false>()) return rc;
  if (int rc = configure_inst<128, 5, EPI_RESID, ACT_NONE, false>()) return rc;
  if (int rc = configure_inst<256, 3, EPI_F16, ACT_NONE, false>()) return rc;
  if (int rc = configure_inst<256, 3, EPI_F16, ACT_GELU_TANH, false>()) return rc;
  if (int rc = configure_inst<256, 3, EPI_F16, ACT_GELU_ERF, false>()) return rc;
  if (int rc = configure_inst<256, 3, EPI_F32, ACT_NONE, false>()) return rc;
  if (int rc = configure_inst<256, 3, EPI_RESID, ACT_NONE, false>()) return rc;
  if (int rc = configure_inst<128, 5, EPI_QKV_ROPE, ACT_NONE, false>()) return rc;
  if (int rc = configure_inst<192, 4, EPI_QKV_ROPE, ACT_NONE, false>()) return rc;
  if (int rc = configure_inst<192, 4, EPI_F16, ACT_NONE, false>()) return rc;
  if (int rc = configure_inst<192, 4, EPI_F16, ACT_GELU_TANH, false>()) return rc;
  if (int rc = configure_inst<192, 4, EPI_RESID, ACT_NONE, false>()) return rc;
  if (int rc = configure_inst<256, 3, EPI_QKV_ROPE, ACT_NONE, false>()) return rc;
  if (int rc = configure_inst<64, 7, EPI_F16, ACT_MISH, true>()) return rc;
  if (int rc = configure_inst<64, 7, EPI_RESID, ACT_MISH, true>()) return rc;
  if (int rc = configure_inst<256, 5, EPI_F16, ACT_NONE, false, true>()) return rc;
  if (int rc = configure_inst<256, 5, EPI_F16, ACT_GELU_TANH, false, true>()) return rc;
  if (int rc = configure_inst<256, 5, EPI_RESID, ACT_NONE, false, true>()) return rc;
  if (int rc = configure_inst<256, 5, EPI_QKV_ROPE, ACT_NONE, false, true>()) return rc;
  if (int rc = configure_inst<192, 6, EPI_F16, ACT_NONE, false, true>()) return rc;
  if (int rc = configure_inst<192, 6, EPI_F16, ACT_GELU_TANH, false, true>()) return rc;
  if (int rc = configure_inst<192, 6, EPI_RESID, ACT_NONE, false, true>()) return rc;
  if (int rc = configure_inst<192, 6, EPI_QKV_ROPE, ACT_NONE, false, true>()) return rc;
  if (int rc = configure_inst<128, 6, EPI_F16, ACT_NONE, false, true>()) return rc;
  if (int rc = configure_inst<128, 6, EPI_F16, ACT_GELU_TANH, false, true>()) return rc;
  if (int rc = configure_inst<128, 6, EPI_RESID, ACT_NONE, false, true>()) return rc;
  if (int rc = configure_inst<128, 6, EPI_QKV_ROPE, ACT_NONE, false, true>()) return rc;
  if (int rc = attn_configure()) return rc;
  g_dev[dev].configured = true;
  return 0;
}

bool pdl_enabled() {
#ifdef F5_TRACE  // diagnostic build only: F5_PDL=0 launches without programmatic dependent launch
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("F5_PDL");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v != 0;
#else
  return true;
#endif
}

int num_sms() {
  const int dev = current_device();
  int n = g_dev[dev].sms;  // written once per device; a racing first call computes the same value
  if (n == 0) {
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    g_dev[dev].sms = n;
  }
  return n;
}

int gemm_run(const GemmPlan& pl, cudaStream_t s) {
  F5_GEMM_CASE(64, 7, EPI_F16, ACT_NONE, false)
  F5_GEMM_CASE(64, 7, EPI_F16, ACT_GELU_TANH, false)
  F5_GEMM_CASE(64, 7, EPI_F16, ACT_GELU_ERF, false)
  F5_GEMM_CASE(64, 7, EPI_F32, ACT_NONE, false)
  F5_GEMM_CASE(64, 7, EPI_RESID, ACT_NONE, false)
  F5_GEMM_CASE(128, 5, EPI_F16, ACT_NONE, false)
  F5_GEMM_CASE(128, 5, EPI_F16, ACT_GELU_TANH, false)
  F5_GEMM_CASE(128, 5, EPI_F16, ACT_GELU_ERF, false)
  F5_GEMM_CASE(128, 5, EPI_F32, ACT_NONE, false)
  F5_GEMM_CASE(128, 5, EPI_RESID, ACT_NONE, false)
  F5_GEMM_CASE(256, 3, EPI_F16, ACT_NONE, false)
  F5_GEMM_CASE(256, 3, EPI_F16, ACT_GELU_TANH, false)
  F5_GEMM_CASE(256, 3, EPI_F16, ACT_GELU_ERF, false)
  F5_GEMM_CASE(256, 3, EPI_F32, ACT_NONE, false)
  F5_GEMM_CASE(256, 3, EPI_RESID, ACT_NONE, false)
  F5_GEMM_CASE(128, 5, EPI_QKV_ROPE, ACT_NONE, false)
  F5_GEMM_CASE(192, 4, EPI_QKV_ROPE, ACT_NONE, false)
  F5_GEMM_CASE(192, 4, EPI_F16, ACT_NONE, false)
  F5_GEMM_CASE(192, 4, EPI_F16, ACT_GELU_TANH, false)
  F5_GEMM_CASE(192, 4, EPI_RESID, ACT_NONE, false)
  F5_GEMM_CASE(256, 3, EPI_QKV_ROPE, ACT_NONE, false)
  F5_GEMM_CASE(64, 7, EPI_F16, ACT_MISH, true)
  F5_GEMM_CASE(64, 7, EPI_RESID, ACT_MISH, true)
  F5_GEMM_PAIR_CASE(256, 5, EPI_F16, ACT_NONE)
  F5_GEMM_PAIR_CASE(256, 5, EPI_F16, ACT_GELU_TANH)
  F5_GEMM_PAIR_CASE(256, 5, EPI_RESID, ACT_NONE)
  F5_GEMM_PAIR_CASE(256, 5, EPI_QKV_ROPE, ACT_NONE)
  F5_GEMM_PAIR_CASE(192, 6, EPI_F16, ACT_NONE)
  F5_GEMM_PAIR_CASE(192, 6, EPI_F16, ACT_GELU_TANH)
  F5_GEMM_PAIR_CASE(192, 6, EPI_RESID, ACT_NONE)
  F5_GEMM_PAIR_CASE(192, 6, EPI_QKV_ROPE, ACT_NONE)
  F5_GEMM_PAIR_CASE(128, 6, EPI_F16, ACT_NONE)
  F5_GEMM_PAIR_CASE(128, 6, EPI_F16, ACT_GELU_TANH)
  F5_GEMM_PAIR_CASE(128, 6, EPI_RESID, ACT_NONE)
  F5_GEMM_PAIR_CASE(128, 6, EPI_QKV_ROPE, ACT_NONE)
  set_error("gemm: no kernel instantiated for bn=%d epi=%d act=%d conv=%d pair=%d", pl.bn, pl.epi, pl.act, pl.conv, pl.pair);
  return -6;
}

struct TileChoice {
  int bn, pair;
};
// Tile shape of a GEMM whose caller left bn = 0.  Cost model in SM clocks, fitted to the graph-timed sweep of
// tools/gemm_sweep.py on B200 (profiles/README.md), all five tile flavours within ~5 %:
//   main loop per tile  = k-blocks x (256 + 2*BN)     single CTA 128 x BN   (shared-memory traffic bound: TMA writes +
//                         k-blocks x {474 | 640}      per CTA of a cta_group::2 256 x {128 | 256} pair (+1500 fixed)
//   epilogue per tile   = BN x {27 plain fp16 / RoPE, 32 fp32 reduce-add, 38 GELU (two warps per scheduler)} clk
//   tiles run in rounds over the SMs (SM pairs); inside a CTA the epilogue of tile i overlaps the main loop of tile
//   i+1, so a round costs max(main, epilogue) and the last tile's epilogue is exposed.
// Diagnostic build (make TRACE=1) only: F5_BN_<n_out>=<bn>[p] overrides the choice.
TileChoice pick_tile(long long rows, int batches, int n_out, int k, int epi, int act) {
#ifdef F5_TRACE
  char key[32];
  snprintf(key, sizeof key, "F5_BN_%d", n_out);
  if (const char* e = getenv(key)) {
    const int bn = atoi(e);
    if (bn == 64 || bn == 128 || bn == 192 || bn == 256) return {bn, strchr(e, 'p') != nullptr ? 1 : 0};
  }
#endif
  const int sms = num_sms();
  const double kb = double((k + 63) / 64);
  const double epi_col = (act == F5_ACT_GELU_TANH || act == F5_ACT_GELU_ERF) ? 38.0 : (epi == F5_EPI_RESID ? 32.0 : 27.0);
  // instantiated combinations only (configure_kernels)
  const bool plain = act == F5_ACT_NONE, gelu = epi == F5_EPI_F16 && act == F5_ACT_GELU_TANH;
  const bool wide_ok = (epi == F5_EPI_F16 && (plain || gelu)) || ((epi == F5_EPI_RESID || epi == F5_EPI_QKV_ROPE) && plain);
  TileChoice best{128, 0};
  double best_cost = 1e30;
  const int cand[6][2] = {{128, 0}, {192, 0}, {256, 0}, {128, 1}, {192, 1}, {256, 1}};
  for (const auto& c : cand) {
    const int bn = c[0], pair = c[1];
    if ((pair || bn == 192) && !wide_ok) continue;
    if (bn > 128 && n_out < bn) continue;
    if (pair && n_out < 256) continue;
    if (pair && bn == 192 && act == F5_ACT_GELU_ERF) continue;
    const long long tm = pair ? (rows + 255) / 256 : (rows + 127) / 128;
    const long long tiles = tm * ((n_out + bn - 1) / bn) * batches;
    const long long units = pair ? sms / 2 : sms;
    const double rounds = double((tiles + units - 1) / units);
    const double main_clk = kb * (pair ? (bn == 256 ? 640.0 : bn == 192 ? 557.0 : 474.0) : 256.0 + 2.0 * bn);
    const double epi_clk = epi_col * bn;               // exposed (last tile): latency-bound, one warp per scheduler
    const double epi_pace = epi_clk * (50.0 / 60.0);  // overlapped with the next main loop it runs a little faster
    const double cost = (rounds - 1.0) * (main_clk > epi_pace ? main_clk : epi_pace) + main_clk + epi_clk + (pair ? 1500.0 /*cluster sync, remote barrier hops*/ : 0.0);
    if (cost < best_cost) {
      best_cost = cost;
      best = {bn, pair};
    }
  }
  return best;
}

int gemm_plan(GemmPlan* pl, const void* A, const void* W, const f5_gemm_args* a) {
  memset(pl, 0, sizeof(*pl));
  const bool conv = a->conv_taps > 0;
  int bn = a->bn;
  int want_pair = a->cta_pair;
  if (conv) bn = 64;
  if (bn == 0) {  // caller leaves the tile shape to the planner
    const TileChoice tc = pick_tile(a->rows, a->batches, a->n_out, a->k, a->epi, a->act);
    bn = tc.bn;
    want_pair = tc.pair;
  }
  if (bn != 64 && bn != 128 && bn != 192 && bn != 256) {
    set_error("gemm: bn must be 64, 128, 192 or 256");
    return -1;
  }
  if (a->rows <= 0 || a->batches <= 0 || a->n_out <= 0) {
    set_error("gemm: empty problem (rows=%d batches=%d n_out=%d)", a->rows, a->batches, a->n_out);
    return -1;
  }
  // every argument is validated before the first driver call (tensor-map encoding), so a bad layout is reported as such
  if (a->epi == F5_EPI_QKV_ROPE && (a->inner % 64 || a->rope_cos == nullptr || a->rope_sin == nullptr || a->seq <= 0)) {
    set_error("gemm: QKV_ROPE needs inner %% 64 == 0, rope tables and seq");
    return -1;
  }
  if (conv) {
    if (a->n_out % 64 || a->lda < a->n_out) {
      set_error("conv gemm: channels must be a multiple of 64 (got %d, lda %d)", a->n_out, a->lda);
      return -1;
    }
  } else if (a->k <= 0 || a->lda < a->k || a->ldw < a->k) {
    set_error("gemm: bad k/lda/ldw (%d, %d, %d)", a->k, a->lda, a->ldw);
    return -1;
  }
  if (a->epi == F5_EPI_F32) {
    if (a->out == nullptr || (reinterpret_cast<uintptr_t>(a->out) & 15)) {
      set_error("gemm: fp32 epilogue needs a 16-byte aligned out (out=%p)", a->out);
      return -1;
    }
    if (a->out16b != nullptr && ((reinterpret_cast<uintptr_t>(a->out16b) & 15) || a->ldo % 8)) {
      set_error("gemm: out16b needs a 16-byte aligned pointer and ldo %% 8 == 0 (out16b=%p ldo=%d)", a->out16b, a->ldo);
      return -1;
    }
  } else if (a->epi == F5_EPI_RESID) {
    if (a->ldo % 4 || a->resid == nullptr) {
      set_error("gemm: RESID epilogue needs resid != NULL and ldo %% 4 == 0 (ldo=%d)", a->ldo);
      return -1;
    }
  } else if (a->ldo % 8 || a->out == nullptr) {
    set_error("gemm: fp16 epilogue needs out != NULL and ldo %% 8 == 0 (ldo=%d)", a->ldo);
    return -1;
  }
  pl->bn = bn;
  pl->epi = a->epi;
  pl->act = a->act;
  pl->conv = conv ? 1 : 0;
  pl->pair = (!conv && want_pair && a->epi != F5_EPI_F32 && bn >= 128) ? 1 : 0;
  GemmParams& p = pl->p;
  p.rows = a->rows;
  p.n_out = a->n_out;
  p.batches = a->batches;
  p.bias = a->bias;
  p.out = a->out;
  p.out16b = reinterpret_cast<__half*>(a->out16b);
  p.resid = a->resid;
  p.ldo = a->ldo;
  p.gate = a->gate;
  p.step_ptr = a->step_ptr;
  p.gate_step_stride = a->gate_step_stride;
  p.row_len = a->row_len;
  p.seq = a->seq;
  p.rope_cos = a->rope_cos;
  p.rope_sin = a->rope_sin;
  p.inner = a->inner > 0 ? a->inner : 64;
  p.pe_heads = a->pe_heads;
  p.conv_pad = a->conv_taps / 2;
  p.skip_pad = (a->skip_padded_tiles && a->row_len != nullptr && a->seq > 0 && (conv || a->batches == 1)) ? 1 : 0;
  // a prefetched W tile belongs to the CTA's first tile: not known to be computed when padded tiles are skipped
  p.w_prefetch = (a->weights_static && !p.skip_pad) ? 1 : 0;
#ifdef F5_TRACE
  {  // instrumented build: F5_GEMM_TRACE=1 records per-CTA phase clocks of every launch (read back by f5_debug_gemm_trace)
    static int want = -1;
    if (want < 0) {
      want = getenv("F5_GEMM_TRACE") ? 1 : 0;
      if (want) cudaMalloc(&g_trace, sizeof(long long) * 16 * 4096);
    }
    p.dbg_ts = want ? g_trace : nullptr;
  }
#endif
  int rc;
  if (conv) {
    p.num_kb = a->conv_taps;
    // activations [batches][rows][lda]: channel slice of 64 = one group
    rc = encode_tmap_f16(&pl->tmA, A, (uint64_t)a->lda, (uint64_t)a->rows, (uint64_t)a->batches, (uint64_t)a->lda * 2,
                         (uint64_t)a->rows * a->lda * 2, 64, 128, 3);
    if (rc) return rc;
    rc = encode_tmap_f16(&pl->tmB, W, 64, (uint64_t)a->conv_taps * a->n_out, 1, 128, 0, 64, 64, 2);
    if (rc) return rc;
  } else {
    p.num_kb = (a->k + kBK - 1) / kBK;
    rc = encode_tmap_f16(&pl->tmA, A, (uint64_t)a->k, (uint64_t)a->rows, (uint64_t)a->batches, (uint64_t)a->lda * 2,
                         (uint64_t)a->rows * a->lda * 2, 64, 128, 3);
    if (rc) return rc;
    rc = encode_tmap_f16(&pl->tmB, W, (uint64_t)a->k, (uint64_t)a->n_out, 1, (uint64_t)a->ldw * 2, 0, 64,
                         (uint32_t)(pl->pair ? bn / 2 : bn), 2);
    if (rc) return rc;
  }
  // output tensor map for the staged epilogues (bulk TMA store of fp16 / reduce-add of fp32); columns clip at n_out
  if (a->epi == F5_EPI_F32) {
    pl->tmC = pl->tmA;  // unused
  } else if (a->epi == F5_EPI_RESID) {
    rc = encode_tmap(&pl->tmC, 1, a->resid, (uint64_t)a->n_out, (uint64_t)a->rows, (uint64_t)a->batches,
                     (uint64_t)a->ldo * 4, (uint64_t)a->rows * a->ldo * 4, 32, 128, 3);
    if (rc) return rc;
  } else {
    rc = encode_tmap(&pl->tmC, 0, a->out, (uint64_t)a->n_out, (uint64_t)a->rows, (uint64_t)a->batches,
                     (uint64_t)a->ldo * 2, (uint64_t)a->rows * a->ldo * 2, 64, 128, 3);
    if (rc) return rc;
  }
  if (pl->pair) {
    const long long ptiles = (long long)((a->n_out + bn - 1) / bn) * ((a->rows + 2 * kBM - 1) / (2 * kBM)) * a->batches;
    const long long pairs = num_sms() / 2;
    pl->grid = dim3((unsigned)(2 * (ptiles < pairs ? ptiles : pairs)), 1, 1);  // persistent CTA pairs
    return 0;
  }
  const long long tiles = (long long)((a->n_out + bn - 1) / bn) * ((a->rows + kBM - 1) / kBM) * a->batches;
  pl->grid = dim3((unsigned)(tiles < num_sms() ? tiles : num_sms()), 1, 1);  // persistent: one CTA per SM
  return 0;
}

}  // namespace f5

extern "C" {

int f5_version(void) { return 101; }  // 101: f5_sample_args.ode_method
const char* f5_last_error(void) { return f5::g_err; }
unsigned long long f5_launch_count(void) { return f5::g_launches.load(); }

// diagnostics: copy the per-CTA timestamp trace of the last GEMM launched with F5_GEMM_TRACE=1 (8 values per CTA)
int f5_debug_gemm_trace(long long* host_out, int n_ctas) {
  if (!f5::g_trace) return -1;
  cudaDeviceSynchronize();
  return cudaMemcpy(host_out, f5::g_trace, sizeof(long long) * 16 * (size_t)n_ctas, cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : -2;
}

int f5_gemm_tile(const f5_gemm_args* args, int* bn, int* cta_pair) {
  if (!args || !bn || !cta_pair) return -1;
  int b = args->conv_taps > 0 ? 64 : args->bn, pr = args->cta_pair;
  if (b == 0) {
    const f5::TileChoice tc = f5::pick_tile(args->rows, args->batches, args->n_out, args->k, args->epi, args->act);
    b = tc.bn;
    pr = tc.pair;
  }
  *bn = b;
  *cta_pair = (args->conv_taps == 0 && pr && args->epi != F5_EPI_F32 && b >= 128) ? 1 : 0;
  return 0;
}

int f5_gemm(const void* A, const void* W, const f5_gemm_args* args, f5_stream_t stream) {
  f5::GemmPlan pl;
  if (int rc = f5::gemm_plan(&pl, A, W, args)) return rc;
  return f5::gemm_run(pl, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"

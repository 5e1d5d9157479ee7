// Internal host-side declarations shared by the translation units of libf5tts_b200.so.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include "../../include/f5tts_b200.h"
#include "kparams.h"

namespace f5 {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);
int check_cuda(cudaError_t e, const char* what);
int check_launch(const char* what);
int configure_kernels();  // cudaFuncSetAttribute for every instantiation (once per process)
int attn_configure();
int num_sms();
bool pdl_enabled();  // F5_PDL=0 disables programmatic dependent launch

// Launch with the programmatic-stream-serialization attribute (PDL); every kernel launched through this helper calls
// griddepcontrol.wait before touching global memory, so stream order is preserved transitively.
struct PdlLaunch {
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[2];
  PdlLaunch(dim3 grid, dim3 block, size_t smem, cudaStream_t s, int cluster_x = 1) {
    cfg = cudaLaunchConfig_t{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    int n = 0;
    if (cluster_x > 1) {  // CTA pair for cta_group::2 kernels
      attr[n].id = cudaLaunchAttributeClusterDimension;
      attr[n].val.clusterDim.x = (unsigned)cluster_x;
      attr[n].val.clusterDim.y = 1;
      attr[n].val.clusterDim.z = 1;
      ++n;
    }
    if (pdl_enabled()) {
      attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      attr[n].val.programmaticStreamSerializationAllowed = 1;
      ++n;
    }
    cfg.attrs = attr;
    cfg.numAttrs = n;
  }
};

struct GemmPlan {
  CUtensorMap tmA, tmB, tmC;
  GemmParams p;
  dim3 grid;
  int bn, epi, act, conv, pair;
};
int gemm_plan(GemmPlan* plan, const void* A, const void* W, const f5_gemm_args* a);
int gemm_run(const GemmPlan& plan, cudaStream_t s);

struct AttnPlan {
  CUtensorMap tm;
  AttnParams p;
  dim3 grid;
};
int attn_plan(AttnPlan* plan, const void* qkv, void* out, int batches, int seq, int heads, const int* kv_len,
              float scale);
int attn_run(const AttnPlan& plan, cudaStream_t s);

// 3-D fp16 tensor map: dims (d0 contiguous, d1, d2), byte strides for d1, d2, box (b0, b1, 1), 128B swizzle
int encode_tmap(CUtensorMap* m, int is_f32, const void* ptr, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1,
                uint64_t stride2, uint32_t b0, uint32_t b1, int rank);
int encode_tmap_f16(CUtensorMap* m, const void* ptr, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1,
                    uint64_t stride2, uint32_t b0, uint32_t b1, int rank);

}  // namespace f5

// ---- launch wrappers of the bandwidth-bound kernels (defined in ops.cu) ----
#include "ew_params.h"
namespace f5 {
int run_row_norm(int mode, const NormParams& p, cudaStream_t s);
int run_dwconv7_ln(const DwConvLnParams& p, cudaStream_t s);
int run_text_gather(const TextGatherParams& p, cudaStream_t s);
int run_mask_rows(float* x, const uint8_t* filler, int BN, int rows, int C, cudaStream_t s);
int run_mask_rows_len(float* x, const int* valid_len, int B, int N, int rows, int C, cudaStream_t s);
int run_mask_rows_len_half(__half* x, const int* valid_len, int B, int N, int rows, int C, cudaStream_t s);
constexpr int kGrnRows = 64;  // sequence rows per partial-sum block
int run_grn(__half* g, float* partial, float* nx, const float* gamma, const float* beta, int B, int N, int C,
            cudaStream_t s);
int run_pack_input(const PackParams& p, cudaStream_t s);
int run_cfg_update(const UpdateParams& p, cudaStream_t s);
int run_small_linear(int act, const float* in, const __half* W, const float* bias, float* out, int S, int K, int Nout,
                     cudaStream_t s);
int run_time_features(const float* t, float* feat, int S, int dim, cudaStream_t s);
int run_silu_to_half(const float* in, __half* out, long long n, cudaStream_t s);
int run_rope_table(float* cs, float* sn, int seq, int half, cudaStream_t s);
int run_prepend_time_token(float* dst, const float* src, const float* t_emb, const int* step_ptr, int N, int D,
                           long long rows_out, cudaStream_t s);
int run_concat_half(const float* x, const float* skip, __half* out, long long rows, int D, cudaStream_t s);
}  // namespace f5

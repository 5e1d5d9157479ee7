// Parameter blocks of the bandwidth-bound kernels (plain structs shared between ops.cu and engine.cu).
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

namespace f5 {

struct NormParams {
  const float* x;
  __half* out;
  int rows, D;
  float eps;
  const float* a;  // MODE0: scale  MODE1: weight  MODE2: g
  const float* b;  // MODE0: shift  MODE1: bias
  const int* step_ptr;
  long long step_stride;
  int params_static;  // a / b / *step_ptr were not written by the kernel preceding this launch: fetch them before the PDL wait
};

struct DwConvLnParams {
  const float* x;   // [B, N, C]
  __half* out;      // [B*N, C]
  int B, N, C;
  const float* w;   // [C, 7]
  const float* wb;  // [C]
  const float* ln_w;
  const float* ln_b;
  float eps;
};

struct TextGatherParams {
  const long long* ids;  // [B, nt] padded with -1
  int B, nt, N, Td;
  const int* valid_len;  // [B] per-sample valid positions or null
  const float* table;    // [V+1, Td]
  int num_embeds;        // V + 1 rows; ids outside [0, V] are clamped (the reference's nn.Embedding raises; the host
                         // side validates ids before the call)
  int add_pos;           // conv_layers > 0
  float* out;            // [2B, N, Td]
  uint8_t* filler;       // [B, N]
};

struct PackParams {
  __half* xin;
  int B, N, mel, Td, Kpad, packed;  // packed: 1 = cond + uncond halves
  const float* y;          // [B, N, mel] current state
  const float* step_cond;  // [B, N, mel]
  const float* text;       // [2B, N, Td] fp32 (cond variant first)
};

// Caller-owned tensors and scalars of one sample() call.  The step kernels read them from this block inside the
// workspace (written by the prologue), so a captured step graph does not bake the caller's pointers in.
struct SampleIo {
  float* y;     // [B*N, mel] ODE state
  float* traj;  // [steps+1, B*N, mel] or null
  float cfg;    // classifier-free-guidance scale
};

// One entry per backbone evaluation of a sample() call, indexed by the device counter.  The update kernel forms
// x = y + coef * g (g: CFG-combined velocity) and writes fp16(x) into the next evaluation's input; commit >= 0 also stores
// x as the ODE state y and as trajectory[commit], commit = -1 leaves y (the state at the start of the grid step) as it is.
//   Euler:    {dt_k, k + 1}
//   midpoint: {dt_k / 2, -1}, {dt_k, k + 1}   (torchdiffeq: y_mid = y + f0 * dt/2, y + dt * f(t_k + dt/2, y_mid))
struct OdeStage {
  float coef;
  int commit;
};

struct UpdateParams {
  const SampleIo* io;
  const float* v;  // [Be*N, mel]
  __half* xin;
  const OdeStage* stages;  // [evaluations] device
  int* step_ptr;
  int BN, mel, Kpad, packed;
  int N;         // frames per sample
  int seq_tok;   // rows per sample in v (N for DiT, N + 1 for UNetT)
  int tok_off;   // first frame row inside a sample of v (0 DiT, 1 UNetT: skips the time token, unett.py:305)
  int B;
};

}  // namespace f5

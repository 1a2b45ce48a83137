// tcgen05 / TMEM / TMA kernel for one observation-propagation layer (rd_obprop_tc.cu).
#pragma once
#include "rd_common.cuh"

namespace rd {

// true when the tensor-core kernel handles this layer shape (C = T*d_ob channels)
bool obprop_tc_supported(int C);

// out[r, :] = epi(x[r, :] . W^T), W: [C, C] row-major ([out, in]); TF32 operands, fp32 accumulation
// in TMEM.  The tensor core reads the top 19 bits of each fp32 operand (truncation), so callers
// hand in operands that are already rounded to TF32 (round_tf32 below / round_out of the producing
// layer); then the truncation is exact and the only error is the unbiased RN rounding.
//   epi(v) = [relu](v + bias[c]) * scale[r % mod] * [gate[r, c] > 0], optionally RN-rounded to TF32
// perm != 0: store into the encoder input [T, B, D] instead of [rows, C] (needs d_ob == 4):
//   row r = b*pN + n, col c = t*4 + k  ->  out[((t*pB + b)*pD) + n*4 + k]
struct ObpropTcArgs {
  const float* x = nullptr; const float* W = nullptr; const float* bias = nullptr;
  // non-null selects the error-compensated mode (3xTF32, fp32-level accuracy): W_lo = W - trunc19(W), same shape as
  // W; x and W are then taken as they are (no TF32 pre-rounding needed) and round_out must be 0
  const float* W_lo = nullptr;
  const float* scale = nullptr; int scale_mod = 1;
  const float* gate = nullptr;      // [rows, C] or null (plain layout only)
  int relu = 1, round_out = 0;
  int64_t rows = 0; int C = 0; float* out = nullptr;
  int perm = 0, pB = 0, pN = 0, pdob = 0, pD = 0;
  // lift_ru != null: backward of the input lift X0 = dropout(relu(v * R_u)) (needs d_ob == 4, gate = X0, W_lo, no
  // bias / relu / scale): row r = b*pN + n, col c = t*4 + k  ->
  //   out[(t*pB + b)*pD + n] = lift_scale * sum_k acc[r, 4t+k] * R_u[4n+k] * [gate[r, 4t+k] != 0]
  const float* lift_ru = nullptr; float lift_scale = 1.f;
};
int obprop_tc_fwd(const ObpropTcArgs& a, cudaStream_t st);
// Which mode a [rows, C] layer should run in (mode: 0 automatic, 1 single-pass TF32, 2 error-compensated).  Automatic =
// error-compensated while 3x the tensor work still hides behind launch latency (2*rows*C^2 <= 2 GFLOP), single
// pass TF32 in the HBM-/tensor-bound regime where it is what reaches the roofline.
bool obprop_tc_exact(int64_t rows, int C, int mode);

// y[i] = RN_tf32(x[i])
int round_tf32(const float* x, int64_t n, float* y, cudaStream_t st);

}  // namespace rd

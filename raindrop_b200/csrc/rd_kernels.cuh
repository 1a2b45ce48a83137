// Launch wrappers for the non-GEMM kernels of the hot path (rd_kernels.cu).
#pragma once
#include "rd_common.cuh"

namespace rd {

// out[t, j, :] = src[t, idx[j], :] for a device-resident training set (code/Raindrop.py:311-315 does this on the host)
int gather_batch(const float* src, const int64_t* idx, int64_t T, int64_t n_total, int width, int B, float* out,
                 cudaStream_t st);

int rng_capture(uint64_t* rng_state, uint64_t* captured, int advance, cudaStream_t st);

// device-side input pipeline (rd_kernels.cu; mirrors code/utils_rd.py:149-175,221-257 and code/Raindrop.py:214-231,311-317)
int64_t feature_stats_scratch_bytes(int64_t n, int T, int F);
int feature_stats(const float* raw, int64_t n, int T, int F, float* mean, float* stdv, void* scratch, cudaStream_t st);
int mask_normalize(const float* raw, const float* mean, const float* stdv, int64_t n, int T, int F, float* out,
                   const float* minutes, float* times_out, cudaStream_t st);
int zero_features(float* P, int64_t T, int B, int width, const int64_t* idx, int K, int per_sample, cudaStream_t st);
int assemble_batch(const float* P, const float* Pt, const float* Ps, const int64_t* y, const int64_t* idx, int T, int64_t n_total,
                   int width, int ds, int B, float* src, float* times, float* statics, int64_t* y_out, int64_t* lengths,
                   cudaStream_t st);

// X0[(b*N+n), t*d_ob+k] = dropout(relu(src[t,b,n] * R_u[n*d_ob+k]))    code/models_rd.py:285-296,323-327
// round != 0: values are rounded (RN) to TF32 so the tensor-core layer reads them exactly.
// The same launch writes the positional encoding of `times` into pe_out[tok*ld + col0 ..+16] (src == nullptr
// or times == nullptr skips that half).
int lift_posenc(const float* src, const float* R_u, int B, int T, int N, int d_ob, float drop_p, const uint64_t* rng,
                int round, float* X0, const float* times, int64_t n_tokens, const float* ts_host, int d_pe, float* pe_out,
                int64_t ld, int col0, cudaStream_t st);

// y [cols, rows] = RN_tf32(x [rows, cols])^T
int transpose_round(const float* x, int rows, int cols, float* y, cudaStream_t st);

int posenc(const float* times, int64_t n_tokens, const float* ts_host, int d_pe, float* out, int64_t ld, int col0,
           cudaStream_t st);

int node_scale(const int64_t* edge_tgt, const float* edge_w, int E, int N, float* s, cudaStream_t st);

// y = LN(x) * gamma + beta over the last dim (width D); stats[row] = {mean, rstd}
int layernorm_fwd(const float* x, const float* gamma, const float* beta, int64_t rows, int D, float eps,
                  float* y, float* stats, cudaStream_t st);
// dx from dy; dgamma/dbeta via partials. scratch >= ln_bwd_scratch_floats(rows, D)
int64_t ln_bwd_scratch_floats(int64_t rows, int D);
// dx_drop (optional, used when drop_p > 0): dx with the dropout mask of `site` re-applied, i.e. the
// gradient w.r.t. the sub-layer output that was dropped before the residual add
// deferred_chunks != nullptr: the reduction of the per-CTA partial rows scratch[chunks][2][D] is left to the caller
// (*deferred_chunks = chunks), who folds it into a later grouped reduction launch (tc_wgrad_group)
int layernorm_bwd(const float* x, const float* stats, const float* gamma, const float* dy, int64_t rows,
                  int D, float* dx, float* dgamma, float* dbeta, float* scratch, float* dx_drop, float drop_p,
                  const uint64_t* rng, uint32_t site, int* deferred_chunks, cudaStream_t st,
                  const uint32_t* keep_bits = nullptr, int keep_ld = 0);   // keep_bits: decisions stored by the forward (else Philox)

// in-place masked softmax over rows of S [B,H,T,T]; key j masked when j >= lengths[b].
// If Pd != nullptr also writes the dropped probabilities (training).
int attn_softmax_fwd(float* S, const int64_t* lengths, int B, int H, int T, float drop_p,
                     const uint64_t* rng, uint32_t site, float* Pd, cudaStream_t st);
// dS = P * (dP - sum_j dP_j P_j), dP = dPd * mask/(1-p); in place on dP
int attn_softmax_bwd(const float* P, float* dP, int B, int H, int T, float drop_p, const uint64_t* rng,
                     uint32_t site, cudaStream_t st);

// fused pooling + classification head (rd_head.cu).  x = encoder output [T, B, D]; writes feat [B, Df], hpre [B, Df],
// logits [B, ncls]; with labels y also the per-sample losses, d(loss)/d(logits) of the batch-mean CrossEntropy and
// the scalar loss (summed by the last CTA, ticket in *counter which must be 0 on entry).
int head_fwd(int B, int T, int D, int N, int ds, int ncls, const float* x, const int64_t* lengths, const float* statics,
             const float* emb_w, const float* emb_b, const float* w0, const float* b0, const float* w2, const float* b2,
             float* feat, float* hpre, float* logits, const int64_t* y, float* loss_ps, float* dlogits, float* loss,
             unsigned* counter, cudaStream_t st);
// dx = d(loss)/d(encoder output) [T, B, D] (masked-mean backward); g_w0 == null: no parameter gradients (no second launch)
int head_bwd(int B, int T, int D, int N, int ds, int ncls, const int64_t* lengths, const float* statics, const float* w0,
             const float* w2, const float* feat, const float* hpre, const float* dlogits, float* dh, float* dfeat, float* dx,
             float* g_w0, float* g_b0, float* g_w2, float* g_b2, float* g_emb_w, float* g_emb_b, cudaStream_t st);

// fused attention for short sequences (rd_attn_small.cu): ctx from qkv in one launch, dqkv in one launch
bool attn_small_supported(int T, int hd);
int attn_small_fwd(const float* qkv, const int64_t* lengths, int B, int H, int T, int hd, float drop_p,
                   const uint64_t* rng, uint32_t site, float* ctx, cudaStream_t st);
int attn_small_bwd(const float* qkv, const float* dctx, const int64_t* lengths, int B, int H, int T, int hd,
                   float drop_p, const uint64_t* rng, uint32_t site, float* dqkv, cudaStream_t st);

// the same on the tensor cores (rd_attn_tc.cu: tcgen05 3xTF32, TMA-staged head slices, T <= 64, hd <= 96, hd % 4 == 0)
bool attn_tc_supported(int T, int hd);
void attn_tc_set_debug(unsigned long long* buf);   // phase timestamps of the forward kernel: [CTA][16] (debug)
int attn_tc_fwd(const float* qkv, const int64_t* lengths, int B, int H, int T, int hd, float drop_p,
                const uint64_t* rng, uint32_t site, float* ctx, cudaStream_t st);
int attn_tc_bwd(const float* qkv, const float* dctx, const int64_t* lengths, int B, int H, int T, int hd,
                float drop_p, const uint64_t* rng, uint32_t site, float* dqkv, cudaStream_t st);

// dZ2[(b*N+n), t*d_ob+k] = dZ[t,b,n*d_ob+k] * s[n] * (Z[t,b,n*d_ob+k] > 0)
int obprop_out_grad(const float* dZ, const float* Z, const float* s, int B, int T, int N, int d_ob, int D,
                    int round, float* dZ2, cudaStream_t st);

// Input gradients of Raindrop_v2 that need no GEMM, one launch (each output may be null):
//   d_src [T, B, 2N]: mask half zeroed; value half from dX0 [B*N, T*d_ob] (gated, scaled: the CUDA-core fallback of the
//                     lift backward) when dX0 != null, else left to the tensor-core store
//   d_times [T, B]  : from dZ / Z [T, B, D] (the encoder input's last d_pe columns are sin | cos of times / ts_host[j])
//   d_static [B, ds]: dfeat[b, D : D+emb] . emb_w [emb, ds]   (dfeat [B, Df] from head_bwd; emb = N for Raindrop_v2,
//                     d_model for legacy Raindrop v1)
int input_grad_tail(int B, int T, int N, int d_ob, int D, const float* dZ, const float* Z, const float* ts_host,
                    int d_pe, const float* dfeat, int Df, const float* emb_w, int emb, int ds, const float* dX0,
                    const float* R_u, float* d_src, float* d_times, float* d_static, cudaStream_t st);
// d_times[tok] from the saved encoding pe and its gradient d_pe (both at [tok*ld + col0 + 0..width)): the times branch of
// the same kernel on its own (no trigonometry: d sin = cos / ts, d cos = -sin / ts)
int posenc_bwd(const float* pe, const float* d_pe, int64_t n_tokens, const float* ts_host, int width, int64_t ld, int col0,
               float* d_times, cudaStream_t st);

// y[i] = x[i] * mask(site, i)   (re-generates the forward's dropout mask)
int apply_dropout(const float* x, int64_t n, float p, const uint64_t* rng, uint32_t site, float* y,
                  cudaStream_t st);

// d_pre = d_out * scale[r % mod] * (out > 0)
int relu_scale_bwd(const float* d_out, const float* out, const float* scale, int mod, int64_t rows, int C,
                   float* d_pre, cudaStream_t st);

int cross_entropy(const float* logits, const int64_t* y, int B, int ncls, float* loss, float* dlogits,
                  cudaStream_t st);
// step: int64[2] = {count, ticket}; the ticket word must be 0 on entry (it is reset by the launch).  The count is
// incremented by the last CTA of the launch, so one launch does tick + update.  lr_dev (optional, device) overrides lr.
int adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, const float* lr_dev, float b1, float b2,
         float eps, float gscale, int64_t* step, cudaStream_t st);

}  // namespace rd

/*
 * raindrop_b200.h -- C ABI of librd_b200.so (sm_100a), the device side of the Raindrop hot path.
 *
 * The reference (mims-harvard/Raindrop) is pure Python; it has no FFI of its own.  The boundary
 * a maintainer binds is therefore the set of Python call sites listed beside each entry point
 * (paths relative to the reference tree).  Our `raindrop_b200/models_rd.py` binds them through
 * ctypes; INTEGRATION.md shows the same stubs applied to the reference's own files.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; all tensors are dense,
 *     row-major fp32 (indices int64) exactly as the reference's torch tensors are laid out;
 *   - `stream` is a cudaStream_t passed as void*; every call is stream-ordered, allocation-free
 *     and sync-free (CUDA-graph capturable).  Scratch memory is provided by the caller: query
 *     the size first;
 *   - return value 0 = ok, negative = error (rd_last_error_string() describes it); nothing
 *     throws across the ABI.
 */
#ifndef RAINDROP_B200_H
#define RAINDROP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RD_ABI_VERSION 2
#define RD_MAX_LAYERS 8
#define RD_D_PE 16 /* d_pe, code/models_rd.py:215 */

/* Shapes of one Raindrop_v2 instance + one batch (code/models_rd.py:208-264, 278-284). */
typedef struct rd_dims {
  int32_t B;         /* samples in this batch (any >= 1)                                  */
  int32_t T;         /* max_len                                                           */
  int32_t N;         /* d_inp = sensors                                                   */
  int32_t d_ob;      /* d_model / d_inp (4 in code/Raindrop.py:125)                       */
  int32_t nhead;     /* temporal attention heads                                          */
  int32_t nhid;      /* feed-forward width                                                */
  int32_t nlayers;   /* encoder layers (<= RD_MAX_LAYERS)                                 */
  int32_t d_static;  /* 0 = no static branch (static=False)                               */
  int32_t n_classes;
  int32_t training;  /* 1: dropout active (model.train()), 0: eval                        */
  float dropout_p;   /* one p for every dropout site, as in the reference                 */
  float ln_eps;      /* 1e-5                                                              */
  float pe_timescales[RD_D_PE / 2]; /* max_len ** linspace(0,1,8) computed in fp64 on host,
                                       cast to fp32 (code/models_rd.py:31,34)             */
  int32_t d_pe;        /* width of the positional encoding concatenated to the encoder input; 0 = 16 (Raindrop_v2,
                          code/models_rd.py:215).  Legacy Raindrop v1 uses 36 (code/models_rd.py:68); only the
                          rd_encoder_head_* entry points accept values other than 16                              */
  int32_t emb_dim;     /* width of emb = Linear(d_static, emb_dim): 0 = N (Raindrop_v2, code/models_rd.py:224);
                          d_model for legacy Raindrop v1 (code/models_rd.py:98)                                    */
  int32_t obprop_mode; /* arithmetic of the two observation-propagation GEMMs on the tensor cores:
                          0 = automatic: error-compensated 3xTF32 (fp32-level, gradients match the fp32 reference
                              to ~1e-3) while 2*B*N*C^2 <= 2 GFLOP per layer, i.e. where the layer is launch-latency
                              bound anyway; single-pass TF32 (operands rounded to TF32, forward error ~3e-4) above,
                              where it is what reaches the HBM / tensor roofline
                          1 = always single-pass TF32        2 = always 3xTF32                          */
} rd_dims;

/* Parameters that take part in the live path (SURVEY.md 8a18).  Names = state-dict keys. */
typedef struct rd_encoder_layer_params {
  const float* in_proj_weight;  /* [3D, D] */
  const float* in_proj_bias;    /* [3D]    */
  const float* out_proj_weight; /* [D, D]  */
  const float* out_proj_bias;   /* [D]     */
  const float* linear1_weight;  /* [nhid, D] */
  const float* linear1_bias;    /* [nhid]  */
  const float* linear2_weight;  /* [D, nhid] */
  const float* linear2_bias;    /* [D]     */
  const float* norm1_weight;    /* [D] */
  const float* norm1_bias;
  const float* norm2_weight;
  const float* norm2_bias;
} rd_encoder_layer_params;

typedef struct rd_params {
  const float* R_u;             /* [1, N*d_ob]  plain tensor, code/models_rd.py:241          */
  const float* emb_weight;      /* [N, d_static] or NULL                                     */
  const float* emb_bias;        /* [N] or NULL                                               */
  const float* ob1_value_weight;/* ob_propagation.lin_value.weight        [C, C], C=T*d_ob   */
  const float* ob1_value_bias;  /* [C] */
  const float* ob2_value_weight;/* ob_propagation_layer2.lin_value.weight [C, C]             */
  const float* ob2_value_bias;
  const float* mlp0_weight;     /* mlp_static.0.weight [Df, Df], Df = D + (static ? N : 0)   */
  const float* mlp0_bias;
  const float* mlp2_weight;     /* mlp_static.2.weight [n_classes, Df]                       */
  const float* mlp2_bias;
  rd_encoder_layer_params layer[RD_MAX_LAYERS];
} rd_params;

/* Same members, writable: gradients (written, not accumulated).  R_u gets no gradient. */
typedef struct rd_encoder_layer_grads {
  float* in_proj_weight; float* in_proj_bias; float* out_proj_weight; float* out_proj_bias;
  float* linear1_weight; float* linear1_bias; float* linear2_weight; float* linear2_bias;
  float* norm1_weight; float* norm1_bias; float* norm2_weight; float* norm2_bias;
} rd_encoder_layer_grads;

typedef struct rd_grads {
  float* emb_weight; float* emb_bias;
  float* ob1_value_weight; float* ob1_value_bias;
  float* ob2_value_weight; float* ob2_value_bias;
  float* mlp0_weight; float* mlp0_bias; float* mlp2_weight; float* mlp2_bias;
  rd_encoder_layer_grads layer[RD_MAX_LAYERS];
} rd_grads;

/* Named views into the activation workspace written by rd_raindrop_v2_fwd (for parity tests). */
enum rd_ws_buffer {
  RD_WS_X0 = 0,    /* lifted input   [B*N, C]  (code/models_rd.py:290-296,326-327)          */
  RD_WS_H1 = 1,    /* layer-1 output [B*N, C]  (code/models_rd.py:329-330)                  */
  RD_WS_ENC_IN = 2,/* cat(obs, pe)   [T, B, D] (code/models_rd.py:341,354)                  */
  RD_WS_ENC_OUT = 3,/* r_out         [T, B, D] (code/models_rd.py:358)                      */
  RD_WS_FEAT = 4,  /* cat(pooled, emb) [B, Df] (code/models_rd.py:379,384)                  */
  RD_WS_RNG = 5    /* 2 x uint64 (seed, step counter) captured by this forward              */
};

int rd_abi_version(void);
const char* rd_last_error_string(void);
/* number of kernels this library has launched so far in this process (host-side counter; a
 * CUDA-graph replay re-runs captured launches without passing through here) */
uint64_t rd_launch_count(void);

/* ---- graph prologue --------------------------------------------------------------------
 * s[n] = sum_{e: tgt[e]==n} softmax_{e->n}(w)   with PyG's  exp(w-max)/(sum+1e-16).
 * Replaces `softmax(gamma, index)` + `scatter(..., reduce='add')` of
 * code/Ob_propagation.py:195,226-228 for the live path where the message depends on the
 * target only (code/Ob_propagation.py:200).  edge_tgt = edge_index[1] (code/models_rd.py:310). */
int rd_node_scale(const int64_t* edge_tgt, const float* edge_w, int32_t E, int32_t N,
                  float* node_scale, void* stream);

/* ---- one observation-propagation layer (operator level) -----------------------------------
 * out[r, :] = relu(x[r, :] . W^T + b) * node_scale[r % scale_mod]      x, out: [rows, C]
 * Replaces Observation_progation.forward with use_beta=False (code/Ob_propagation.py:94-132,
 * 157-160,187-211,213-228) for `rows / N` samples at once (code/models_rd.py:322-336).
 * The tensor cores take TF32 operands: x and weight are first rounded (RN) into `scratch`
 * (rd_obprop_fwd_scratch_bytes(rows, C) bytes); accumulation is fp32.  scratch == NULL promises that
 * x and weight are already TF32-representable (low 13 mantissa bits zero): no rounding pass. */
size_t rd_obprop_fwd_scratch_bytes(int64_t rows, int32_t C);
int rd_obprop_fwd(const float* x, const float* weight, const float* bias, const float* node_scale,
                  int32_t scale_mod, int64_t rows, int32_t C, float* out, void* scratch, void* stream);

/* Backward of the above.  d_out, out: [rows, C].  Writes d_x (may be NULL), d_weight, d_bias.
 * scratch: rd_obprop_bwd_scratch_bytes(rows, C) bytes. */
size_t rd_obprop_bwd_scratch_bytes(int64_t rows, int32_t C);
int rd_obprop_bwd(const float* x, const float* out, const float* d_out, const float* weight,
                  const float* node_scale, int32_t scale_mod, int64_t rows, int32_t C,
                  float* d_x, float* d_weight, float* d_bias, void* scratch, void* stream);

/* Observation_progation.forward with use_beta=True (code/Ob_propagation.py:161-186,191,195-228; dormant in
 * Raindrop_v2, code/models_rd.py:317, but part of the operator's API).  One sample: x [N, C=T*d_ob],
 * p_t [T, 16].  Keeps the K = E/2 edges with the highest mean gamma (in that order), regroups them by
 * SOURCE for the per-channel segment softmax and scatters to the source (as the reference does).
 * Outputs: out [N, C]; pruned edge list edge_src_out/edge_tgt_out [K]; alpha_out [K].  Forward only. */
size_t rd_obprop_beta_scratch_bytes(int32_t N, int32_t T, int32_t d_ob, int32_t E);
int rd_obprop_beta_fwd(const float* x, const float* p_t, const int64_t* edge_src, const int64_t* edge_tgt,
                       const float* edge_w, int32_t E, int32_t N, int32_t T, int32_t d_ob,
                       const float* increase_dim_w, const float* increase_dim_b, const float* map_weights,
                       const float* value_w, const float* value_b, float* out, int64_t* edge_src_out,
                       int64_t* edge_tgt_out, float* alpha_out, void* scratch, void* stream);

/* Backward of rd_obprop_beta_fwd (same inputs; the forward is recomputed; the top-K edge selection is piecewise
 * constant and carries no gradient).  d_out [N, C]; d_alpha [K] or NULL = gradient w.r.t. the returned alpha (mean
 * gamma of the kept edges, which becomes layer 2's edge weights in code/models_rd.py:332-336).  Writes d_x [N, C]
 * (may be NULL), d_edge_w [E], d_p_t [T, 16] (may be NULL), d_increase_dim_{w [8C, C], b [8C]}, d_map_weights [N, 16],
 * d_value_{w [C, C], b [C]} -- the tensors autograd reaches through code/Ob_propagation.py:161-211.
 * scratch: rd_obprop_beta_bwd_scratch_bytes(N, T, d_ob, E) bytes. */
size_t rd_obprop_beta_bwd_scratch_bytes(int32_t N, int32_t T, int32_t d_ob, int32_t E);
int rd_obprop_beta_bwd(const float* x, const float* p_t, const int64_t* edge_src, const int64_t* edge_tgt,
                       const float* edge_w, int32_t E, int32_t N, int32_t T, int32_t d_ob,
                       const float* increase_dim_w, const float* increase_dim_b, const float* map_weights,
                       const float* value_w, const float* value_b, const float* d_out, const float* d_alpha,
                       float* d_x, float* d_edge_w, float* d_p_t, float* d_increase_dim_w, float* d_increase_dim_b,
                       float* d_map_weights, float* d_value_w, float* d_value_b, void* scratch, void* stream);

/* ---- whole Raindrop_v2 forward / backward ---------------------------------------------------
 * Replaces Raindrop_v2.forward (code/models_rd.py:278-387) for the live configuration
 * (sensor_wise_mask=False, aggreg='mean', use_beta=False) and its autograd backward
 * (code/Raindrop.py:323).
 *   src     [T, B, 2N]   times [T, B]   lengths [B] int64   statics [B, d_static] or NULL
 *   node_scale [N]       from rd_node_scale on the model's graph
 *   rng_state  2 x uint64 on the device: {seed, counter}; the forward copies it into the
 *              workspace and increments the counter (only when training && dropout_p > 0)
 *   workspace  rd_workspace_bytes(dims) bytes, kept by the caller until backward is done
 *   logits  [B, n_classes]
 *   y       optional int64 labels [B]: when given, the head kernel also evaluates
 *           torch.nn.CrossEntropyLoss (mean) -- code/Raindrop.py:322 -- writing the scalar `loss` and
 *           `d_logits` [B, n_classes] = d(loss)/d(logits), ready for rd_raindrop_v2_bwd.  NULL: plain forward
 *           (loss / d_logits ignored).                                                            */
size_t rd_workspace_bytes(const rd_dims* dims);
size_t rd_backward_scratch_bytes(const rd_dims* dims);
/* offset (bytes) and element count of a named buffer inside the workspace; -1 if unknown */
int64_t rd_workspace_offset(const rd_dims* dims, int32_t which, int64_t* n_floats);

int rd_raindrop_v2_fwd(const rd_dims* dims, const rd_params* params, const float* src,
                       const float* statics, const float* times, const int64_t* lengths,
                       const float* node_scale, uint64_t* rng_state, void* workspace,
                       float* logits, const int64_t* y, float* loss, float* d_logits, void* stream);

/* Backward (autograd of the above, code/Raindrop.py:323).  `phases` selects what one call does so that a
 * data-parallel caller can start reducing the first gradient bucket while the rest is still being computed
 * (SURVEY.md 8e):
 *   RD_BWD_ENCODER  head + temporal-attention encoder: every gradient except the two lin_value pairs is final
 *                   when the call's work completes; d(loss)/d(encoder input) stays in `scratch`
 *   RD_BWD_OBPROP   observation propagation: ob1/ob2 lin_value gradients (needs the same scratch, after ENCODER)
 *   both (3)        whole backward, weight gradients in one grouped tensor-core launch                    */
#define RD_BWD_ENCODER 1
#define RD_BWD_OBPROP 2
#define RD_BWD_ALL 3
int rd_raindrop_v2_bwd(const rd_dims* dims, const rd_params* params, const float* statics,
                       const int64_t* lengths, const float* node_scale, const void* workspace,
                       const float* d_logits, const rd_grads* grads, void* scratch, int32_t phases,
                       void* stream);

/* Gradients with respect to the float inputs of Raindrop_v2.forward (code/models_rd.py:278-296, 33-35), written, not
 * accumulated.  Any member may be NULL (not wanted).
 *   src     [T, B, 2N]   value half through the lift relu(v * R_u) and its dropout; the mask half is exactly 0
 *   statics [B, d_static] through emb (needs d_static > 0)
 *   times   [T, B]       through the positional encoding                                                      */
typedef struct rd_input_grads {
  float* src;
  float* statics;
  float* times;
} rd_input_grads;
/* bytes of `in_scratch` for rd_raindrop_v2_bwd_inputs (W1^T with its remainder, or the fallback's d(lifted input)) */
size_t rd_input_grad_scratch_bytes(const rd_dims* dims);
/* The whole backward of rd_raindrop_v2_fwd with input gradients.  grads == NULL: no parameter gradient is computed
 * (frozen model, attribution): the weight-gradient GEMMs, LayerNorm column sums and head parameter outputs are
 * skipped.  grads != NULL: every parameter gradient is bit-identical to rd_raindrop_v2_bwd(..., RD_BWD_ALL).
 * scratch: rd_backward_scratch_bytes(dims) bytes; in_scratch: rd_input_grad_scratch_bytes(dims) bytes. */
int rd_raindrop_v2_bwd_inputs(const rd_dims* dims, const rd_params* params, const float* statics,
                              const int64_t* lengths, const float* node_scale, const void* workspace,
                              const float* d_logits, const rd_grads* grads, const rd_input_grads* in_grads,
                              void* scratch, void* in_scratch, void* stream);

/* ---- temporal encoder + pooling + head on a caller-provided encoder input ------------------------------------
 * The second half of Raindrop_v2.forward (code/models_rd.py:354-385) and all of legacy Raindrop v1 after its
 * per-sample TransformerConv (code/models_rd.py:168-191): nn.TransformerEncoder with key-padding mask, masked mean
 * (divisor lengths + 1), concat emb(static), mlp_static.  The caller writes the encoder input cat(features, pe)
 * [T, B, D = N*d_ob + d_pe] into the workspace buffer RD_WS_ENC_IN first (rd_workspace_offset), then calls _fwd;
 * _bwd fills every encoder / emb / mlp_static gradient of `grads` (the ob-prop members are ignored) and writes
 * d(loss)/d(encoder input) to d_enc_in [T, B, D].  Same workspace / scratch sizes and rng protocol as
 * rd_raindrop_v2_fwd / _bwd. */
int rd_encoder_head_fwd(const rd_dims* dims, const rd_params* params, const float* statics, const int64_t* lengths,
                        uint64_t* rng_state, void* workspace, float* logits, const int64_t* y, float* loss,
                        float* d_logits, void* stream);
int rd_encoder_head_bwd(const rd_dims* dims, const rd_params* params, const float* statics, const int64_t* lengths,
                        const void* workspace, const float* d_logits, const rd_grads* grads, void* scratch,
                        float* d_enc_in, void* stream);
/* rd_encoder_head_bwd plus d_statics [B, d_static] = d(loss)/d(statics) through emb (code/models_rd.py:134,188), written,
 * not accumulated (may be NULL; needs d_static > 0).  d_enc_in may be NULL when only d_statics is wanted.  grads == NULL:
 * no parameter gradient is computed (frozen model, attribution): the weight-gradient GEMMs, LayerNorm column sums and
 * head parameter outputs are skipped, and with d_enc_in also NULL the encoder layers are not visited at all.  grads !=
 * NULL: every parameter gradient and d_enc_in are bit-identical to rd_encoder_head_bwd. */
int rd_encoder_head_bwd_inputs(const rd_dims* dims, const rd_params* params, const float* statics, const int64_t* lengths,
                               const void* workspace, const float* d_logits, const rd_grads* grads, float* d_enc_in,
                               float* d_statics, void* scratch, void* stream);
/* y[i] = x[i] * keep(site, i) / (1 - p): nn.Dropout driven by the library's counter-based stream (rng_captured =
 * {seed, counter} on the device).  The same call on a gradient is its backward. */
int rd_dropout(const float* x, int64_t n, float p, const uint64_t* rng_captured, uint32_t site, float* y, void* stream);

/* ---- pieces exposed on their own (module-level drop-ins and tests) -------------------------
 * pe[t,b,:] = [sin(times/ts_k), cos(times/ts_k)], k < d_pe/2 (d_pe <= 64)  -> out[(t*B+b)*ld + col0 + 0..d_pe-1]
 * Replaces PositionalEncodingTF.getPE (code/models_rd.py:28-37) without the host round trip. */
int rd_positional_encoding(const float* times, int64_t n_tokens, const float* timescales_host, int32_t d_pe,
                           float* out, int64_t ld, int32_t col0, void* stream);
/* Its backward: d_times[tok] = sum_j (d_sin_j cos_j - d_cos_j sin_j) / ts_j, from the saved encoding pe and its gradient
 * d_pe (both laid out as `out` above: [tok*ld + col0 + 0..d_pe_width-1]; d_pe_width even, <= 64).  No trigonometry: the
 * sin / cos columns of the forward are the derivative.  d_times [n_tokens], written, not accumulated. */
int rd_positional_encoding_bwd(const float* pe, const float* d_pe, int64_t n_tokens, const float* timescales_host,
                               int32_t d_pe_width, int64_t ld, int32_t col0, float* d_times, void* stream);

/* out[rows, out_f] = [relu](x[rows, in_f] . weight[out_f, in_f]^T + bias): the encoder's projection
 * GEMM on its own (torch.nn.Linear inside nn.TransformerEncoderLayer, code/models_rd.py:232-237).
 * Error-compensated TF32 on the tensor cores (fp32-level accuracy) when in_f % 4 == out_f % 4 == 0,
 * CUDA cores otherwise.  scratch: rd_linear_scratch_bytes(in_f, out_f) bytes (weight remainder). */
size_t rd_linear_scratch_bytes(int32_t in_features, int32_t out_features);
int rd_linear_fwd(const float* x, const float* weight, const float* bias, int64_t rows, int32_t in_features,
                  int32_t out_features, int32_t relu, float* out, void* scratch, void* stream);

/* Temporal self-attention core of nn.TransformerEncoderLayer.self_attn (code/models_rd.py:232-237,358) for one
 * packed projection qkv [T, B, 3*H*hd] (seq-first, as F.multi_head_attention_forward lays it out):
 *   ctx[t, b, h*hd:(h+1)*hd] = dropout(softmax_j(q_t . k_j / sqrt(hd), keys j >= lengths[b] masked)) . v
 * and its backward d_qkv [T, B, 3*H*hd] from d_ctx [T, B, H*hd] (probabilities are recomputed, nothing T x T is
 * stored).  rng_captured = 2 x uint64 {seed, counter} on the device (ignored when drop_p == 0); `site` selects the
 * dropout stream (16 + layer inside the model).  impl: 0 = automatic, 1 = tcgen05 tensor-core kernels
 * (T <= 64, hd <= 96, hd % 4 == 0), 2 = CUDA-core kernels (T <= 64, hd <= 96).  Longer sequences are handled inside
 * rd_raindrop_v2_fwd/_bwd (they need workspace). */
int rd_temporal_attention_fwd(const float* qkv, const int64_t* lengths, int32_t B, int32_t H, int32_t T, int32_t hd,
                              float drop_p, const uint64_t* rng_captured, uint32_t site, int32_t impl, float* ctx,
                              void* stream);
int rd_temporal_attention_bwd(const float* qkv, const float* d_ctx, const int64_t* lengths, int32_t B, int32_t H,
                              int32_t T, int32_t hd, float drop_p, const uint64_t* rng_captured, uint32_t site,
                              int32_t impl, float* d_qkv, void* stream);

/* Weight/bias gradients of up to 12 torch.nn.Linear layers in ONE grouped tensor-core launch (+ one reduction
 * launch): d_weight[out_f, in_f] = d_out[rows, out_f]^T . x[rows, in_f], d_bias[out_f] = column sums of d_out.
 * This is what autograd computes for every Linear on the path (code/Raindrop.py:323); a training step has ten of
 * them (8 encoder weights + the two lin_value).  Error-compensated TF32 (fp32-level accuracy), deterministic.
 * `partial`: rd_linear_wgrad_partial_bytes(rows, out_f, in_f) bytes of scratch per problem, 16-byte aligned. */
typedef struct rd_wgrad_item {
  const float* d_out; const float* x; int64_t rows; int32_t out_features; int32_t in_features;
  float* d_weight; float* d_bias; void* partial;
} rd_wgrad_item;
size_t rd_linear_wgrad_partial_bytes(int64_t rows, int32_t out_features, int32_t in_features);
int rd_linear_wgrad_group(const rd_wgrad_item* items, int32_t n, void* stream);

/* TransformerConv.forward (code/transformer_conv.py:139-207), concat=True, root_weight=True, beta=False, no edge
 * features -- and its backward.  Batched over `n_graphs` independent graphs that share ONE edge list (legacy Raindrop v1
 * applies the layer to every sample of a batch, code/models_rd.py:158-166): the row of node i of graph g in x / out is
 * i * node_stride + g * graph_stride (single graph: n_graphs = 1, node_stride = 1, graph_stride = 0).
 *   x [rows, in];  weights [H*F, in];  edge_w [E] or NULL (then the logits are q_i.k_j / sqrt(F));
 *   out [rows, H*F];  alpha [n_graphs, E, H] (post-softmax, as returned by the reference).
 * Backward: writes d_x (may be NULL), d_w* / d_b* (written, not accumulated; with edge_w the q/k projections take no
 * part in the output, code/transformer_conv.py:199-200, so their gradients are zeros) and d_edge_w [E] (optional,
 * only with edge_w).  The weight / bias gradient pointers may be NULL: a NULL d_w* skips that projection's weight gradient
 * (its d_b* must then be NULL too); with all eight NULL (frozen layer) no weight-gradient launch is issued, and d_x /
 * d_edge_w are the same as with them.  scratch: rd_transformer_conv_scratch_bytes(..., backward) bytes. */
size_t rd_transformer_conv_scratch_bytes(int32_t n_nodes, int32_t n_graphs, int32_t in_ch, int32_t heads,
                                         int32_t out_ch, int32_t E, int32_t backward);
int rd_transformer_conv_fwd(const float* x, int32_t n_nodes, int32_t n_graphs, int64_t node_stride,
                            int64_t graph_stride, int32_t in_ch, int32_t heads, int32_t out_ch,
                            const int64_t* edge_src, const int64_t* edge_tgt, const float* edge_w, int32_t E,
                            const float* wq, const float* bq, const float* wk, const float* bk, const float* wv,
                            const float* bv, const float* ws, const float* bs, float* out, float* alpha,
                            void* scratch, void* stream);
int rd_transformer_conv_bwd(const float* x, int32_t n_nodes, int32_t n_graphs, int64_t node_stride,
                            int64_t graph_stride, int32_t in_ch, int32_t heads, int32_t out_ch,
                            const int64_t* edge_src, const int64_t* edge_tgt, const float* edge_w, int32_t E,
                            const float* wq, const float* bq, const float* wk, const float* bk, const float* wv,
                            const float* bv, const float* ws, const float* alpha, const float* d_out, float* d_x,
                            float* d_wq, float* d_bq, float* d_wk, float* d_bk, float* d_wv, float* d_bv,
                            float* d_ws, float* d_bs, float* d_edge_w, void* scratch, void* stream);

/* ---- device-side batch assembly (SURVEY.md 8f2) ---------------------------------------------------
 * out[t, j, :] = src[t, idx[j], :] for t < T, j < B: selects a batch out of a training set that stays
 * resident in HBM, replacing the host-side `Ptrain_tensor[:, idx, :].cuda()` copies of
 * code/Raindrop.py:311-315 (T = 1 for the [n, d_static] statics and labels viewed as float rows). */
int rd_gather_batch(const float* src, const int64_t* idx, int64_t T, int64_t n_total, int32_t width, int32_t B,
                    float* out, void* stream);

/* Whole-batch assembly in ONE launch: for j < B copies sample idx[j] of the resident tensors P [T, n_total, width],
 * Ptime [T, n_total], Pstatic [n_total, d_static] (may be NULL), y [n_total] (may be NULL) into the batch buffers and
 * writes lengths[j] = #(Ptime[:, idx[j]] > 0)  (code/Raindrop.py:311-317). */
int rd_assemble_batch(const float* P, const float* Ptime, const float* Pstatic, const int64_t* y, const int64_t* idx,
                      int32_t T, int64_t n_total, int32_t width, int32_t d_static, int32_t B, float* src, float* times,
                      float* statics, int64_t* y_out, int64_t* lengths, void* stream);

/* Per-feature statistics of the OBSERVED entries (value > 0) of raw [n, T, F]: mean and population standard deviation
 * (floored at 1e-7), accumulated in double -- getStats, code/utils_rd.py:149-161.
 * scratch: rd_feature_stats_scratch_bytes(n, T, F) bytes. */
size_t rd_feature_stats_scratch_bytes(int64_t n, int32_t T, int32_t F);
int rd_feature_stats(const float* raw, int64_t n, int32_t T, int32_t F, float* mean, float* std, void* scratch,
                     void* stream);
/* mask_normalize (code/utils_rd.py:164-175) fused with the concat of the observation mask and the permute to the
 * training layout (code/Raindrop.py:233): raw [n, T, F] -> out [T, n, 2F] with
 *   out[t, i, f] = raw > 0 ? (raw - mean_f) / (std_f + 1e-18) : 0      out[t, i, F + f] = raw > 0
 * minutes (optional) [n, T] -> times_out [T, n] = minutes / 60 (code/utils_rd.py:235). */
int rd_mask_normalize(const float* raw, const float* mean, const float* std, int64_t n, int32_t T, int32_t F,
                      float* out, const float* minutes, float* times_out, void* stream);
/* Leave-sensors-out masking of a batch P [T, B, width = 2F] (code/Raindrop.py:214-231): zero the VALUE columns
 * idx[k], k < K; per_sample != 0: idx is [B, K] (feature_removal_level 'sample'), else [K] ('set').  The mask columns
 * are left untouched, exactly as in the reference. */
int rd_zero_features(float* P, int64_t T, int32_t B, int32_t width, const int64_t* idx, int32_t K, int32_t per_sample,
                     void* stream);

/* ---- training-step helpers (the caller-side ops of code/Raindrop.py:321-324) ----------------
 * mean cross entropy + d(loss)/d(logits), torch.nn.CrossEntropyLoss semantics. */
int rd_cross_entropy_fwd_bwd(const float* logits, const int64_t* y, int32_t B, int32_t n_classes,
                             float* loss, float* d_logits, void* stream);
/* torch.optim.Adam (no weight decay, no amsgrad) on flat buffers, ONE launch.  `step` is int64[2] on the
 * device: step[0] = number of updates so far (incremented by the call, by the last CTA to finish),
 * step[1] = ticket word that must be 0 on entry (the call leaves it 0).  grad is multiplied by grad_scale
 * first (1/world_size after a sum all-reduce).  lr_dev: optional device scalar that overrides `lr`, so a
 * captured CUDA graph follows a scheduler (ReduceLROnPlateau, code/Raindrop.py:257-259) without re-capture. */
int rd_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                 float lr, const float* lr_dev, float beta1, float beta2, float eps, float grad_scale,
                 int64_t* step, void* stream);

/* debug: when `buffer` is non-NULL ([n_ctas][16] uint64 on the device), the tensor-core attention forward kernel writes
 * %globaltimer phase stamps into it (tools/attn_timing.py); NULL switches it off. */
int rd_debug_attention_timing(uint64_t* buffer);
/* same for the projection GEMM kernel behind rd_linear_fwd: [n_ctas][8] uint64 */
int rd_debug_gemm_timing(uint64_t* buffer);

/* debug: materialise the dropout keep/scale mask (0 or 1/(1-p)) of one dropout site, so tests can
 * replay train-mode forward/backward in the oracle with identical masks.  `site` ids in DESIGN.md. */
int rd_debug_dropout_mask(const uint64_t* rng_captured, uint32_t site, int64_t n, float p, float* out,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RAINDROP_B200_H */

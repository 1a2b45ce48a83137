// TransformerConv forward AND backward (code/transformer_conv.py:139-207), batched over independent graphs that
// share one edge list (legacy Raindrop v1 applies the layer to every sample of a batch, code/models_rd.py:158-166).
//
//   out[i] = sum_{e: tgt(e)=i} alpha[e,h] * v[src(e),h,:] + skip[i]        q,k,v,skip = Linear(x) per NODE
//   alpha  = segment softmax over the edges of one target of  edge_w[e]  (when given, code/transformer_conv.py:199-200)
//                                                          or q[tgt].k[src] / sqrt(F)
// The reference projects per EDGE (E/N times redundant); here the projections are node-level GEMMs, the edge
// softmax is one warp per (graph, target, head) and the aggregation a deterministic gather (ascending edge order, no
// atomics).  Graphs on this path are tiny (<= a few hundred nodes, ~10^3 edges), so every kernel simply scans the
// edge list.  Row of node i of graph g in x / out: i * node_stride + g * graph_stride.
#include <math.h>

#include "rd_kernels.cuh"

namespace rd {
namespace {

struct TcP {
  int n_nodes, n_graphs, H, F, E;
  long long node_stride, graph_stride;
  const int64_t* src; const int64_t* tgt;
};
__device__ __forceinline__ long long row_of(const TcP& p, long long node, int g) { return node * p.node_stride + (long long)g * p.graph_stride; }

// logit[g, e, h] = edge_w[e]  or  q[tgt].k[src] / sqrt(F)
__global__ void tconv_logits_kernel(TcP p, const float* __restrict__ q, const float* __restrict__ k,
                                    const float* __restrict__ edge_w, float* __restrict__ logit) {
  const int g = blockIdx.y;
  const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (w >= p.E * p.H) return;
  const int e = w / p.H, h = w - e * p.H;
  float* dst = logit + ((long long)g * p.E + e) * p.H + h;
  if (edge_w) { if (lane == 0) *dst = edge_w[e]; return; }
  const float* qi = q + (row_of(p, p.tgt[e], g) * p.H + h) * p.F;
  const float* kj = k + (row_of(p, p.src[e], g) * p.H + h) * p.F;
  float s = 0.f;
  for (int f = lane; f < p.F; f += 32) s += qi[f] * kj[f];
  s = warp_sum(s);
  if (lane == 0) *dst = s / sqrtf((float)p.F);
}

// alpha[g, e, h] = exp(logit - max) / (sum + 1e-16) over the edges of tgt(e)   (PyG utils.softmax)
__global__ void tconv_softmax_kernel(TcP p, const float* __restrict__ logit, float* __restrict__ alpha) {
  const int g = blockIdx.y;
  const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (w >= p.n_nodes * p.H) return;
  const int node = w / p.H, h = w - node * p.H;
  const float* lg = logit + (long long)g * p.E * p.H;
  float* al = alpha + (long long)g * p.E * p.H;
  float mx = -INFINITY;
  for (int e = lane; e < p.E; e += 32) if (p.tgt[e] == node) mx = fmaxf(mx, lg[e * p.H + h]);
  mx = warp_max(mx);
  if (mx == -INFINITY) return;
  float sum = 0.f;
  for (int e = lane; e < p.E; e += 32) if (p.tgt[e] == node) sum += expf(lg[e * p.H + h] - mx);
  sum = warp_sum(sum) + 1e-16f;
  for (int e = lane; e < p.E; e += 32) if (p.tgt[e] == node) al[e * p.H + h] = expf(lg[e * p.H + h] - mx) / sum;
}

// out[row(node)] += sum_{e -> node} alpha[e, h] v[row(src e)]        (out holds the skip term on entry)
__global__ void tconv_aggregate_kernel(TcP p, const float* __restrict__ v, const float* __restrict__ alpha, float* __restrict__ out) {
  const int node = blockIdx.x, g = blockIdx.y, HF = p.H * p.F;
  const float* al = alpha + (long long)g * p.E * p.H;
  for (int c = threadIdx.x; c < HF; c += blockDim.x) {
    const int h = c / p.F;
    float acc = 0.f;
    for (int e = 0; e < p.E; ++e)
      if (p.tgt[e] == node) acc += al[e * p.H + h] * v[row_of(p, p.src[e], g) * HF + c];
    out[row_of(p, node, g) * HF + c] += acc;
  }
}

// ---- backward ---------------------------------------------------------------------------------------
// d_alpha[e,h] = d_out[tgt].v[src];  d_logit = alpha * (d_alpha - sum_{e' -> tgt} alpha d_alpha)      one warp per (g, target, h)
__global__ void tconv_bwd_softmax_kernel(TcP p, const float* __restrict__ v, const float* __restrict__ alpha,
                                         const float* __restrict__ dout, float* __restrict__ dlogit) {
  const int g = blockIdx.y;
  const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (w >= p.n_nodes * p.H) return;
  const int node = w / p.H, h = w - node * p.H, HF = p.H * p.F;
  const float* al = alpha + (long long)g * p.E * p.H;
  float* dl = dlogit + (long long)g * p.E * p.H;
  const float* go = dout + row_of(p, node, g) * HF + h * p.F;
  float dot = 0.f;
  for (int e = 0; e < p.E; ++e) {
    if (p.tgt[e] != node) continue;                 // warp-uniform
    const float* vj = v + row_of(p, p.src[e], g) * HF + h * p.F;
    float s = 0.f;
    for (int f = lane; f < p.F; f += 32) s += go[f] * vj[f];
    s = warp_sum(s);
    if (lane == 0) dl[e * p.H + h] = s;             // d_alpha for now
    dot += al[e * p.H + h] * s;
  }
  __syncwarp();
  for (int e = lane; e < p.E; e += 32)
    if (p.tgt[e] == node) dl[e * p.H + h] = al[e * p.H + h] * (dl[e * p.H + h] - dot);
}

// per SOURCE node j: dv[j] = sum_{e: src=j} alpha[e,h] d_out[tgt e];  dk[j] = sum_{e: src=j} d_logit[e,h] q[tgt e] / sqrt(F)
__global__ void tconv_bwd_src_kernel(TcP p, const float* __restrict__ q, const float* __restrict__ alpha,
                                     const float* __restrict__ dlogit, const float* __restrict__ dout, float* __restrict__ dv,
                                     float* __restrict__ dk) {
  const int node = blockIdx.x, g = blockIdx.y, HF = p.H * p.F;
  const float* al = alpha + (long long)g * p.E * p.H;
  const float* dl = dlogit + (long long)g * p.E * p.H;
  const float rs = 1.f / sqrtf((float)p.F);
  for (int c = threadIdx.x; c < HF; c += blockDim.x) {
    const int h = c / p.F;
    float av = 0.f, ak = 0.f;
    for (int e = 0; e < p.E; ++e) {
      if (p.src[e] != node) continue;
      const long long tr = row_of(p, p.tgt[e], g) * HF + c;
      av += al[e * p.H + h] * dout[tr];
      if (dk) ak += dl[e * p.H + h] * q[tr];
    }
    dv[row_of(p, node, g) * HF + c] = av;
    if (dk) dk[row_of(p, node, g) * HF + c] = ak * rs;
  }
}

// per TARGET node i: dq[i] = sum_{e -> i} d_logit[e,h] k[src e] / sqrt(F)
__global__ void tconv_bwd_tgt_kernel(TcP p, const float* __restrict__ k, const float* __restrict__ dlogit, float* __restrict__ dq) {
  const int node = blockIdx.x, g = blockIdx.y, HF = p.H * p.F;
  const float* dl = dlogit + (long long)g * p.E * p.H;
  const float rs = 1.f / sqrtf((float)p.F);
  for (int c = threadIdx.x; c < HF; c += blockDim.x) {
    const int h = c / p.F;
    float a = 0.f;
    for (int e = 0; e < p.E; ++e)
      if (p.tgt[e] == node) a += dl[e * p.H + h] * k[row_of(p, p.src[e], g) * HF + c];
    dq[row_of(p, node, g) * HF + c] = a * rs;
  }
}

// d_edge_w[e] = sum over graphs and heads of d_logit[g, e, h]   (fixed order)
__global__ void tconv_bwd_edgew_kernel(TcP p, const float* __restrict__ dlogit, float* __restrict__ dw) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= p.E) return;
  float s = 0.f;
  for (int g = 0; g < p.n_graphs; ++g)
    for (int h = 0; h < p.H; ++h) s += dlogit[((long long)g * p.E + e) * p.H + h];
  dw[e] = s;
}

GemmP proj(const float* x, int in_ch, const float* W, const float* b, float* y, long long rows, int HF) {
  GemmP g;
  g.A = x; g.ta = 0; g.sAi = in_ch; g.sAk = 1;
  g.B = W; g.tb = 1; g.sBj = in_ch; g.sBk = 1;
  g.C = y; g.sCi = HF; g.sCj = 1;
  g.M = (int)rows; g.N = HF; g.K = in_ch; g.bias = b;
  return g;
}
// dx[rows, in] (+)= dy[rows, HF] . W[HF, in]
GemmP back(const float* dy, int HF, const float* W, int in_ch, float* dx, long long rows, bool accumulate) {
  GemmP g;
  g.A = dy; g.ta = 0; g.sAi = HF; g.sAk = 1;
  g.B = W; g.tb = 0; g.sBk = in_ch; g.sBj = 1;
  g.C = dx; g.sCi = in_ch; g.sCj = 1;
  g.M = (int)rows; g.N = in_ch; g.K = HF;
  if (accumulate) { g.resid = dx; g.resid_ld = in_ch; }
  return g;
}
// dW[HF, in] = dy^T x, db = column sums of dy (split over rows, deterministic)
int wgrad(const float* dy, int HF, const float* x, int in_ch, long long rows, float* dW, float* db, float* partial, cudaStream_t st) {
  GemmP g;
  g.A = dy; g.ta = 1; g.sAk = HF; g.sAi = 1;
  g.B = x; g.tb = 0; g.sBk = in_ch; g.sBj = 1;
  g.C = dW; g.sCi = in_ch; g.sCj = 1;
  g.M = HF; g.N = in_ch; g.K = (int)rows;
  int ns;
  gemm_splitk_plan(HF, in_ch, (int)rows, &ns);
  g.nsplit = ns; g.partial = partial; g.asum = db;
  return gemm(g, st);
}

struct Lay { long long rows, hf, q, k, v, logit, dq, dk, dv, partial, total; };
Lay layout(int n_nodes, int n_graphs, int in_ch, int H, int F, int E, bool bwd) {
  Lay l;
  l.rows = (long long)n_nodes * n_graphs; l.hf = (long long)H * F;
  long long o = 0;
  auto take = [&](long long n) { long long r = o; o += round_up(n > 0 ? n : 1, 64); return r; };
  l.q = take(l.rows * l.hf); l.k = take(l.rows * l.hf); l.v = take(l.rows * l.hf);
  l.logit = take((long long)n_graphs * E * H);
  l.dq = l.dk = l.dv = l.partial = 0;
  if (bwd) {
    l.dq = take(l.rows * l.hf); l.dk = take(l.rows * l.hf); l.dv = take(l.rows * l.hf);
    int ns;
    l.partial = take(gemm_splitk_plan((int)l.hf, in_ch, (int)l.rows, &ns));
  }
  l.total = o;
  return l;
}

int check_common(const char* who, const float* x, const int64_t* s, const int64_t* t, int n_nodes, int n_graphs, int in_ch, int H,
                 int F, int E, long long ns, long long gs) {
  if (!x || !s || !t || n_nodes < 1 || n_graphs < 1 || in_ch < 1 || H < 1 || F < 1 || E < 0 || ns < 1 || gs < 0 ||
      (long long)n_nodes * n_graphs > 0x7fffffffLL) {
    set_error("%s: bad arguments", who);
    return -2;
  }
  return 0;
}

}  // namespace
}  // namespace rd

using namespace rd;

extern "C" size_t rd_transformer_conv_scratch_bytes(int32_t n_nodes, int32_t n_graphs, int32_t in_ch, int32_t heads,
                                                    int32_t out_ch, int32_t E, int32_t backward) {
  if (n_nodes < 1 || n_graphs < 1 || heads < 1 || out_ch < 1 || E < 0 || in_ch < 1) return 0;
  return (size_t)layout(n_nodes, n_graphs, in_ch, heads, out_ch, E, backward != 0).total * sizeof(float);
}

extern "C" int rd_transformer_conv_fwd(const float* x, int32_t n_nodes, int32_t n_graphs, int64_t node_stride,
                                       int64_t graph_stride, int32_t in_ch, int32_t heads, int32_t out_ch,
                                       const int64_t* edge_src, const int64_t* edge_tgt, const float* edge_w, int32_t E,
                                       const float* wq, const float* bq, const float* wk, const float* bk, const float* wv,
                                       const float* bv, const float* ws, const float* bs, float* out, float* alpha,
                                       void* scratch, void* stream) {
  RD_TRY(check_common("rd_transformer_conv_fwd", x, edge_src, edge_tgt, n_nodes, n_graphs, in_ch, heads, out_ch, E, node_stride,
                      graph_stride));
  if (!wq || !wk || !wv || !ws || !out || !alpha || !scratch) { set_error("rd_transformer_conv_fwd: NULL argument"); return -2; }
  cudaStream_t st = (cudaStream_t)stream;
  const Lay l = layout(n_nodes, n_graphs, in_ch, heads, out_ch, E, false);
  const int HF = heads * out_ch;
  float* q = (float*)scratch + l.q; float* k = (float*)scratch + l.k; float* v = (float*)scratch + l.v;
  float* logit = (float*)scratch + l.logit;
  if (!edge_w) {    // the q.k logits are only needed when no edge weights replace them
    RD_TRY(gemm(proj(x, in_ch, wq, bq, q, l.rows, HF), st));
    RD_TRY(gemm(proj(x, in_ch, wk, bk, k, l.rows, HF), st));
  }
  RD_TRY(gemm(proj(x, in_ch, wv, bv, v, l.rows, HF), st));
  RD_TRY(gemm(proj(x, in_ch, ws, bs, out, l.rows, HF), st));   // root/skip term, code/transformer_conv.py:168-175
  if (E == 0) return 0;
  TcP p{n_nodes, n_graphs, heads, out_ch, E, node_stride, graph_stride, edge_src, edge_tgt};
  tconv_logits_kernel<<<dim3((unsigned)ceil_div((int64_t)E * heads * 32, 256), n_graphs), 256, 0, st>>>(p, q, k, edge_w, logit);
  RD_CHECK_LAUNCH("tconv_logits_kernel");
  if (cudaMemsetAsync(alpha, 0, sizeof(float) * (size_t)n_graphs * E * heads, st) != cudaSuccess) { set_error("rd_transformer_conv_fwd: memset failed"); return -1; }
  tconv_softmax_kernel<<<dim3((unsigned)ceil_div((int64_t)n_nodes * heads * 32, 256), n_graphs), 256, 0, st>>>(p, logit, alpha);
  RD_CHECK_LAUNCH("tconv_softmax_kernel");
  tconv_aggregate_kernel<<<dim3(n_nodes, n_graphs), 128, 0, st>>>(p, v, alpha, out);
  RD_CHECK_LAUNCH("tconv_aggregate_kernel");
  return 0;
}

// d_x (may be NULL), d_w*/d_b* [HF, in] / [HF] (written, not accumulated), d_edge_w [E] (only with edge_w, may be NULL).
// With edge_w given, lin_query / lin_key take no part in the output (code/transformer_conv.py:199-200): their
// gradients are written as zeros.  A NULL d_w* skips that projection's weight gradient (its d_b* must be NULL too); with
// all eight NULL (frozen layer) no weight-gradient launch is issued and d_x / d_edge_w are computed as before.
extern "C" int rd_transformer_conv_bwd(const float* x, int32_t n_nodes, int32_t n_graphs, int64_t node_stride,
                                       int64_t graph_stride, int32_t in_ch, int32_t heads, int32_t out_ch,
                                       const int64_t* edge_src, const int64_t* edge_tgt, const float* edge_w, int32_t E,
                                       const float* wq, const float* bq, const float* wk, const float* bk, const float* wv,
                                       const float* bv, const float* ws, const float* alpha, const float* d_out, float* d_x,
                                       float* d_wq, float* d_bq, float* d_wk, float* d_bk, float* d_wv, float* d_bv,
                                       float* d_ws, float* d_bs, float* d_edge_w, void* scratch, void* stream) {
  RD_TRY(check_common("rd_transformer_conv_bwd", x, edge_src, edge_tgt, n_nodes, n_graphs, in_ch, heads, out_ch, E, node_stride,
                      graph_stride));
  if (!wq || !wk || !wv || !ws || !alpha || !d_out || !scratch) {
    set_error("rd_transformer_conv_bwd: NULL argument");
    return -2;
  }
  if ((!d_wq && d_bq) || (!d_wk && d_bk) || (!d_wv && d_bv) || (!d_ws && d_bs)) {
    set_error("rd_transformer_conv_bwd: a bias gradient needs its weight gradient");
    return -2;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const Lay l = layout(n_nodes, n_graphs, in_ch, heads, out_ch, E, true);
  const int HF = heads * out_ch;
  float* sc = (float*)scratch;
  float* q = sc + l.q; float* k = sc + l.k; float* v = sc + l.v; float* dlogit = sc + l.logit;
  float* dq = sc + l.dq; float* dk = sc + l.dk; float* dv = sc + l.dv; float* partial = sc + l.partial;
  const bool qk = edge_w == nullptr;
  // recompute the node projections the edge stage needs
  if (qk) {
    RD_TRY(gemm(proj(x, in_ch, wq, bq, q, l.rows, HF), st));
    RD_TRY(gemm(proj(x, in_ch, wk, bk, k, l.rows, HF), st));
  }
  RD_TRY(gemm(proj(x, in_ch, wv, bv, v, l.rows, HF), st));
  // skip term: out = ... + x Ws^T + bs
  if (d_ws) RD_TRY(wgrad(d_out, HF, x, in_ch, l.rows, d_ws, d_bs, partial, st));
  if (d_x) RD_TRY(gemm(back(d_out, HF, ws, in_ch, d_x, l.rows, false), st));
  const size_t wbytes = sizeof(float) * (size_t)HF * in_ch, bbytes = sizeof(float) * (size_t)HF;
  auto zero = [&](float* p, size_t n) { if (p) cudaMemsetAsync(p, 0, n, st); };
  if (E == 0) {
    zero(d_wq, wbytes); zero(d_wk, wbytes); zero(d_wv, wbytes);
    zero(d_bq, bbytes); zero(d_bk, bbytes); zero(d_bv, bbytes);
    return 0;
  }
  TcP p{n_nodes, n_graphs, heads, out_ch, E, node_stride, graph_stride, edge_src, edge_tgt};
  if (cudaMemsetAsync(dlogit, 0, sizeof(float) * (size_t)n_graphs * E * heads, st) != cudaSuccess) { set_error("rd_transformer_conv_bwd: memset failed"); return -1; }
  tconv_bwd_softmax_kernel<<<dim3((unsigned)ceil_div((int64_t)n_nodes * heads * 32, 256), n_graphs), 256, 0, st>>>(p, v, alpha, d_out, dlogit);
  RD_CHECK_LAUNCH("tconv_bwd_softmax_kernel");
  tconv_bwd_src_kernel<<<dim3(n_nodes, n_graphs), 128, 0, st>>>(p, q, alpha, dlogit, d_out, dv, qk ? dk : nullptr);
  RD_CHECK_LAUNCH("tconv_bwd_src_kernel");
  if (d_wv) RD_TRY(wgrad(dv, HF, x, in_ch, l.rows, d_wv, d_bv, partial, st));
  if (d_x) RD_TRY(gemm(back(dv, HF, wv, in_ch, d_x, l.rows, true), st));
  if (qk) {
    tconv_bwd_tgt_kernel<<<dim3(n_nodes, n_graphs), 128, 0, st>>>(p, k, dlogit, dq);
    RD_CHECK_LAUNCH("tconv_bwd_tgt_kernel");
    if (d_wq) RD_TRY(wgrad(dq, HF, x, in_ch, l.rows, d_wq, d_bq, partial, st));
    if (d_wk) RD_TRY(wgrad(dk, HF, x, in_ch, l.rows, d_wk, d_bk, partial, st));
    if (d_x) {
      RD_TRY(gemm(back(dq, HF, wq, in_ch, d_x, l.rows, true), st));
      RD_TRY(gemm(back(dk, HF, wk, in_ch, d_x, l.rows, true), st));
    }
  } else {
    zero(d_wq, wbytes); zero(d_wk, wbytes);
    zero(d_bq, bbytes); zero(d_bk, bbytes);
    if (d_edge_w) {
      tconv_bwd_edgew_kernel<<<(unsigned)ceil_div(E, 256), 256, 0, st>>>(p, dlogit, d_edge_w);
      RD_CHECK_LAUNCH("tconv_bwd_edgew_kernel");
    }
  }
  return 0;
}

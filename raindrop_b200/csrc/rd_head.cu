// Pooling + classification head of Raindrop_v2 (code/models_rd.py:366-385) as three launches:
//   forward   (one CTA per sample): pooled = masked mean over time (divisor lengths+1, :379),
//             feat = [pooled || emb(static)], h = relu(mlp_static.0(feat)), logits = mlp_static.2(h),
//             and -- when labels are given -- CrossEntropyLoss forward/backward (code/Raindrop.py:322);
//   backward A (one CTA per sample): dh, dfeat, and the masked-mean backward written straight into the
//             encoder-output gradient [T, B, D];
//   backward B (one launch): the three weight gradients (mlp_static.0, mlp_static.2, emb) as tiled
//             outer-product sums over the batch, fixed summation order (deterministic).
// At the reference's batch sizes these are 128 x 186 problems: pure launch latency, hence the fusion.
#include "rd_kernels.cuh"

namespace rd {
namespace {

constexpr int HT = 512;

struct HeadP {
  int B, T, D, N, ds, Df, ncls;
  const float* statics; const float* emb_w; const float* emb_b;
  const float* w0; const float* b0; const float* w2; const float* b2;
  const int64_t* lengths;
};

// grid = B, block = HT.  x = encoder output [T, B, D].
__global__ void __launch_bounds__(HT) head_fwd_kernel(HeadP p, const float* __restrict__ x, float* __restrict__ feat,
                                                      float* __restrict__ hpre, float* __restrict__ logits,
                                                      const int64_t* __restrict__ y, float* __restrict__ loss_ps,
                                                      float* __restrict__ dlogits, float* __restrict__ loss,
                                                      unsigned* __restrict__ counter) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float sm[];
  float* fs = sm; float* hs = fs + p.Df; float* red = sm + ((2 * p.Df + 3) & ~3);     // red (16-byte aligned): [8][D] pooling partials, later logits
  __shared__ int s_last;
  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float* fb = feat + (long long)b * p.Df;
  // ---- masked mean over time: 8 time groups x 64 column quads, fixed-order combine ---------------
  {
    const long long len = p.lengths[b];
    const int nv = (int)(len < p.T ? (len < 0 ? 0 : len) : p.T);
    const int tg = tid >> 6, dq0 = tid & 63, nq = p.D >> 2;
    for (int dq = dq0; dq < nq; dq += 64) {
      float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8
      for (int t = tg; t < nv; t += 8) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(x + ((long long)t * p.B + b) * p.D) + dq);
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      }
      *reinterpret_cast<float4*>(red + tg * p.D + 4 * dq) = s;
    }
    __syncthreads();
    const float inv = 1.f / (float)(len + 1);
    for (int k = tid; k < p.D; k += HT) {
      float s = 0.f;
#pragma unroll
      for (int g = 0; g < 8; ++g) s += red[g * p.D + k];
      s *= inv;
      fs[k] = s;
      fb[k] = s;
    }
  }
  if (p.ds > 0) {   // emb = Linear(d_static, N)(static)                      code/models_rd.py:293-294
    for (int n = tid; n < p.N; n += HT) {
      float a = __ldg(p.emb_b + n);
      for (int k = 0; k < p.ds; ++k) a = fmaf(__ldg(p.statics + (long long)b * p.ds + k), __ldg(p.emb_w + n * p.ds + k), a);
      fs[p.D + n] = a;
      fb[p.D + n] = a;
    }
  }
  __syncthreads();
  // a warp owns HU hidden units at a time; all weight loads of a 256-wide k pass are issued before the FMAs
  // (HU = 6: the 186 units of the P19 head take two L2 round trips per warp instead of three)
  constexpr int HU = 6;
  for (int j0 = warp * HU; j0 < p.Df; j0 += (HT / 32) * HU) {
    float a[HU];
#pragma unroll
    for (int u = 0; u < HU; ++u) a[u] = 0.f;
    for (int kb = 0; kb < p.Df; kb += 256) {
      float w[HU][8], f[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int k = kb + lane + 32 * e;
        const bool ok = k < p.Df;
        f[e] = ok ? fs[k] : 0.f;
#pragma unroll
        for (int u = 0; u < HU; ++u) w[u][e] = (ok && j0 + u < p.Df) ? __ldg(p.w0 + (long long)(j0 + u) * p.Df + k) : 0.f;
      }
#pragma unroll
      for (int e = 0; e < 8; ++e)
#pragma unroll
        for (int u = 0; u < HU; ++u) a[u] = fmaf(f[e], w[u][e], a[u]);
    }
#pragma unroll
    for (int u = 0; u < HU; ++u) {
      const float v = warp_sum(a[u]);
      if (lane == 0 && j0 + u < p.Df) {
        const float h = fmaxf(v + __ldg(p.b0 + j0 + u), 0.f);
        hs[j0 + u] = h;
        hpre[(long long)b * p.Df + j0 + u] = h;
      }
    }
  }
  __syncthreads();
  float* lg = red;      // this sample's logits
  for (int c = warp; c < p.ncls; c += HT / 32) {
    const float* wr = p.w2 + (long long)c * p.Df;
    float a = 0.f;
    for (int jb = 0; jb < p.Df; jb += 256) {       // all weight loads of a 256-wide pass in flight before the FMAs
      float w[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) { const int j = jb + lane + 32 * e; w[e] = j < p.Df ? __ldg(wr + j) : 0.f; }
#pragma unroll
      for (int e = 0; e < 8; ++e) { const int j = jb + lane + 32 * e; if (j < p.Df) a = fmaf(hs[j], w[e], a); }
    }
    a = warp_sum(a);
    if (lane == 0) { a += __ldg(p.b2 + c); logits[(long long)b * p.ncls + c] = a; lg[c] = a; }
  }
  if (!y) return;
  // ---- CrossEntropyLoss (mean over the batch) forward + d(loss)/d(logits) ------------------------
  __syncthreads();
  if (warp == 0) {
    float mx = -INFINITY;
    for (int c = lane; c < p.ncls; c += 32) mx = fmaxf(mx, lg[c]);
    mx = warp_max(mx);
    float sum = 0.f;
    for (int c = lane; c < p.ncls; c += 32) sum += expf(lg[c] - mx);
    sum = warp_sum(sum);
    const float lse = mx + logf(sum);
    const int yy = (int)y[b];
    const float invB = 1.f / (float)p.B;
    for (int c = lane; c < p.ncls; c += 32)
      dlogits[(long long)b * p.ncls + c] = (expf(lg[c] - lse) - (c == yy ? 1.f : 0.f)) * invB;
    if (lane == 0) {
      loss_ps[b] = lse - lg[yy];
      __threadfence();
      s_last = (atomicAdd(counter, 1u) == (unsigned)(p.B - 1));
    }
    __syncwarp();
    if (s_last) {      // the last sample to finish sums the per-sample losses in a fixed order
      __threadfence();
      float s = 0.f;
      for (int i = lane; i < p.B; i += 32) s += __ldcg(loss_ps + i);
      s = warp_sum(s);
      if (lane == 0) { *loss = s * invB; *counter = 0u; }
    }
  }
}

// grid = B: dh = (dlogits . W2) * [h > 0];  dfeat = dh . W0;  d(encoder output)[t, b, :] = dfeat[:D] / (len+1) for t < len
__global__ void __launch_bounds__(HT) head_bwd_sample_kernel(HeadP p, const float* __restrict__ hpre,
                                                             const float* __restrict__ dlogits, float* __restrict__ dh,
                                                             float* __restrict__ dfeat, float* __restrict__ dx) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float sm[];
  float* ds_ = sm;                 // dh of this sample [Df]
  float* part = sm + p.Df;         // [groups][Df] partial dfeat
  float* df = part;                // final dfeat (group 0's row after the combine)
  const int b = blockIdx.x, tid = threadIdx.x;
  for (int j = tid; j < p.Df; j += HT) {
    float a = 0.f;
    for (int c = 0; c < p.ncls; ++c) a = fmaf(__ldg(dlogits + (long long)b * p.ncls + c), __ldg(p.w2 + (long long)c * p.Df + j), a);
    a = hpre[(long long)b * p.Df + j] > 0.f ? a : 0.f;
    ds_[j] = a;
    dh[(long long)b * p.Df + j] = a;
  }
  __syncthreads();
  // dfeat[k] = sum_j dh[j] W0[j, k]: a warp owns rows j = warp, warp + 16, ...; its lanes sweep k in chunks of 256 with the
  // loads of 4 rows x 8 columns in flight together; the 16 per-warp partial rows are then summed in a fixed order
  const int warp = tid >> 5, lane = tid & 31, nwarp = HT / 32;
  for (int kb = 0; kb < p.Df; kb += 256) {
    float acc[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = 0.f;
    for (int j0 = warp; j0 < p.Df; j0 += 4 * nwarp) {
      float w[4][8];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = j0 + u * nwarp;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int k = kb + lane + 32 * e;
          w[u][e] = (j < p.Df && k < p.Df) ? __ldg(p.w0 + (long long)j * p.Df + k) : 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = j0 + u * nwarp;
        const float d = j < p.Df ? ds_[j] : 0.f;
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] = fmaf(d, w[u][e], acc[e]);
      }
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = kb + lane + 32 * e;
      if (k < p.Df) part[warp * p.Df + k] = acc[e];
    }
  }
  __syncthreads();
  for (int k = tid; k < p.Df; k += HT) {
    float a = part[k];
    for (int g = 1; g < nwarp; ++g) a += part[g * p.Df + k];
    dfeat[(long long)b * p.Df + k] = a;
    df[k] = a;          // only thread `k` touched part[.][k] above: no hazard
  }
  __syncthreads();
  // masked-mean backward (code/models_rd.py:366-379)
  const long long len = p.lengths[b];
  const float inv = 1.f / (float)(len + 1);
  const int nq = p.D >> 2;
  for (int i = tid; i < p.T * nq; i += HT) {
    const int t = i / nq, dq = i - t * nq;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t < len) v = make_float4(df[4 * dq] * inv, df[4 * dq + 1] * inv, df[4 * dq + 2] * inv, df[4 * dq + 3] * inv);
    *(reinterpret_cast<float4*>(dx + ((long long)t * p.B + b) * p.D) + dq) = v;
  }
}

// out[j, k] = sum_b L[b, j] * R[b, k]  (j < J, k < K), bias[j] = sum_b L[b, j]: 32 x 32 output tile per CTA,
// the batch is staged through shared memory 32 samples at a time (all loads of a chunk in flight together)
struct OuterItem { const float* L; long long ldl; const float* R; long long ldr; int J, K, kt, blk0; float* out; float* bias; };
struct OuterGroup { OuterItem it[3]; int n, B; };
__global__ void __launch_bounds__(256) head_outer_kernel(const __grid_constant__ OuterGroup g) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float Ls[32][33], Rs[32][33];
  int ii = 0;
  for (int k = 1; k < g.n; ++k) if ((int)blockIdx.x >= g.it[k].blk0) ii = k;
  const OuterItem& o = g.it[ii];
  const int blk = (int)blockIdx.x - o.blk0;
  const int kt = blk % o.kt, jt = blk / o.kt;
  const int j0 = jt * 32, k0 = kt * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  float a[4] = {0.f, 0.f, 0.f, 0.f};
  float bsum = 0.f;
  for (int b0 = 0; b0 < g.B; b0 += 32) {
    float lv[4], rv[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int bb = ty + 8 * i, b = b0 + bb;
      lv[i] = (b < g.B && j0 + tx < o.J) ? __ldg(o.L + (long long)b * o.ldl + j0 + tx) : 0.f;
      rv[i] = (b < g.B && k0 + tx < o.K) ? __ldg(o.R + (long long)b * o.ldr + k0 + tx) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) { Ls[ty + 8 * i][tx] = lv[i]; Rs[ty + 8 * i][tx] = rv[i]; }
    __syncthreads();
#pragma unroll 8
    for (int bb = 0; bb < 32; ++bb) {
      const float r = Rs[bb][tx];
#pragma unroll
      for (int u = 0; u < 4; ++u) a[u] = fmaf(Ls[bb][ty * 4 + u], r, a[u]);
    }
    if (kt == 0 && ty == 0) {
#pragma unroll 8
      for (int bb = 0; bb < 32; ++bb) bsum += Ls[bb][tx];
    }
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int j = j0 + ty * 4 + u, k = k0 + tx;
    if (j < o.J && k < o.K) o.out[(long long)j * o.K + k] = a[u];
  }
  if (o.bias && kt == 0 && ty == 0 && j0 + tx < o.J) o.bias[j0 + tx] = bsum;
}

HeadP make(int B, int T, int D, int N, int ds, int ncls, const float* statics, const float* emb_w, const float* emb_b,
           const float* w0, const float* b0, const float* w2, const float* b2, const int64_t* lengths) {
  HeadP p;
  p.B = B; p.T = T; p.D = D; p.N = N; p.ds = ds; p.Df = D + (ds > 0 ? N : 0); p.ncls = ncls;
  p.statics = statics; p.emb_w = emb_w; p.emb_b = emb_b; p.w0 = w0; p.b0 = b0; p.w2 = w2; p.b2 = b2; p.lengths = lengths;
  return p;
}

}  // namespace

int head_fwd(int B, int T, int D, int N, int ds, int ncls, const float* x, const int64_t* lengths, const float* statics,
             const float* emb_w, const float* emb_b, const float* w0, const float* b0, const float* w2, const float* b2,
             float* feat, float* hpre, float* logits, const int64_t* y, float* loss_ps, float* dlogits, float* loss,
             unsigned* counter, cudaStream_t st) {
  HeadP p = make(B, T, D, N, ds, ncls, statics, emb_w, emb_b, w0, b0, w2, b2, lengths);
  const int red = 8 * D > ncls ? 8 * D : ncls;
  const size_t smem = (size_t)(((2 * p.Df + 3) & ~3) + red) * sizeof(float);
  if (smem > 48 * 1024 || (D & 3)) { set_error("head_fwd: feature width %d not supported", p.Df); return -2; }
  if (y && (!loss_ps || !dlogits || !loss || !counter)) { set_error("head_fwd: labels given without loss outputs"); return -2; }
  launch_pdl(head_fwd_kernel, dim3(B), dim3(HT), smem, st, p, x, feat, hpre, logits, y, loss_ps, dlogits, loss, counter);
  RD_CHECK_LAUNCH("head_fwd_kernel");
  return 0;
}

int head_bwd(int B, int T, int D, int N, int ds, int ncls, const int64_t* lengths, const float* statics, const float* w0,
             const float* w2, const float* feat, const float* hpre, const float* dlogits, float* dh, float* dfeat, float* dx,
             float* g_w0, float* g_b0, float* g_w2, float* g_b2, float* g_emb_w, float* g_emb_b, cudaStream_t st) {
  HeadP p = make(B, T, D, N, ds, ncls, statics, nullptr, nullptr, w0, nullptr, w2, nullptr, lengths);
  const size_t smem = (size_t)(1 + HT / 32) * p.Df * sizeof(float);       // dh + one partial dfeat row per warp
  if (smem > 48 * 1024) { set_error("head_bwd: feature width %d too large", p.Df); return -2; }
  launch_pdl(head_bwd_sample_kernel, dim3(B), dim3(HT), smem, st, p, hpre, dlogits, dh, dfeat, dx);
  RD_CHECK_LAUNCH("head_bwd_sample_kernel");
  if (!g_w0) return 0;      // input gradients only: dfeat and dx are all the caller needs
  OuterGroup g;
  g.B = B; g.n = 0;
  int blk = 0;
  auto add = [&](const float* L, long long ldl, const float* R, long long ldr, int J, int K, float* out, float* bias) {
    OuterItem& o = g.it[g.n++];
    o.L = L; o.ldl = ldl; o.R = R; o.ldr = ldr; o.J = J; o.K = K; o.kt = (int)ceil_div(K, 32); o.blk0 = blk; o.out = out; o.bias = bias;
    blk += o.kt * (int)ceil_div(J, 32);
  };
  add(dh, p.Df, feat, p.Df, p.Df, p.Df, g_w0, g_b0);                   // d mlp_static.0
  add(dlogits, ncls, hpre, p.Df, ncls, p.Df, g_w2, g_b2);              // d mlp_static.2
  if (ds > 0) add(dfeat + D, p.Df, statics, ds, N, ds, g_emb_w, g_emb_b);   // d emb
  launch_pdl(head_outer_kernel, dim3(blk), dim3(256), 0, st, g);
  RD_CHECK_LAUNCH("head_outer_kernel");
  return 0;
}

}  // namespace rd

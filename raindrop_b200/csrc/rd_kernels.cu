// Non-GEMM kernels of the Raindrop hot path: input lift, positional encoding, graph prologue,
// LayerNorm, masked attention softmax, masked mean, loss and optimiser.  All are HBM-bound
// streaming kernels: coalesced along the fastest tensor dimension, one warp per row for the
// row-wise reductions (warp-shuffle, no shared memory), grid sized from the element count.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include "rd_kernels.cuh"

namespace rd {

// ---- error plumbing ---------------------------------------------------------------------------
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* last_error() { return g_err; }
static unsigned long long g_launches = 0;
unsigned long long launch_count() { return g_launches; }
bool pdl_enabled() {
  static int v = -1;
  // programmatic dependent launch: a kernel's prologue (barrier init, TMEM allocation, descriptor prefetch) overlaps the tail
  // of its predecessor; every kernel waits (griddepcontrol.wait) before it touches global memory.  0.539 -> 0.518 ms per
  // P19 step inside the graph (it measured at no gain before the kernels were shortened).  RD_PDL=0 turns it off.
  if (v < 0) { const char* e = getenv("RD_PDL"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}
int check_launch(const char* what) {
  ++g_launches;
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    cudaGetLastError();
    return -1;
  }
  return 0;
}

namespace {

constexpr int TPB = 256;
inline unsigned blocks_for(int64_t n, int tpb = TPB) { return (unsigned)ceil_div(n, tpb); }

__device__ __forceinline__ float to_tf32(float v) {   // round-to-nearest TF32 (10-bit mantissa)
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}

// y[j*rows + i] = RN_tf32(x[i*cols + j]): transposed, rounded copy of a weight matrix
__global__ void transpose_round_kernel(const float* __restrict__ x, int rows, int cols, float* __restrict__ y) {
  __shared__ float tile[32][33];
  int bx = blockIdx.x * 32, by = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    int i = by + r, j = bx + threadIdx.x;
    tile[r][threadIdx.x] = (i < rows && j < cols) ? x[(long long)i * cols + j] : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    int j = bx + r, i = by + threadIdx.x;
    if (i < rows && j < cols) y[(long long)j * rows + i] = to_tf32(tile[threadIdx.x][r]);
  }
}

// out[t, j, :] = src[t, idx[j], :]  (rows of `width` floats; 128-bit copies when width % 4 == 0)
__global__ void gather_batch_kernel(const float* __restrict__ src, const int64_t* __restrict__ idx, long long T,
                                    long long n_total, int width, int B, float* __restrict__ out) {
  const int vec = (width & 3) == 0 ? 4 : 1;
  const long long per_row = width / vec;
  long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= T * B * per_row) return;
  const long long c = o % per_row, tj = o / per_row, j = tj % B, t = tj / B;
  const long long s = idx[j];
  if (s < 0 || s >= n_total) return;                      // out-of-range indices leave the row untouched
  const float* in = src + (t * n_total + s) * width;
  float* dst = out + (t * B + j) * width;
  if (vec == 4) reinterpret_cast<float4*>(dst)[c] = __ldg(reinterpret_cast<const float4*>(in) + c);
  else dst[c] = __ldg(in + c);
}

// ---- device-side input pipeline (code/utils_rd.py:149-175,221-257, code/Raindrop.py:214-231,293-317) -------------
// per-feature {count, sum, sum of squares} over the OBSERVED entries (value > 0) of raw[n, T, F], in double;
// grid (chunks, F): each CTA walks a slice of the n*T entries of one feature, fixed-order tree reduce
constexpr int FS_THREADS = 256;
__global__ void __launch_bounds__(FS_THREADS) feature_stats_partial_kernel(const float* __restrict__ raw, long long nT, int F,
                                                                          double* __restrict__ partial) {
  __shared__ double sh[3][FS_THREADS];
  const int f = blockIdx.y;
  const long long per = (nT + gridDim.x - 1) / gridDim.x;
  const long long i0 = (long long)blockIdx.x * per, i1 = min(nT, i0 + per);
  double c = 0.0, s = 0.0, q = 0.0;
  for (long long i = i0 + threadIdx.x; i < i1; i += FS_THREADS) {
    const float v = __ldg(raw + i * F + f);
    if (v > 0.f) { c += 1.0; s += (double)v; q += (double)v * (double)v; }
  }
  sh[0][threadIdx.x] = c; sh[1][threadIdx.x] = s; sh[2][threadIdx.x] = q;
  __syncthreads();
  for (int o = FS_THREADS / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      sh[0][threadIdx.x] += sh[0][threadIdx.x + o]; sh[1][threadIdx.x] += sh[1][threadIdx.x + o]; sh[2][threadIdx.x] += sh[2][threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    double* o = partial + ((long long)f * gridDim.x + blockIdx.x) * 3;
    o[0] = sh[0][0]; o[1] = sh[1][0]; o[2] = sh[2][0];
  }
}
// mean / population std (np.mean, np.std of getStats, code/utils_rd.py:149-161), std floored at 1e-7
__global__ void feature_stats_final_kernel(const double* __restrict__ partial, int chunks, int F, float* __restrict__ mean,
                                           float* __restrict__ stdv) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= F) return;
  double c = 0.0, s = 0.0, q = 0.0;
  for (int k = 0; k < chunks; ++k) { const double* p = partial + ((long long)f * chunks + k) * 3; c += p[0]; s += p[1]; q += p[2]; }
  const double m = c > 0.0 ? s / c : 0.0;            // np.mean of an empty selection is nan in the reference; 0 keeps the pipeline finite
  double var = c > 0.0 ? q / c - m * m : 0.0;
  if (var < 0.0) var = 0.0;
  double sd = sqrt(var);
  if (sd < 1e-7) sd = 1e-7;
  mean[f] = (float)m;
  stdv[f] = (float)sd;
}
// out[t, i, f] = raw[i, t, f] > 0 ? (raw - mean_f) / (std_f + 1e-18) : 0;  out[t, i, F + f] = raw[i, t, f] > 0
// (mask_normalize + the permute(1, 0, 2) of code/Raindrop.py:233); times_out[t, i] = minutes[i, t] / 60
__global__ void mask_normalize_kernel(const float* __restrict__ raw, const float* __restrict__ mean, const float* __restrict__ stdv,
                                      long long n, int T, int F, float* __restrict__ out, const float* __restrict__ minutes,
                                      float* __restrict__ times_out) {
  const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = n * T * F;
  if (o < total) {
    const int f = (int)(o % F);
    const long long it = o / F;
    const int t = (int)(it % T);
    const long long i = it / T;
    const float v = __ldg(raw + o);
    const bool obs = v > 0.f;
    // the reference divides in float64 and casts once: do the same so the values agree to the last fp32 bit or two
    const double z = ((double)v - (double)__ldg(mean + f)) / ((double)__ldg(stdv + f) + 1e-18);
    float* dst = out + ((long long)t * n + i) * (2 * F);
    dst[f] = obs ? (float)z : 0.f;
    dst[F + f] = obs ? 1.f : 0.f;
  }
  if (minutes && o < n * T) {
    const int t = (int)(o % T);
    const long long i = o / T;
    times_out[(long long)t * n + i] = __ldg(minutes + o) / 60.0f;
  }
}
// zero the VALUE columns idx[k] (k < K) of P[t, j, :] (width = 2F; mask columns untouched): the leave-sensors-out
// settings of code/Raindrop.py:214-231.  per_sample != 0: idx is [B, K] (setting 'sample'), else [K] ('set')
__global__ void zero_features_kernel(float* __restrict__ P, long long T, int B, int width, const int64_t* __restrict__ idx,
                                     int K, int per_sample) {
  const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= T * B * K) return;
  const int k = (int)(o % K);
  const long long tj = o / K;
  const int j = (int)(tj % B);
  const long long f = idx[per_sample ? (long long)j * K + k : k];
  if (f >= 0 && f < width / 2) P[tj * width + f] = 0.f;
}
// One launch assembles a training batch out of device-resident tensors (code/Raindrop.py:311-317 does this on the
// host and copies 2 MB over PCIe): CTA j copies sample idx[j]'s [T, width] rows, its times, statics and label and
// counts lengths[j] = #(times > 0).
__global__ void __launch_bounds__(256) assemble_batch_kernel(const float* __restrict__ P, const float* __restrict__ Pt,
                                                            const float* __restrict__ Ps, const int64_t* __restrict__ y,
                                                            const int64_t* __restrict__ idx, int T, long long n_total, int width,
                                                            int ds, int B, float* __restrict__ src, float* __restrict__ times,
                                                            float* __restrict__ statics, int64_t* __restrict__ y_out,
                                                            int64_t* __restrict__ lengths) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ int cnt[8];
  const int j = blockIdx.x;
  const long long sidx = idx[j];
  if (sidx < 0 || sidx >= n_total) return;
  if ((width & 3) == 0) {                                      // 128-bit copies (tensors 16-byte aligned: checked by the wrapper)
    const int wq = width >> 2;
    for (int o = threadIdx.x; o < T * wq; o += 256) {
      const int t = o / wq, c = o - t * wq;
      reinterpret_cast<float4*>(src + ((long long)t * B + j) * width)[c] =
          __ldg(reinterpret_cast<const float4*>(P + ((long long)t * n_total + sidx) * width) + c);
    }
  } else {                                                     // e.g. PAM: 2 * 17 sensors
    for (int o = threadIdx.x; o < T * width; o += 256) {
      const int t = o / width, c = o - t * width;
      src[((long long)t * B + j) * width + c] = __ldg(P + ((long long)t * n_total + sidx) * width + c);
    }
  }
  int local = 0;
  for (int t = threadIdx.x; t < T; t += 256) {
    const float tv = __ldg(Pt + (long long)t * n_total + sidx);
    times[(long long)t * B + j] = tv;
    local += tv > 0.f ? 1 : 0;
  }
  for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
  if ((threadIdx.x & 31) == 0) cnt[threadIdx.x >> 5] = local;
  if (Ps) for (int k = threadIdx.x; k < ds; k += 256) statics[(long long)j * ds + k] = __ldg(Ps + sidx * ds + k);
  __syncthreads();
  if (threadIdx.x == 0) {
    int tot = 0;
    for (int w = 0; w < 8; ++w) tot += cnt[w];
    lengths[j] = tot;
    if (y) y_out[j] = y[sidx];
  }
}

__global__ void rng_capture_kernel(uint64_t* state, uint64_t* cap, int advance) {
  cap[0] = state[0];
  cap[1] = state[1];
  if (advance) state[1] = state[1] + 1;
}

struct TS8 { float v[32]; int d_pe; };      // up to 32 timescales (d_pe <= 64)
// One launch for the two element-wise producers of the forward's inputs:
//   o <  n_lift : X0[(b*N+n), t*d_ob + 0..d_ob) = dropout(relu(src[t,b,n] * R_u[n*d_ob + k]))   code/models_rd.py:285-296,323-327
//                 (one thread per (row, t); for d_ob == 4 one 128-bit store and ONE Philox block per thread)
//   o >= n_lift : positional encoding of token (o - n_lift) / 16 into out[tok*ld + col0 + j]   code/models_rd.py:28-43
__global__ void lift_posenc_kernel(const float* __restrict__ src, const float* __restrict__ R_u, int B, int T, int N,
                                   int d_ob, float drop_p, const uint64_t* __restrict__ rng, int round,
                                   float* __restrict__ X0, long long n_lift, const float* __restrict__ times,
                                   long long n_tokens, TS8 ts, float* __restrict__ pe_out, long long ld, int col0) {
  pdl_launch_dependents();
  pdl_wait();
  long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (o < n_lift) {
    const long long row = o / T;
    const int t = (int)(o - row * T);
    const int b = (int)(row / N), n = (int)(row - (long long)b * N);
    const float sv = __ldg(src + ((long long)t * B + b) * (2 * N) + n);
    const float ik = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
    const uint64_t idx0 = ((uint64_t)t * B + b) * (uint64_t)(N * d_ob) + (uint64_t)(n * d_ob);
    float* dst = X0 + row * ((long long)T * d_ob) + (long long)t * d_ob;
    if (d_ob == 4) {       // idx0 % 4 == 0: the four channels share one Philox block
      const float4 r = __ldg(reinterpret_cast<const float4*>(R_u) + n);
      float4 v = make_float4(fmaxf(sv * r.x, 0.f), fmaxf(sv * r.y, 0.f), fmaxf(sv * r.z, 0.f), fmaxf(sv * r.w, 0.f));
      if (drop_p > 0.f) {
        const float4 m = dropout_scale4(rng, SITE_LIFT, idx0, drop_p, ik);
        v.x *= m.x; v.y *= m.y; v.z *= m.z; v.w *= m.w;
      }
      if (round) v = make_float4(to_tf32(v.x), to_tf32(v.y), to_tf32(v.z), to_tf32(v.w));
      *reinterpret_cast<float4*>(dst) = v;
    } else {
      for (int k = 0; k < d_ob; ++k) {
        float v = fmaxf(sv * __ldg(R_u + n * d_ob + k), 0.f);
        if (drop_p > 0.f) v *= dropout_scale(rng, SITE_LIFT, idx0 + k, drop_p, ik);
        dst[k] = round ? to_tf32(v) : v;
      }
    }
    return;
  }
  o -= n_lift;
  if (o >= n_tokens * ts.d_pe) return;
  const long long tok = o / ts.d_pe;
  const int j = (int)(o - tok * ts.d_pe), half = ts.d_pe >> 1;
  const float scaled = __ldg(times + tok) / ts.v[j < half ? j : j - half];
  pe_out[tok * ld + col0 + j] = (j < half) ? sinf(scaled) : cosf(scaled);
}

// Input gradients that need no GEMM, in one launch (segments as in lift_posenc_kernel):
//   o <  n_src            : token (t, b), sensor n: d_src[t, b, N + n] = 0 (the mask half takes no part in the output,
//                           code/models_rd.py:290); with dX0 (CUDA-core fallback of the lift backward, already gated and
//                           scaled) also d_src[t, b, n] = sum_k dX0[(b*N+n), t*d_ob+k] * R_u[n*d_ob+k]
//   next n_times          : d_times[tok] = sum_j (dZ[tok, pe+j] Z[tok, pe+h+j] - dZ[tok, pe+h+j] Z[tok, pe+j]) / ts_j,
//                           from the saved sin / cos columns (row stride pe_ld) of the encoder input
//                           (code/models_rd.py:33-35); with n_src = n_static = 0 this is rd_positional_encoding_bwd
//   next n_static         : d_static[b, i] = sum_{j < emb} dfeat[b, D+j] emb_w[j, i]        (code/models_rd.py:293-294)
__global__ void input_grad_tail_kernel(int B, int T, int N, int d_ob, int D, long long pe_ld, int pe_col,
                                       const float* __restrict__ dZ, const float* __restrict__ Z, TS8 ts,
                                       const float* __restrict__ dfeat, int Df, const float* __restrict__ emb_w, int emb,
                                       int ds, const float* __restrict__ dX0,
                                       const float* __restrict__ R_u, long long n_src, long long n_times,
                                       long long n_static, float* __restrict__ d_src, float* __restrict__ d_times,
                                       float* __restrict__ d_static) {
  pdl_launch_dependents();
  pdl_wait();
  long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (o < n_src) {
    const long long tok = o / N;
    const int n = (int)(o - tok * N);
    float* dst = d_src + tok * (2LL * N);
    dst[N + n] = 0.f;
    if (dX0) {
      const int t = (int)(tok / B), b = (int)(tok - (long long)t * B);
      const float* g = dX0 + ((long long)b * N + n) * ((long long)T * d_ob) + (long long)t * d_ob;
      float a = 0.f;
      for (int k = 0; k < d_ob; ++k) a += g[k] * __ldg(R_u + n * d_ob + k);
      dst[n] = a;
    }
    return;
  }
  o -= n_src;
  if (o < n_times) {
    const int h = ts.d_pe >> 1;
    const float* dz = dZ + o * pe_ld + pe_col;
    const float* z = Z + o * pe_ld + pe_col;
    float a = 0.f;
    for (int j = 0; j < h; ++j) a += (dz[j] * z[h + j] - dz[h + j] * z[j]) / ts.v[j];
    d_times[o] = a;
    return;
  }
  o -= n_times;
  if (o < n_static) {
    const int b = (int)(o / ds), i = (int)(o - (long long)b * ds);
    const float* df = dfeat + (long long)b * Df + D;
    float a = 0.f;
    for (int j = 0; j < emb; ++j) a += df[j] * __ldg(emb_w + (long long)j * ds + i);
    d_static[o] = a;
  }
}

// one warp per node: segment max, then sum of exp, then s = sum(exp / (sum + 1e-16))
__global__ void node_scale_kernel(const int64_t* __restrict__ tgt, const float* __restrict__ w, int E, int N,
                                  float* __restrict__ s) {
  int node = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (node >= N) return;
  float mx = -INFINITY;
  for (int e = lane; e < E; e += 32)
    if (tgt[e] == node) mx = fmaxf(mx, w[e]);
  mx = warp_max(mx);
  if (mx == -INFINITY) {  // no incoming edge: scatter-add leaves the row at exactly zero
    if (lane == 0) s[node] = 0.f;
    return;
  }
  float sum = 0.f;
  for (int e = lane; e < E; e += 32)
    if (tgt[e] == node) sum += expf(w[e] - mx);
  sum = warp_sum(sum);
  float den = sum + 1e-16f;
  float acc = 0.f;
  for (int e = lane; e < E; e += 32)
    if (tgt[e] == node) acc += expf(w[e] - mx) / den;
  acc = warp_sum(acc);
  if (lane == 0) s[node] = acc;
}

__global__ void layernorm_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                     const float* __restrict__ beta, long long rows, int D, float eps,
                                     float* __restrict__ y, float* __restrict__ stats) {
  pdl_launch_dependents();
  pdl_wait();
  long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + row * D;
  float s = 0.f;
  for (int j = lane; j < D; j += 32) s += xr[j];
  float mean = warp_sum(s) / (float)D;
  float q = 0.f;
  for (int j = lane; j < D; j += 32) { float d = xr[j] - mean; q += d * d; }
  float var = warp_sum(q) / (float)D;
  float rstd = 1.f / sqrtf(var + eps);
  float* yr = y + row * D;
  for (int j = lane; j < D; j += 32) yr[j] = (xr[j] - mean) * rstd * __ldg(gamma + j) + __ldg(beta + j);
  if (lane == 0) { stats[2 * row] = mean; stats[2 * row + 1] = rstd; }
}

// The same with the row held in registers (ITERS float4 per lane, D % 4 == 0, D <= 128 * ITERS): one global read instead of
// three, 128-bit accesses.
template <int ITERS>
__global__ void __launch_bounds__(256) layernorm_fwd_vec_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                                const float* __restrict__ beta, long long rows, int D, float eps,
                                                                float* __restrict__ y, float* __restrict__ stats) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr int RB = 1;      // one row per warp: more warps in flight beats fewer, fatter ones at these sizes
  const int lane = threadIdx.x & 31;
  const long long row0 = ((long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * RB;
  float4 v[RB][ITERS];
  float s[RB], q[RB];
#pragma unroll
  for (int k = 0; k < RB; ++k) {
    s[k] = 0.f;
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
      const int j = 4 * lane + 128 * it;
      v[k][it] = (row0 + k < rows && j < D) ? *reinterpret_cast<const float4*>(x + (row0 + k) * D + j) : make_float4(0.f, 0.f, 0.f, 0.f);
      s[k] += (v[k][it].x + v[k][it].y) + (v[k][it].z + v[k][it].w);
    }
  }
#pragma unroll
  for (int k = 0; k < RB; ++k) s[k] = warp_sum(s[k]) / (float)D;
#pragma unroll
  for (int k = 0; k < RB; ++k) {
    q[k] = 0.f;
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
      if (4 * lane + 128 * it < D) {
        const float a = v[k][it].x - s[k], b = v[k][it].y - s[k], c = v[k][it].z - s[k], d = v[k][it].w - s[k];
        q[k] += (a * a + b * b) + (c * c + d * d);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < RB; ++k) q[k] = 1.f / sqrtf(warp_sum(q[k]) / (float)D + eps);
#pragma unroll
  for (int it = 0; it < ITERS; ++it) {
    const int j = 4 * lane + 128 * it;
    if (j < D) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + j)), bt = __ldg(reinterpret_cast<const float4*>(beta + j));
#pragma unroll
      for (int k = 0; k < RB; ++k) {
        if (row0 + k < rows) {
          float4 o;
          o.x = (v[k][it].x - s[k]) * q[k] * g.x + bt.x; o.y = (v[k][it].y - s[k]) * q[k] * g.y + bt.y;
          o.z = (v[k][it].z - s[k]) * q[k] * g.z + bt.z; o.w = (v[k][it].w - s[k]) * q[k] * g.w + bt.w;
          *reinterpret_cast<float4*>(y + (row0 + k) * D + j) = o;
        }
      }
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < RB; ++k)
      if (row0 + k < rows) { stats[2 * (row0 + k)] = s[k]; stats[2 * (row0 + k) + 1] = q[k]; }
  }
}

// LayerNorm backward, one pass over (x, dy): every warp walks LNB_ROWS/8 rows, writes dx (and the
// dropout-masked copy the sub-layer's weight gradient needs) and keeps per-lane column sums of
// dy*xhat / dy in registers; the 8 warps of a CTA combine them through shared memory into one
// partial row [2][D] per CTA (summed later in a fixed order).  128-bit accesses (D % 4 == 0).
constexpr int LNB_ROWS = 32;    // rows per CTA of the wide (D > 256) variant: 4 sequential rows per warp
constexpr int LNB_ROWS_NARROW = 8;   // D <= 256: one row per warp -- 7680 rows = 52 warps per SM in flight; with 4 rows per warp
                                     // there were 13, and the kernel sat at 9 cycles per issued instruction (latency bound)
constexpr int LNB_MAXIT = 5;    // D <= 640
// ITERS float4 per lane and row (D <= 128 * ITERS); RB rows of a warp are in flight together: their loads are all issued
// before the first reduction, so a warp pays one memory round trip for RB rows instead of RB dependent ones.
template <int ITERS, int RB, int ROWS>
__global__ void __launch_bounds__(256, (ITERS <= 2 && RB == 1) ? 4 : 2) layernorm_bwd_fused_kernel(
    const float* __restrict__ x, const float* __restrict__ stats, const float* __restrict__ gamma,
    const float* __restrict__ dy, long long rows, int D, float* __restrict__ dx, float* __restrict__ dx_drop,
    float drop_p, const uint64_t* __restrict__ rng, uint32_t site, float* __restrict__ partial,
    const uint32_t* __restrict__ keep_bits, int keep_ld) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float lsm[];                     // [8 warps][2][D]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float ik = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
  const RngKey key = load_rng_key(dx_drop && !keep_bits ? rng : nullptr);
  float4 ag[ITERS], ab[ITERS], g4[ITERS];
#pragma unroll
  for (int it = 0; it < ITERS; ++it) {
    ag[it] = make_float4(0.f, 0.f, 0.f, 0.f); ab[it] = ag[it];
    const int j = 4 * lane + 128 * it;
    g4[it] = j < D ? __ldg(reinterpret_cast<const float4*>(gamma + j)) : ag[it];
  }
  const long long r0 = (long long)blockIdx.x * ROWS;
  for (int rr = warp; rr < ROWS; rr += 8 * RB) {
    float4 d4[RB][ITERS], xh[RB][ITERS];
    float rstd[RB], s1[RB], s2[RB];
#pragma unroll
    for (int k = 0; k < RB; ++k) {
      const long long row = r0 + rr + 8 * k;
      const bool ok = row < rows;
      const float mean = ok ? stats[2 * row] : 0.f;
      rstd[k] = ok ? stats[2 * row + 1] : 0.f;
      s1[k] = 0.f; s2[k] = 0.f;
#pragma unroll
      for (int it = 0; it < ITERS; ++it) {
        const int j = 4 * lane + 128 * it;
        d4[k][it] = make_float4(0.f, 0.f, 0.f, 0.f); xh[k][it] = d4[k][it];
        if (ok && j < D) {
          d4[k][it] = *reinterpret_cast<const float4*>(dy + row * D + j);
          const float4 x4 = *reinterpret_cast<const float4*>(x + row * D + j);
          xh[k][it] = make_float4((x4.x - mean) * rstd[k], (x4.y - mean) * rstd[k], (x4.z - mean) * rstd[k], (x4.w - mean) * rstd[k]);
        }
      }
    }
#pragma unroll
    for (int k = 0; k < RB; ++k) {
#pragma unroll
      for (int it = 0; it < ITERS; ++it) {
        const float4 d = d4[k][it], g = g4[it], h = xh[k][it];
        s1[k] += d.x * g.x + d.y * g.y + d.z * g.z + d.w * g.w;
        s2[k] += d.x * g.x * h.x + d.y * g.y * h.y + d.z * g.z * h.z + d.w * g.w * h.w;
      }
    }
#pragma unroll
    for (int k = 0; k < RB; ++k) { s1[k] = warp_sum(s1[k]) / (float)D; s2[k] = warp_sum(s2[k]) / (float)D; }
#pragma unroll
    for (int k = 0; k < RB; ++k) {
      const long long row = r0 + rr + 8 * k;
      if (row >= rows) continue;
#pragma unroll
      for (int it = 0; it < ITERS; ++it) {
        const int j = 4 * lane + 128 * it;
        if (j < D) {
          const float4 d = d4[k][it], g = g4[it], h = xh[k][it];
          float4 o;
          o.x = rstd[k] * (d.x * g.x - s1[k] - h.x * s2[k]);
          o.y = rstd[k] * (d.y * g.y - s1[k] - h.y * s2[k]);
          o.z = rstd[k] * (d.z * g.z - s1[k] - h.z * s2[k]);
          o.w = rstd[k] * (d.w * g.w - s1[k] - h.w * s2[k]);
          *reinterpret_cast<float4*>(dx + row * D + j) = o;
          if (dx_drop) {
            float4 m;
            if (keep_bits) {      // decisions stored by the forward GEMM epilogue: word [row, j / 32], bit j % 32
              const uint32_t b4 = (__ldg(keep_bits + row * keep_ld + (j >> 5)) >> (j & 31)) & 15u;
              m = make_float4(b4 & 1u ? ik : 0.f, b4 & 2u ? ik : 0.f, b4 & 4u ? ik : 0.f, b4 & 8u ? ik : 0.f);
            } else {
              m = dropout_scale4(key, site, (uint64_t)row * D + j, drop_p, ik);
            }
            *reinterpret_cast<float4*>(dx_drop + row * D + j) = make_float4(o.x * m.x, o.y * m.y, o.z * m.z, o.w * m.w);
          }
          ag[it].x += d.x * h.x; ag[it].y += d.y * h.y; ag[it].z += d.z * h.z; ag[it].w += d.w * h.w;
          ab[it].x += d.x; ab[it].y += d.y; ab[it].z += d.z; ab[it].w += d.w;
        }
      }
    }
  }
#pragma unroll
  for (int it = 0; it < ITERS; ++it) {
    const int j = 4 * lane + 128 * it;
    if (j < D) {
      *reinterpret_cast<float4*>(lsm + (warp * 2) * D + j) = ag[it];
      *reinterpret_cast<float4*>(lsm + (warp * 2 + 1) * D + j) = ab[it];
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * D; c += blockDim.x) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += lsm[w * 2 * D + c];     // c < D: dgamma column, else dbeta column
    partial[(long long)blockIdx.x * 2 * D + c] = s;
  }
}

__global__ void layernorm_bwd_dx_kernel(const float* __restrict__ x, const float* __restrict__ stats,
                                        const float* __restrict__ gamma, const float* __restrict__ dy,
                                        long long rows, int D, float* __restrict__ dx, float* __restrict__ dx_drop,
                                        float drop_p, const uint64_t* __restrict__ rng, uint32_t site) {
  long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + row * D;
  const float* dyr = dy + row * D;
  float mean = stats[2 * row], rstd = stats[2 * row + 1];
  const float ik = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
  float s1 = 0.f, s2 = 0.f;
  if ((D & 3) == 0 && ((reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dy) |
                        reinterpret_cast<uintptr_t>(dx) | reinterpret_cast<uintptr_t>(dx_drop)) & 15) == 0) {   // 128-bit path: lane owns columns 4*lane + 128*it
    for (int j = 4 * lane; j < D; j += 128) {
      const float4 d4 = *reinterpret_cast<const float4*>(dyr + j), x4 = *reinterpret_cast<const float4*>(xr + j);
      const float4 g4 = __ldg(reinterpret_cast<const float4*>(gamma + j));
      const float g[4] = {d4.x * g4.x, d4.y * g4.y, d4.z * g4.z, d4.w * g4.w};
      const float xh[4] = {(x4.x - mean) * rstd, (x4.y - mean) * rstd, (x4.z - mean) * rstd, (x4.w - mean) * rstd};
#pragma unroll
      for (int e = 0; e < 4; ++e) { s1 += g[e]; s2 += g[e] * xh[e]; }
    }
    s1 = warp_sum(s1) / (float)D;
    s2 = warp_sum(s2) / (float)D;
    for (int j = 4 * lane; j < D; j += 128) {
      const float4 d4 = *reinterpret_cast<const float4*>(dyr + j), x4 = *reinterpret_cast<const float4*>(xr + j);
      const float4 g4 = __ldg(reinterpret_cast<const float4*>(gamma + j));
      float4 o;
      o.x = rstd * (d4.x * g4.x - s1 - (x4.x - mean) * rstd * s2);
      o.y = rstd * (d4.y * g4.y - s1 - (x4.y - mean) * rstd * s2);
      o.z = rstd * (d4.z * g4.z - s1 - (x4.z - mean) * rstd * s2);
      o.w = rstd * (d4.w * g4.w - s1 - (x4.w - mean) * rstd * s2);
      *reinterpret_cast<float4*>(dx + row * D + j) = o;
      if (dx_drop) {
        const float4 m = dropout_scale4(rng, site, (uint64_t)row * D + j, drop_p, ik);
        *reinterpret_cast<float4*>(dx_drop + row * D + j) = make_float4(o.x * m.x, o.y * m.y, o.z * m.z, o.w * m.w);
      }
    }
    return;
  }
  for (int j = lane; j < D; j += 32) {
    float g = dyr[j] * __ldg(gamma + j);
    float xh = (xr[j] - mean) * rstd;
    s1 += g;
    s2 += g * xh;
  }
  s1 = warp_sum(s1) / (float)D;
  s2 = warp_sum(s2) / (float)D;
  float* dxr = dx + row * D;
  for (int j = lane; j < D; j += 32) {
    float g = dyr[j] * __ldg(gamma + j);
    float xh = (xr[j] - mean) * rstd;
    float v = rstd * (g - s1 - xh * s2);
    dxr[j] = v;
    if (dx_drop) dx_drop[row * D + j] = v * dropout_scale(rng, site, (uint64_t)row * D + j, drop_p, ik);
  }
}

constexpr int LN_ROWS = 256;   // rows per CTA: 8 row groups x 32 rows, reduced through shared memory
// partial[chunk][0][j] = sum_rows dy * xhat, partial[chunk][1][j] = sum_rows dy
__global__ void layernorm_bwd_param_kernel(const float* __restrict__ x, const float* __restrict__ stats,
                                           const float* __restrict__ dy, long long rows, int D,
                                           float* __restrict__ partial) {
  __shared__ float sg[8][33], sb[8][33];
  const int j = blockIdx.x * 32 + threadIdx.x;
  const long long r0 = (long long)blockIdx.y * LN_ROWS + threadIdx.y * 32;
  float dg = 0.f, db = 0.f;
  if (j < D) {
    const long long r1 = min(rows, r0 + 32);
    for (long long r = r0; r < r1; ++r) {
      float d = dy[r * D + j];
      dg += d * (x[r * D + j] - stats[2 * r]) * stats[2 * r + 1];
      db += d;
    }
  }
  sg[threadIdx.y][threadIdx.x] = dg;
  sb[threadIdx.y][threadIdx.x] = db;
  __syncthreads();
  if (threadIdx.y == 0 && j < D) {
#pragma unroll
    for (int g = 1; g < 8; ++g) { dg += sg[g][threadIdx.x]; db += sb[g][threadIdx.x]; }
    partial[((long long)blockIdx.y * 2) * D + j] = dg;
    partial[((long long)blockIdx.y * 2 + 1) * D + j] = db;
  }
}

__global__ void attn_softmax_fwd_kernel(float* __restrict__ S, const int64_t* __restrict__ lengths, int B, int H,
                                        int T, float drop_p, const uint64_t* __restrict__ rng, uint32_t site,
                                        float* __restrict__ Pd) {
  long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  long long rows = (long long)B * H * T;
  if (row >= rows) return;
  int b = (int)(row / ((long long)H * T));
  long long len = lengths[b];
  int nv = (int)(len < T ? (len < 0 ? 0 : len) : T);
  float* sr = S + row * T;
  float mx = -INFINITY;
  for (int j = lane; j < nv; j += 32) mx = fmaxf(mx, sr[j]);
  mx = warp_max(mx);
  float sum = 0.f;
  for (int j = lane; j < nv; j += 32) sum += expf(sr[j] - mx);
  sum = warp_sum(sum);
  float inv = nv > 0 ? 1.f / sum : 0.f;
  float ik = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
  for (int j = lane; j < T; j += 32) {
    float p = j < nv ? expf(sr[j] - mx) * inv : 0.f;
    sr[j] = p;
    if (Pd) {
      float m = drop_p > 0.f ? dropout_scale(rng, site, (uint64_t)row * T + j, drop_p, ik) : 1.f;
      Pd[row * T + j] = p * m;
    }
  }
}

__global__ void attn_softmax_bwd_kernel(const float* __restrict__ P, float* __restrict__ dP, long long rows, int T,
                                        float drop_p, const uint64_t* __restrict__ rng, uint32_t site) {
  long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* pr = P + row * T;
  float* dr = dP + row * T;
  float ik = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
  float dot = 0.f;
  for (int j = lane; j < T; j += 32) {
    float m = drop_p > 0.f ? dropout_scale(rng, site, (uint64_t)row * T + j, drop_p, ik) : 1.f;
    dot += dr[j] * m * pr[j];
  }
  dot = warp_sum(dot);
  for (int j = lane; j < T; j += 32) {
    float m = drop_p > 0.f ? dropout_scale(rng, site, (uint64_t)row * T + j, drop_p, ik) : 1.f;
    dr[j] = pr[j] * (dr[j] * m - dot);
  }
}

__global__ void obprop_out_grad_kernel(const float* __restrict__ dZ, const float* __restrict__ Z,
                                       const float* __restrict__ s, int B, int T, int N, int d_ob, int D,
                                       int round, float* __restrict__ dZ2) {
  pdl_launch_dependents();
  pdl_wait();
  const long long C = (long long)T * d_ob;
  long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= (long long)B * N * C) return;
  long long row = o / C;
  int c = (int)(o - row * C);
  int b = (int)(row / N), n = (int)(row - (long long)b * N);
  int t = c / d_ob, k = c - t * d_ob;
  long long zi = ((long long)t * B + b) * D + n * d_ob + k;
  float v = (Z[zi] > 0.f) ? dZ[zi] * __ldg(s + n) : 0.f;
  dZ2[o] = round ? to_tf32(v) : v;
}

// d_ob == 4: one thread per (row, timestamp), the four channels as one 128-bit access (Z0 rows are 16-byte aligned: D % 4 == 0)
__global__ void obprop_out_grad_vec4_kernel(const float* __restrict__ dZ, const float* __restrict__ Z,
                                            const float* __restrict__ s, int B, int T, int N, int D, int round,
                                            float* __restrict__ dZ2) {
  pdl_launch_dependents();
  pdl_wait();
  const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= (long long)B * N * T) return;
  const long long row = o / T;
  const int t = (int)(o - row * T);
  const int b = (int)(row / N), n = (int)(row - (long long)b * N);
  const long long zi = ((long long)t * B + b) * D + n * 4;
  const float4 z = *reinterpret_cast<const float4*>(Z + zi), g = *reinterpret_cast<const float4*>(dZ + zi);
  const float sc = __ldg(s + n);
  float4 v = make_float4(z.x > 0.f ? g.x * sc : 0.f, z.y > 0.f ? g.y * sc : 0.f, z.z > 0.f ? g.z * sc : 0.f, z.w > 0.f ? g.w * sc : 0.f);
  if (round) v = make_float4(to_tf32(v.x), to_tf32(v.y), to_tf32(v.z), to_tf32(v.w));
  *reinterpret_cast<float4*>(dZ2 + o * 4) = v;
}

__global__ void apply_dropout_kernel(const float* __restrict__ x, long long n, float p,
                                     const uint64_t* __restrict__ rng, uint32_t site, float* __restrict__ y) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float xv = x ? x[i] : 1.f;
  y[i] = xv * dropout_scale(rng, site, (uint64_t)i, p, 1.f / (1.f - p));
}

__global__ void relu_scale_bwd_kernel(const float* __restrict__ d_out, const float* __restrict__ out,
                                      const float* __restrict__ scale, int mod, long long rows, int C,
                                      float* __restrict__ d_pre) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * C) return;
  long long r = i / C;
  d_pre[i] = out[i] > 0.f ? d_out[i] * __ldg(scale + (r % mod)) : 0.f;
}

__global__ void cross_entropy_kernel(const float* __restrict__ logits, const int64_t* __restrict__ y, int B, int ncls,
                                     float* __restrict__ loss, float* __restrict__ dlogits) {
  __shared__ float red[TPB / 32];
  float local = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const float* l = logits + (long long)b * ncls;
    float mx = -INFINITY;
    for (int c = 0; c < ncls; ++c) mx = fmaxf(mx, l[c]);
    float sum = 0.f;
    for (int c = 0; c < ncls; ++c) sum += expf(l[c] - mx);
    float lse = mx + logf(sum);
    int yy = (int)y[b];
    local += lse - l[yy];
    if (dlogits) {
      float invB = 1.f / (float)B;
      for (int c = 0; c < ncls; ++c)
        dlogits[(long long)b * ncls + c] = (expf(l[c] - lse) - (c == yy ? 1.f : 0.f)) * invB;
    }
  }
  local = warp_sum(local);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
    *loss = s / (float)B;
  }
}

// One launch: every CTA reads the step count t (before anyone changes it), updates its slice with bias
// corrections for t + 1, and the LAST CTA to finish stores t + 1 (ticket in step[1], self-resetting).
__device__ __forceinline__ void adam_el(float& p, float g, float& m, float& v, float b1, float b2, float eps, float gscale,
                                        float bc1, float bc2s, float lr) {
  const float gi = g * gscale;
  m = b1 * m + (1.f - b1) * gi;
  v = b2 * v + (1.f - b2) * gi * gi;
  const float denom = sqrtf(v) / bc2s + eps;
  p -= (lr / bc1) * (m / denom);
}
// A few CTAs per SM stride over the flat buffers in 128-bit pieces (`vec`: all four pointers 16-byte aligned): the bias
// corrections (two double-precision pow) and the ticket atomic are per CTA, and with one element per thread there were
// ~2000 CTAs each paying them for 256 elements of work.
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, long long n, int vec, float lr, const float* __restrict__ lr_dev, float b1,
                            float b2, float eps, float gscale, int64_t* __restrict__ step) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float bc[3];
  if (threadIdx.x == 0) {
    double t = (double)(*reinterpret_cast<volatile int64_t*>(step) + 1);
    bc[0] = (float)(1.0 - pow((double)b1, t));
    bc[1] = (float)sqrt(1.0 - pow((double)b2, t));
    bc[2] = lr_dev ? *lr_dev : lr;
  }
  __syncthreads();
  const float bc1 = bc[0], bc2s = bc[1], lrv = bc[2];
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, stride = (long long)gridDim.x * blockDim.x;
  const long long n4 = vec ? n >> 2 : 0;
  for (long long i = tid; i < n4; i += stride) {
    float4 pp = reinterpret_cast<float4*>(p)[i], mm = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
    const float4 gg = reinterpret_cast<const float4*>(g)[i];
    adam_el(pp.x, gg.x, mm.x, vv.x, b1, b2, eps, gscale, bc1, bc2s, lrv);
    adam_el(pp.y, gg.y, mm.y, vv.y, b1, b2, eps, gscale, bc1, bc2s, lrv);
    adam_el(pp.z, gg.z, mm.z, vv.z, b1, b2, eps, gscale, bc1, bc2s, lrv);
    adam_el(pp.w, gg.w, mm.w, vv.w, b1, b2, eps, gscale, bc1, bc2s, lrv);
    reinterpret_cast<float4*>(p)[i] = pp; reinterpret_cast<float4*>(m)[i] = mm; reinterpret_cast<float4*>(v)[i] = vv;
  }
  for (long long i = 4 * n4 + tid; i < n; i += stride) adam_el(p[i], g[i], m[i], v[i], b1, b2, eps, gscale, bc1, bc2s, lrv);
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long* ticket = reinterpret_cast<unsigned long long*>(step + 1);
    if (atomicAdd(ticket, 1ull) == (unsigned long long)(gridDim.x - 1)) {
      *ticket = 0ull;
      step[0] = step[0] + 1;
    }
  }
}

}  // namespace

// ---- wrappers ----------------------------------------------------------------------------------
int64_t feature_stats_scratch_bytes(int64_t n, int T, int F) {
  int64_t chunks = ceil_div(n * T, 4096);
  if (chunks > 512) chunks = 512;
  if (chunks < 1) chunks = 1;
  return chunks * F * 3 * (int64_t)sizeof(double);
}
int feature_stats(const float* raw, int64_t n, int T, int F, float* mean, float* stdv, void* scratch, cudaStream_t st) {
  int64_t chunks = ceil_div(n * T, 4096);
  if (chunks > 512) chunks = 512;
  if (chunks < 1) chunks = 1;
  if (F > 65535) { set_error("feature_stats: too many features"); return -2; }
  feature_stats_partial_kernel<<<dim3((unsigned)chunks, (unsigned)F), FS_THREADS, 0, st>>>(raw, n * T, F, (double*)scratch);
  RD_CHECK_LAUNCH("feature_stats_partial_kernel");
  feature_stats_final_kernel<<<blocks_for(F), TPB, 0, st>>>((const double*)scratch, (int)chunks, F, mean, stdv);
  RD_CHECK_LAUNCH("feature_stats_final_kernel");
  return 0;
}
int mask_normalize(const float* raw, const float* mean, const float* stdv, int64_t n, int T, int F, float* out,
                   const float* minutes, float* times_out, cudaStream_t st) {
  if (n * T * F <= 0) return 0;
  mask_normalize_kernel<<<blocks_for(n * T * F), TPB, 0, st>>>(raw, mean, stdv, n, T, F, out, minutes, times_out);
  RD_CHECK_LAUNCH("mask_normalize_kernel");
  return 0;
}
int zero_features(float* P, int64_t T, int B, int width, const int64_t* idx, int K, int per_sample, cudaStream_t st) {
  if (T * B * K <= 0) return 0;
  zero_features_kernel<<<blocks_for(T * B * K), TPB, 0, st>>>(P, T, B, width, idx, K, per_sample);
  RD_CHECK_LAUNCH("zero_features_kernel");
  return 0;
}
int assemble_batch(const float* P, const float* Pt, const float* Ps, const int64_t* y, const int64_t* idx, int T, int64_t n_total,
                   int width, int ds, int B, float* src, float* times, float* statics, int64_t* y_out, int64_t* lengths,
                   cudaStream_t st) {
  if ((width & 3) == 0 && ((reinterpret_cast<uintptr_t>(P) | reinterpret_cast<uintptr_t>(src)) & 15)) {
    set_error("assemble_batch: 16-byte aligned tensors required when width %% 4 == 0");
    return -2;
  }
  if (B <= 0) return 0;
  launch_pdl(assemble_batch_kernel, dim3(B), dim3(256), 0, st, P, Pt, Ps, y, idx, T, (long long)n_total, width, ds, B, src, times, statics,
             y_out, lengths);
  RD_CHECK_LAUNCH("assemble_batch_kernel");
  return 0;
}

int rng_capture(uint64_t* state, uint64_t* cap, int advance, cudaStream_t st) {
  rng_capture_kernel<<<1, 1, 0, st>>>(state, cap, advance);
  RD_CHECK_LAUNCH("rng_capture_kernel");
  return 0;
}

int transpose_round(const float* x, int rows, int cols, float* y, cudaStream_t st) {
  dim3 grid((unsigned)ceil_div(cols, 32), (unsigned)ceil_div(rows, 32));
  transpose_round_kernel<<<grid, dim3(32, 8), 0, st>>>(x, rows, cols, y);
  RD_CHECK_LAUNCH("transpose_round_kernel");
  return 0;
}

int gather_batch(const float* src, const int64_t* idx, int64_t T, int64_t n_total, int width, int B, float* out,
                 cudaStream_t st) {
  if ((width & 3) == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(out)) & 15)) {
    set_error("gather_batch: 16-byte aligned buffers required when width %% 4 == 0");
    return -2;
  }
  const int64_t n = T * B * (int64_t)(width / ((width & 3) == 0 ? 4 : 1));
  if (n <= 0) return 0;
  gather_batch_kernel<<<blocks_for(n), TPB, 0, st>>>(src, idx, T, n_total, width, B, out);
  RD_CHECK_LAUNCH("gather_batch_kernel");
  return 0;
}

int lift_posenc(const float* src, const float* R_u, int B, int T, int N, int d_ob, float drop_p, const uint64_t* rng,
                int round, float* X0, const float* times, int64_t n_tokens, const float* ts_host, int d_pe, float* pe_out,
                int64_t ld, int col0, cudaStream_t st) {
  if (times && (d_pe < 2 || d_pe > 64 || (d_pe & 1))) { set_error("positional encoding width must be even and <= 64"); return -2; }
  const int64_t n_lift = src ? (int64_t)B * N * T : 0;      // one thread per (row, t)
  const int64_t n_pe = times ? n_tokens * d_pe : 0;
  TS8 ts;
  memset(&ts, 0, sizeof(ts));
  ts.d_pe = times ? d_pe : 2;
  if (times) memcpy(ts.v, ts_host, sizeof(float) * (d_pe / 2));
  if (n_lift + n_pe <= 0) return 0;
  launch_pdl(lift_posenc_kernel, dim3(blocks_for(n_lift + n_pe)), dim3(TPB), 0, st, src, R_u, B, T, N, d_ob, drop_p, rng, round, X0,
             (long long)n_lift, times, (long long)(times ? n_tokens : 0), ts, pe_out, (long long)ld, col0);
  RD_CHECK_LAUNCH("lift_posenc_kernel");
  return 0;
}

int posenc(const float* times, int64_t n_tokens, const float* ts_host, int d_pe, float* out, int64_t ld, int col0,
           cudaStream_t st) {
  return lift_posenc(nullptr, nullptr, 0, 0, 0, 0, 0.f, nullptr, 0, nullptr, times, n_tokens, ts_host, d_pe, out, ld, col0, st);
}

static int launch_input_grad_tail(int B, int T, int N, int d_ob, int D, int64_t pe_ld, int pe_col, const float* dZ,
                                  const float* Z, const float* ts_host, int d_pe, const float* dfeat, int Df,
                                  const float* emb_w, int emb, int ds, const float* dX0, const float* R_u, int64_t n_src,
                                  int64_t n_times, int64_t n_static, float* d_src, float* d_times, float* d_static,
                                  cudaStream_t st) {
  if (d_pe < 2 || d_pe > 64 || (d_pe & 1)) { set_error("positional encoding width must be even and <= 64"); return -2; }
  TS8 ts;
  memset(&ts, 0, sizeof(ts));
  ts.d_pe = d_pe;
  memcpy(ts.v, ts_host, sizeof(float) * (d_pe / 2));
  const int64_t total = n_src + n_times + n_static;
  if (total <= 0) return 0;
  launch_pdl(input_grad_tail_kernel, dim3(blocks_for(total)), dim3(TPB), 0, st, B, T, N, d_ob, D, (long long)pe_ld, pe_col,
             dZ, Z, ts, dfeat, Df, emb_w, emb, ds, dX0, R_u, (long long)n_src, (long long)n_times, (long long)n_static, d_src,
             d_times, d_static);
  RD_CHECK_LAUNCH("input_grad_tail_kernel");
  return 0;
}

int input_grad_tail(int B, int T, int N, int d_ob, int D, const float* dZ, const float* Z, const float* ts_host,
                    int d_pe, const float* dfeat, int Df, const float* emb_w, int emb, int ds, const float* dX0,
                    const float* R_u, float* d_src, float* d_times, float* d_static, cudaStream_t st) {
  const int64_t n_src = d_src ? (int64_t)T * B * N : 0;
  const int64_t n_times = d_times ? (int64_t)T * B : 0;
  const int64_t n_static = d_static ? (int64_t)B * ds : 0;
  return launch_input_grad_tail(B, T, N, d_ob, D, D, D - d_pe, dZ, Z, ts_host, d_pe, dfeat, Df, emb_w, emb, ds, dX0, R_u,
                                n_src, n_times, n_static, d_src, d_times, d_static, st);
}

int posenc_bwd(const float* pe, const float* d_pe, int64_t n_tokens, const float* ts_host, int width, int64_t ld, int col0,
               float* d_times, cudaStream_t st) {
  return launch_input_grad_tail(0, 0, 0, 0, 0, ld, col0, d_pe, pe, ts_host, width, nullptr, 0, nullptr, 0, 0, nullptr,
                                nullptr, 0, n_tokens, 0, nullptr, d_times, nullptr, st);
}

int node_scale(const int64_t* edge_tgt, const float* edge_w, int E, int N, float* s, cudaStream_t st) {
  node_scale_kernel<<<blocks_for((int64_t)N * 32), TPB, 0, st>>>(edge_tgt, edge_w, E, N, s);
  RD_CHECK_LAUNCH("node_scale_kernel");
  return 0;
}

int layernorm_fwd(const float* x, const float* gamma, const float* beta, int64_t rows, int D, float eps, float* y,
                  float* stats, cudaStream_t st) {
  const uintptr_t bits = reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(beta);
  if ((D & 3) == 0 && D <= 640 && (bits & 15) == 0) {
    const unsigned blocks = (unsigned)ceil_div(rows, (int64_t)(TPB / 32));          // 8 warps, one row each
    if (D <= 128) launch_pdl(layernorm_fwd_vec_kernel<1>, dim3(blocks), dim3(TPB), 0, st, x, gamma, beta, (long long)rows, D, eps, y, stats);
    else if (D <= 256) launch_pdl(layernorm_fwd_vec_kernel<2>, dim3(blocks), dim3(TPB), 0, st, x, gamma, beta, (long long)rows, D, eps, y, stats);
    else launch_pdl(layernorm_fwd_vec_kernel<5>, dim3(blocks), dim3(TPB), 0, st, x, gamma, beta, (long long)rows, D, eps, y, stats);
    RD_CHECK_LAUNCH("layernorm_fwd_vec_kernel");
    return 0;
  }
  launch_pdl(layernorm_fwd_kernel, dim3(blocks_for(rows * 32)), dim3(TPB), 0, st, x, gamma, beta, (long long)rows, D, eps, y, stats);
  RD_CHECK_LAUNCH("layernorm_fwd_kernel");
  return 0;
}

int64_t ln_bwd_scratch_floats(int64_t rows, int D) {
  int64_t a = ceil_div(rows, LN_ROWS), b = ceil_div(rows, D <= 256 ? LNB_ROWS_NARROW : LNB_ROWS);
  return (a > b ? a : b) * 2 * D;
}

int layernorm_bwd(const float* x, const float* stats, const float* gamma, const float* dy, int64_t rows, int D,
                  float* dx, float* dgamma, float* dbeta, float* scratch, float* dx_drop, float drop_p,
                  const uint64_t* rng, uint32_t site, int* deferred_chunks, cudaStream_t st, const uint32_t* keep_bits,
                  int keep_ld) {
  const uintptr_t bits = reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dy) |
                         reinterpret_cast<uintptr_t>(dx) | reinterpret_cast<uintptr_t>(dx_drop);
  int chunks;
  if ((D & 3) == 0 && D <= 128 * LNB_MAXIT && (bits & 15) == 0) {     // fused single pass
    chunks = (int)ceil_div(rows, D <= 256 ? LNB_ROWS_NARROW : LNB_ROWS);
    auto kern = D <= 128 ? layernorm_bwd_fused_kernel<1, 1, LNB_ROWS_NARROW>
                         : (D <= 256 ? layernorm_bwd_fused_kernel<2, 1, LNB_ROWS_NARROW> : layernorm_bwd_fused_kernel<LNB_MAXIT, 1, LNB_ROWS>);
    launch_pdl(kern, dim3(chunks), dim3(256), 8 * 2 * D * sizeof(float), st, x, stats, gamma, dy, (long long)rows, D,
               dx, drop_p > 0.f ? dx_drop : (float*)nullptr, drop_p, rng, site, scratch, keep_bits, keep_ld);
    RD_CHECK_LAUNCH("layernorm_bwd_fused_kernel");
  } else {
    layernorm_bwd_dx_kernel<<<blocks_for(rows * 32), TPB, 0, st>>>(x, stats, gamma, dy, rows, D, dx,
                                                                drop_p > 0.f ? dx_drop : nullptr, drop_p, rng, site);
    RD_CHECK_LAUNCH("layernorm_bwd_dx_kernel");
    chunks = (int)ceil_div(rows, LN_ROWS);
    if (chunks > 65535) { set_error("layernorm_bwd: too many row chunks"); return -2; }
    dim3 grid((unsigned)ceil_div(D, 32), (unsigned)chunks);
    layernorm_bwd_param_kernel<<<grid, dim3(32, 8), 0, st>>>(x, stats, dy, rows, D, scratch);
    RD_CHECK_LAUNCH("layernorm_bwd_param_kernel");
  }
  // scratch = [chunks][2][D] partial column sums -> dgamma, dbeta (fixed order, deterministic)
  if (deferred_chunks) { *deferred_chunks = chunks; return 0; }     // the caller folds this into a later reduction launch
  return reduce_partials2(scratch, chunks, D, dgamma, D, dbeta, st);
}

int attn_softmax_fwd(float* S, const int64_t* lengths, int B, int H, int T, float drop_p, const uint64_t* rng,
                     uint32_t site, float* Pd, cudaStream_t st) {
  int64_t rows = (int64_t)B * H * T;
  attn_softmax_fwd_kernel<<<blocks_for(rows * 32), TPB, 0, st>>>(S, lengths, B, H, T, drop_p, rng, site, Pd);
  RD_CHECK_LAUNCH("attn_softmax_fwd_kernel");
  return 0;
}

int attn_softmax_bwd(const float* P, float* dP, int B, int H, int T, float drop_p, const uint64_t* rng,
                     uint32_t site, cudaStream_t st) {
  int64_t rows = (int64_t)B * H * T;
  attn_softmax_bwd_kernel<<<blocks_for(rows * 32), TPB, 0, st>>>(P, dP, rows, T, drop_p, rng, site);
  RD_CHECK_LAUNCH("attn_softmax_bwd_kernel");
  return 0;
}

int obprop_out_grad(const float* dZ, const float* Z, const float* s, int B, int T, int N, int d_ob, int D,
                    int round, float* dZ2, cudaStream_t st) {
  int64_t total = (int64_t)B * N * T * d_ob;
  const uintptr_t bits = reinterpret_cast<uintptr_t>(dZ) | reinterpret_cast<uintptr_t>(Z) | reinterpret_cast<uintptr_t>(dZ2);
  if (d_ob == 4 && (D & 3) == 0 && (bits & 15) == 0) {
    launch_pdl(obprop_out_grad_vec4_kernel, dim3(blocks_for(total / 4)), dim3(TPB), 0, st, dZ, Z, s, B, T, N, D, round, dZ2);
    RD_CHECK_LAUNCH("obprop_out_grad_vec4_kernel");
    return 0;
  }
  launch_pdl(obprop_out_grad_kernel, dim3(blocks_for(total)), dim3(TPB), 0, st, dZ, Z, s, B, T, N, d_ob, D, round, dZ2);
  RD_CHECK_LAUNCH("obprop_out_grad_kernel");
  return 0;
}

int apply_dropout(const float* x, int64_t n, float p, const uint64_t* rng, uint32_t site, float* y,
                  cudaStream_t st) {
  apply_dropout_kernel<<<blocks_for(n), TPB, 0, st>>>(x, n, p, rng, site, y);
  RD_CHECK_LAUNCH("apply_dropout_kernel");
  return 0;
}

int relu_scale_bwd(const float* d_out, const float* out, const float* scale, int mod, int64_t rows, int C,
                   float* d_pre, cudaStream_t st) {
  relu_scale_bwd_kernel<<<blocks_for(rows * C), TPB, 0, st>>>(d_out, out, scale, mod, rows, C, d_pre);
  RD_CHECK_LAUNCH("relu_scale_bwd_kernel");
  return 0;
}

int cross_entropy(const float* logits, const int64_t* y, int B, int ncls, float* loss, float* dlogits,
                  cudaStream_t st) {
  cross_entropy_kernel<<<1, TPB, 0, st>>>(logits, y, B, ncls, loss, dlogits);
  RD_CHECK_LAUNCH("cross_entropy_kernel");
  return 0;
}

int adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, const float* lr_dev, float b1, float b2,
         float eps, float gscale, int64_t* step, cudaStream_t st) {
  const int vec = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v)) & 15) == 0;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  long long blocks = ceil_div(n, (int64_t)TPB * 4);
  if (blocks > 4LL * sms) blocks = 4LL * sms;
  if (blocks < 1) blocks = 1;
  launch_pdl(adam_kernel, dim3((unsigned)blocks), dim3(TPB), 0, st, p, g, m, v, (long long)n, vec, lr, lr_dev, b1, b2, eps, gscale, step);
  RD_CHECK_LAUNCH("adam_kernel");
  return 0;
}

}  // namespace rd

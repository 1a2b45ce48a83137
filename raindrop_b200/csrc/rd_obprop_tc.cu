// Observation-propagation layer forward on the 5th-gen tensor cores (sm_100a).
//
//   out[r, :] = relu(x[r, :] . W^T + b) * s[r % N]            x: [B*N, C] fp32, W: [C, C] fp32
//
// which is what `Observation_progation` computes on the live path (code/Ob_propagation.py:187-228:
// the message relu(lin_value(x_i)) depends on the target only, so segment-softmax + scatter-add
// collapse to the per-node factor s, see rd_node_scale).  Roofline: 8*C bytes and 2*C^2 flops per
// row -> C/4 flop/B (60 at P19): HBM-bound, so the design goal is to stream x exactly once:
//
//   * persistent CTAs (one per SM), static round-robin over 128-row tiles x n-tiles;
//   * warp 0: TMA producer  - x tile [128 x 32] and W tile [BN x 32] fp32 per k-block into a
//             4-stage 128B-swizzled shared-memory ring (W comes from L2, x from HBM);
//   * warp 1: one elected thread issues tcgen05.mma kind::tf32 (M=128, N=BN<=256, K=8), fp32
//             accumulators in TMEM, double buffered (2 x 256 columns) so the epilogue of tile i
//             overlaps the MMAs of tile i+1;
//   * warps 2-5: epilogue - tcgen05.ld 32 columns at a time, + bias, relu, * s, stage through
//             shared memory and write with TMA bulk stores (coalesced 128 B lines).  For the second
//             layer the result goes straight into the [T, B, D] encoder input
//             (code/models_rd.py:338-341): there a lane's 4 values of one timestamp are 16 contiguous
//             bytes and consecutive lanes are consecutive sensors, so plain st.global.v4 is already
//             a coalesced 512-byte warp store - no staging, no separate permute pass.
// fp32 bits are fed to the tensor core unchanged (TF32 reads the top 19 bits); SURVEY.md section 7
// measured the effect on the logits at 1e-5 normwise.
#include <cuda.h>
#include <stdlib.h>

#include "rd_obprop_tc.cuh"
#include "rd_tc_common.cuh"

namespace rd {
using namespace tc;
namespace {

constexpr int BM = 128;
constexpr int BK = 32;                 // tf32 per k-block: 128 bytes = one swizzle row
constexpr int MAX_STAGES = 4;
constexpr int NTHREADS = 192;                // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue
constexpr int NTHREADS_EXACT = 320;          // + warps 6-9: remainder pass of the error-compensated mode
constexpr int A_STAGE_BYTES = BM * BK * 4;   // 16 KB
constexpr int STG_BYTES = 4096;              // 32 rows x 32 floats per epilogue warp buffer

struct TcParams {
  int M, C, BN, n_tiles, m_tiles, k_blocks, nstages;
  const float* bias;
  const float* scale;
  const float* gate;
  int scale_mod;
  int relu, round_out;
  int perm, pB, pN, pD;
  float* out;
  const float* lift_ru;
  float lift_scale;
};

__device__ __forceinline__ float epi1(float acc, float bias, float sc, int relu, int rnd) {
  float v = acc + bias;
  if (relu) v = fmaxf(v, 0.f);
  v *= sc;
  return rnd ? rn_tf32(v) : v;
}

// PERM / GATE / RELU / ROUND are compile-time so the streaming epilogue carries no runtime branches.
// EXACT: error-compensated products (3xTF32, fp32-level accuracy) for the latency-bound row counts where the
// tensor pipe has slack: the weight tile comes with its precomputed remainder (tmWlo), four extra warps derive the
// activation remainder x - trunc19(x) in shared memory, and every k-step issues lo.hi + hi.lo + hi.hi.
// LIFT_BWD: the input-gradient store of the lift X0 = dropout(relu(v * R_u)): a lane's 4 columns of one timestamp are
// gated by X0 != 0 (relu' and the keep bit at once), weighted by R_u and summed into ONE value of d_src [T, B, 2N];
// consecutive lanes are consecutive sensors, so the warp's stores coalesce.
template <bool PERM, bool GATE, bool RELU, bool ROUND, bool EXACT, bool LIFT_BWD = false>
__global__ void __launch_bounds__(EXACT ? NTHREADS_EXACT : NTHREADS, 1)
obprop_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                 const __grid_constant__ CUtensorMap tmWlo, const __grid_constant__ CUtensorMap tmOut, const TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  pdl_launch_dependents();
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t w_tile = (uint32_t)p.BN * 128u;
  // stage: x hi [| x lo] | W hi [| W lo]
  const uint32_t stage_bytes = EXACT ? 2u * A_STAGE_BYTES + 2u * w_tile : A_STAGE_BYTES + w_tile;
  const uint32_t w_off = EXACT ? 2u * A_STAGE_BYTES : (uint32_t)A_STAGE_BYTES;
  const uint32_t stg_base = base + (uint32_t)p.nstages * stage_bytes;        // 8 x 4 KB staging
  const uint32_t bias_base = stg_base + 8 * STG_BYTES;                        // 2 x 256 floats
  const uint32_t bar_base = bias_base + 2 * 256 * 4;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (MAX_STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * MAX_STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * MAX_STAGES + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * MAX_STAGES + 4);
  auto ready_bar = [&](int s) { return bar_base + 8u * (2 * MAX_STAGES + 6 + s); };     // EXACT: remainders written
  float* bias_s = reinterpret_cast<float*>(smem_raw + (bias_base - smem_u32(smem_raw)));
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmW) : "memory");
    if (EXACT) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmWlo) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmOut) : "memory");
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < MAX_STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); mbar_init(ready_bar(s), 4); }
      for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(tmem_slot) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();
  const uint32_t tmem_base = *tmem_slot_ptr;
  const int total_tiles = p.m_tiles * p.n_tiles;

  if (warp == 0) {
    // ===== TMA producer ==========================================================================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int m_t = tile / p.n_tiles, n_t = tile - m_t * p.n_tiles;
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          mbar_expect_tx(full_bar(stage), EXACT ? A_STAGE_BYTES + 2u * w_tile : stage_bytes);
          const uint32_t sa = base + (uint32_t)stage * stage_bytes;
          tma_load_2d(&tmA, full_bar(stage), sa, kb * BK, m_t * BM);
          tma_load_2d(&tmW, full_bar(stage), sa + w_off, kb * BK, n_t * p.BN);
          if (EXACT) tma_load_2d(&tmWlo, full_bar(stage), sa + w_off + w_tile, kb * BK, n_t * p.BN);
          if (++stage == p.nstages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one thread) ==============================================================
    if (lane == 0) {
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(p.BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * 256u;
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(EXACT ? ready_bar(stage) : full_bar(stage), phase);
          tc_fence_after();
          const uint32_t sa = base + (uint32_t)stage * stage_bytes;
          const uint64_t adesc = umma_desc_sw128(sa), bdesc = umma_desc_sw128(sa + w_off);
          if (EXACT) {
            const uint64_t alo = umma_desc_sw128(sa + A_STAGE_BYTES), blo = umma_desc_sw128(sa + w_off + w_tile);
#pragma unroll
            for (int kk = 0; kk < BK / 8; ++kk) {
              const uint64_t o = (uint64_t)(kk * 2);
              umma_tf32(d_tmem, alo + o, bdesc + o, idesc, (kb | kk) ? 1u : 0u);     // small terms first
              umma_tf32(d_tmem, adesc + o, blo + o, idesc, 1u);
              umma_tf32(d_tmem, adesc + o, bdesc + o, idesc, 1u);
            }
          } else {
#pragma unroll
            for (int kk = 0; kk < BK / 8; ++kk)  // advance 32 bytes (8 tf32) inside the swizzle row
              umma_tf32(d_tmem, adesc + (uint64_t)(kk * 2), bdesc + (uint64_t)(kk * 2), idesc, (kb | kk) ? 1u : 0u);
          }
          umma_commit(empty_bar(stage));  // smem slot reusable once these MMAs have read it
          if (++stage == p.nstages) { stage = 0; phase ^= 1u; }
        }
        umma_commit(tfull_bar(acc));       // accumulator complete -> epilogue
        acc ^= 1; if (acc == 0) acc_phase ^= 1u;
      }
    }
  } else if (EXACT && warp >= 6) {
    // ===== remainder pass (warps 6..9): x_lo = x - trunc19(x), same swizzled addresses =================
    const int lt = threadIdx.x - 192;
    int stage = 0; uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      for (int kb = 0; kb < p.k_blocks; ++kb) {
        mbar_wait(full_bar(stage), phase);
        const uint32_t sa = base + (uint32_t)stage * stage_bytes;
        lo_image<8>(sa, sa + A_STAGE_BYTES, A_STAGE_BYTES / 16, (uint32_t)lt, 128u);
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(ready_bar(stage));
        if (++stage == p.nstages) { stage = 0; phase ^= 1u; }
      }
    }
  } else {
    // ===== epilogue warps 2..5: TMEM -> registers -> smem -> TMA store ===========================
    const int q = warp & 3;               // TMEM lane quarter this warp may access
    const int et = threadIdx.x - 64;      // 0..127
    const uint32_t my_stg = stg_base + (uint32_t)(warp - 2) * 2u * STG_BYTES;
    int acc = 0; uint32_t acc_phase = 0; int buf = 0;
    const int n_chunks = (p.BN + 31) / 32;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int m_t = tile / p.n_tiles, n_t = tile - m_t * p.n_tiles;
      const int col0 = n_t * p.BN;
      for (int c = et; c < 256; c += 128) bias_s[acc * 256 + c] = (p.bias && c < p.BN && col0 + c < p.C) ? __ldg(p.bias + col0 + c) : 0.f;
      asm volatile("bar.sync 1, 128;" ::: "memory");
      const int row0 = m_t * BM + q * 32;
      const int row = row0 + lane;
      const float sc = (!LIFT_BWD && row < p.M) ? __ldg(p.scale + (row % p.scale_mod)) : 0.f;
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
      float* lift_row = nullptr;
      float4 ru = make_float4(0.f, 0.f, 0.f, 0.f);
      if (LIFT_BWD && row < p.M) {
        const int b = row / p.pN, n = row - b * p.pN;
        lift_row = p.out + (size_t)b * p.pD + n;
        ru = __ldg(reinterpret_cast<const float4*>(p.lift_ru) + n);
      }
      // perm: this lane's row is sensor n of sample b; its 4 values of one timestamp are 16
      // contiguous bytes of out[t, b, n*4 .. n*4+3] and consecutive lanes are consecutive sensors,
      // so one st.global.v4 per timestamp is a fully coalesced 512-byte warp store (no staging).
      float* perm_row = nullptr;
      if (PERM && row < p.M) {
        const int b = row / p.pN, n = row - b * p.pN;
        perm_row = p.out + (size_t)b * p.pD + (size_t)n * 4;
      }
      for (int ch = 0; ch < n_chunks; ++ch) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * 256 + ch * 32), v);
        const float* bs = bias_s + acc * 256 + ch * 32;
        const int c0 = col0 + ch * 32;
        if (LIFT_BWD) {
          if (lift_row) {
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              const int t = (c0 >> 2) + j4;
              if (4 * t < p.C && ch * 32 + 4 * j4 < p.BN) {
                const float4 g = __ldg(reinterpret_cast<const float4*>(p.gate + (size_t)row * p.C + 4 * t));
                float s = g.x != 0.f ? __uint_as_float(v[4 * j4 + 0]) * ru.x : 0.f;
                s += g.y != 0.f ? __uint_as_float(v[4 * j4 + 1]) * ru.y : 0.f;
                s += g.z != 0.f ? __uint_as_float(v[4 * j4 + 2]) * ru.z : 0.f;
                s += g.w != 0.f ? __uint_as_float(v[4 * j4 + 3]) * ru.w : 0.f;
                lift_row[(size_t)t * p.pB * p.pD] = s * p.lift_scale;
              }
            }
          }
          continue;
        }
        if (PERM) {
          if (perm_row) {
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              const int t = (c0 >> 2) + j4;
              if (4 * t < p.C && ch * 32 + 4 * j4 < p.BN) {
                float4 o;
                o.x = epi1(__uint_as_float(v[4 * j4 + 0]), bs[4 * j4 + 0], sc, RELU, ROUND);
                o.y = epi1(__uint_as_float(v[4 * j4 + 1]), bs[4 * j4 + 1], sc, RELU, ROUND);
                o.z = epi1(__uint_as_float(v[4 * j4 + 2]), bs[4 * j4 + 2], sc, RELU, ROUND);
                o.w = epi1(__uint_as_float(v[4 * j4 + 3]), bs[4 * j4 + 3], sc, RELU, ROUND);
                *reinterpret_cast<float4*>(perm_row + (size_t)t * p.pB * p.pD) = o;
              }
            }
          }
          continue;
        }
        if (lane == 0) bulk_wait_read<1>();   // the store that used this staging buffer has drained
        __syncwarp();
        const uint32_t stg = my_stg + (uint32_t)buf * STG_BYTES;
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          float4 o;
          o.x = epi1(__uint_as_float(v[4 * j4 + 0]), bs[4 * j4 + 0], sc, RELU, ROUND);
          o.y = epi1(__uint_as_float(v[4 * j4 + 1]), bs[4 * j4 + 1], sc, RELU, ROUND);
          o.z = epi1(__uint_as_float(v[4 * j4 + 2]), bs[4 * j4 + 2], sc, RELU, ROUND);
          o.w = epi1(__uint_as_float(v[4 * j4 + 3]), bs[4 * j4 + 3], sc, RELU, ROUND);
          if (GATE) {   // backward: pass the gradient only where the forward output was positive
            float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
            if (row < p.M && c0 + 4 * j4 < p.C) g = __ldg(reinterpret_cast<const float4*>(p.gate + (size_t)row * p.C + c0 + 4 * j4));
            o.x = g.x > 0.f ? o.x : 0.f; o.y = g.y > 0.f ? o.y : 0.f; o.z = g.z > 0.f ? o.z : 0.f; o.w = g.w > 0.f ? o.w : 0.f;
          }
          // [32 rows][128 B] with the 128B swizzle the tensor map expects
          const uint32_t off = (uint32_t)(lane * 128 + ((j4 ^ (lane & 7)) << 4));
          asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(stg + off), "f"(o.x), "f"(o.y), "f"(o.z), "f"(o.w) : "memory");
        }
        fence_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&tmOut, stg, c0, row0);
          bulk_commit();
        }
        buf ^= 1;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
      acc ^= 1; if (acc == 0) acc_phase ^= 1u;
    }
    if (lane == 0) bulk_wait_read<0>();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
  }
}

// max_bn: widest n-tile (256 for the single-pass kernel; the error-compensated kernel carries two images of both
// operands per stage and takes 128 so that >= 2 stages still fit)
void plan_n(int C, int max_bn, int* BN, int* n_tiles) {
  if (C <= max_bn) { *n_tiles = 1; *BN = (int)round_up(C, 16); return; }
  int best_bn = max_bn, best_nt = (int)ceil_div(C, max_bn), best_pad = best_nt * max_bn;
  for (int bn = max_bn; bn >= max_bn / 2; bn -= 32) {   // multi-tile: BN % 32 == 0 so no epilogue chunk straddles tiles
    int nt = (int)ceil_div(C, bn);
    if (nt * bn < best_pad) { best_pad = nt * bn; best_bn = bn; best_nt = nt; }
  }
  *BN = best_bn; *n_tiles = best_nt;
}

}  // namespace

bool obprop_tc_supported(int C) {
  static int env = -1;
  if (env < 0) { const char* e = getenv("RD_OBPROP_TC"); env = (e && e[0] == '0') ? 0 : 1; }
  return env == 1 && C % 4 == 0 && C >= 16;
}

bool obprop_tc_exact(int64_t rows, int C, int mode) {
  static int env = -1;
  if (env < 0) { const char* e = getenv("RD_OBPROP_EXACT"); env = e ? (e[0] == '0' ? 1 : 2) : 0; }
  if (mode == 0) mode = env;
  if (mode == 1) return false;
  if (mode == 2) return true;
  return 2.0 * (double)rows * C * C <= 2.0e9;
}

__global__ void round_tf32_kernel(const float* __restrict__ x, long long n, float* __restrict__ y) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x[i]));
    y[i] = __uint_as_float(r);
  }
}

int round_tf32(const float* x, int64_t n, float* y, cudaStream_t st) {
  if (n <= 0) return 0;
  round_tf32_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(x, n, y);
  RD_CHECK_LAUNCH("round_tf32_kernel");
  return 0;
}

int obprop_tc_fwd(const ObpropTcArgs& a, cudaStream_t st) {
  const float* x = a.x; const float* W = a.W; float* out = a.out;
  const int64_t rows = a.rows; const int C = a.C; const int perm = a.perm, pB = a.pB, pN = a.pN, pdob = a.pdob, pD = a.pD;
  if (perm && pdob != 4) { set_error("obprop_tc_fwd: permuted store needs d_ob == 4"); return -2; }
  if (perm && a.gate) { set_error("obprop_tc_fwd: gate is only built for the plain layout"); return -2; }
  const bool lift = a.lift_ru != nullptr;
  if (lift && (perm || !a.gate || !a.W_lo || a.bias || a.relu || a.round_out || pdob != 4 ||
               (reinterpret_cast<uintptr_t>(a.lift_ru) & 15))) {
    set_error("obprop_tc_fwd: the lift-backward store needs d_ob == 4, the X0 gate, the error-compensated mode, no "
              "bias / relu / rounding and a 16-byte aligned R_u");
    return -2;
  }
  if (rows > 0x7fffffffLL) { set_error("obprop_tc_fwd: too many rows"); return -2; }
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(W) | reinterpret_cast<uintptr_t>(out) |
       reinterpret_cast<uintptr_t>(a.gate)) & 15) {
    set_error("obprop_tc_fwd: pointers must be 16-byte aligned");
    return -2;
  }
  const bool exact = a.W_lo != nullptr;
  if (exact && (reinterpret_cast<uintptr_t>(a.W_lo) & 15)) { set_error("obprop_tc_fwd: W_lo must be 16-byte aligned"); return -2; }
  TcParams p;
  p.M = (int)rows; p.C = C;
  plan_n(C, exact ? 128 : 256, &p.BN, &p.n_tiles);     // exact: 3x the MMAs per tile -> narrower tiles, more CTAs
  p.m_tiles = (int)ceil_div(rows, BM);
  p.k_blocks = (int)ceil_div(C, BK);
  const int stage_bytes = exact ? 2 * A_STAGE_BYTES + 2 * p.BN * 128 : A_STAGE_BYTES + p.BN * 128;
  const int fixed = 1024 + 8 * STG_BYTES + 2 * 256 * 4 + 256;
  p.nstages = (SMEM_LIMIT - fixed) / stage_bytes;
  if (p.nstages > MAX_STAGES) p.nstages = MAX_STAGES;
  if (p.nstages < 2) { set_error("obprop_tc_fwd: not enough shared memory"); return -2; }
  const int smem_bytes = fixed + p.nstages * stage_bytes;
  p.bias = a.bias; p.scale = a.scale; p.scale_mod = a.scale_mod; p.gate = a.gate;
  p.relu = a.relu; p.round_out = a.round_out;
  p.perm = perm; p.pB = pB; p.pN = pN; p.pD = pD; p.out = out;
  p.lift_ru = a.lift_ru; p.lift_scale = a.lift_scale;

  CUtensorMap tmA, tmW, tmWlo, tmOut;
  {
    cuuint64_t dims[2] = {(cuuint64_t)C, (cuuint64_t)rows};
    cuuint64_t str[1] = {(cuuint64_t)C * 4};
    cuuint32_t box[2] = {BK, BM};
    RD_TRY(encode(&tmA, x, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B, "x"));
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)C, (cuuint64_t)C};
    cuuint64_t str[1] = {(cuuint64_t)C * 4};
    cuuint32_t box[2] = {BK, (cuuint32_t)p.BN};
    RD_TRY(encode(&tmW, W, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B, "W"));
    if (exact) RD_TRY(encode(&tmWlo, a.W_lo, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B, "W_lo"));
    else tmWlo = tmW;
  }
  if (!perm && !lift) {
    cuuint64_t dims[2] = {(cuuint64_t)C, (cuuint64_t)rows};
    cuuint64_t str[1] = {(cuuint64_t)C * 4};
    cuuint32_t box[2] = {32, 32};
    RD_TRY(encode(&tmOut, out, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B, "out"));
  } else {
    tmOut = tmA;   // permuted / lift-backward output is written with plain stores; the map is not used
  }
  int total = p.m_tiles * p.n_tiles;
  int grid = total < num_sms() ? total : num_sms();
  auto launch = [&](auto kern, int nthreads) -> int {
    RD_TRY(ensure_max_smem((const void*)kern, SMEM_LIMIT));   // once per (instantiation, device)
    launch_pdl(kern, dim3(grid), dim3(nthreads), smem_bytes, st, tmA, tmW, tmWlo, tmOut, p);
    return 0;
  };
  int rc;
  const bool relu = a.relu != 0, rnd = a.round_out != 0;
  if (!exact) {
    if (perm && !a.gate && relu && !rnd) rc = launch(obprop_tc_kernel<true, false, true, false, false>, NTHREADS);        // layer 2 -> encoder input
    else if (!perm && !a.gate && relu && rnd) rc = launch(obprop_tc_kernel<false, false, true, true, false>, NTHREADS);   // layer 1
    else if (!perm && !a.gate && relu && !rnd) rc = launch(obprop_tc_kernel<false, false, true, false, false>, NTHREADS); // operator
    else if (!perm && a.gate && !relu && !rnd) rc = launch(obprop_tc_kernel<false, true, false, false, false>, NTHREADS); // backward d(input)
    else { set_error("obprop_tc_fwd: epilogue combination not instantiated"); return -2; }
  } else {
    if (rnd) { set_error("obprop_tc_fwd: the error-compensated mode does not round its output"); return -2; }
    if (lift) rc = launch(obprop_tc_kernel<false, true, false, false, true, true>, NTHREADS_EXACT);         // backward d(src)
    else if (perm && !a.gate && relu) rc = launch(obprop_tc_kernel<true, false, true, false, true>, NTHREADS_EXACT);
    else if (!perm && !a.gate && relu) rc = launch(obprop_tc_kernel<false, false, true, false, true>, NTHREADS_EXACT);
    else if (!perm && a.gate && !relu) rc = launch(obprop_tc_kernel<false, true, false, false, true>, NTHREADS_EXACT);
    else { set_error("obprop_tc_fwd: epilogue combination not instantiated"); return -2; }
  }
  if (rc != 0) return rc;
  RD_CHECK_LAUNCH("obprop_tc_kernel");
  return 0;
}

}  // namespace rd

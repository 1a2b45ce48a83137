// Host-side orchestration of the Raindrop_v2 hot path and the C ABI (include/raindrop_b200.h).
//
// Data layout in HBM (all fp32, row-major, 256-byte aligned sub-buffers of one caller-provided
// workspace so that nothing is allocated between forward and backward):
//   X0, H1          [B*N, C]   sensor-major rows, C = T*d_ob  (observation propagation operands)
//   Z[l]            [T, B, D]  encoder layer inputs/outputs, seq-first exactly like the reference
//   qkv, ctx, r1, x1, f, r2    per encoder layer, token-major [T*B, .]
//   P (and Pd)      [B, H, T, T] attention probabilities (and their dropped copy when training)
#include <math.h>
#include <string.h>

#include "rd_kernels.cuh"
#include "rd_obprop_tc.cuh"
#include "rd_tc_gemm.cuh"

namespace rd {
namespace {

struct Shape {
  int B, T, N, dob, H, nhid, L, ds, ncls;
  int C, Dm, D, Df, hd, dpe, emb;
  int64_t M1, M2;
  float p;  // effective dropout probability (0 in eval)
  int tc, exact;   // ob-prop layers: tensor-core kernel usable / error-compensated (3xTF32) mode chosen
};

int make_shape(const rd_dims* d, Shape* s) {
  if (!d) { set_error("dims is NULL"); return -2; }
  s->B = d->B; s->T = d->T; s->N = d->N; s->dob = d->d_ob; s->H = d->nhead; s->nhid = d->nhid;
  s->L = d->nlayers; s->ds = d->d_static; s->ncls = d->n_classes;
  if (s->B < 1 || s->T < 1 || s->N < 1 || s->dob < 1 || s->H < 1 || s->nhid < 1 || s->L < 1 ||
      s->L > RD_MAX_LAYERS || s->ncls < 1 || s->ds < 0) {
    set_error("invalid dims (B=%d T=%d N=%d d_ob=%d nhead=%d nhid=%d nlayers=%d d_static=%d n_classes=%d)",
              s->B, s->T, s->N, s->dob, s->H, s->nhid, s->L, s->ds, s->ncls);
    return -2;
  }
  s->dpe = d->d_pe > 0 ? d->d_pe : RD_D_PE;
  s->emb = d->emb_dim > 0 ? d->emb_dim : s->N;
  if (s->dpe > 64 || (s->dpe & 3)) { set_error("d_pe = %d must be a multiple of 4 and <= 64", s->dpe); return -2; }
  s->C = s->T * s->dob; s->Dm = s->N * s->dob; s->D = s->Dm + s->dpe;
  if (s->D % s->H != 0) { set_error("d_model+16 = %d not divisible by nhead = %d", s->D, s->H); return -2; }
  s->hd = s->D / s->H;
  s->Df = s->D + (s->ds > 0 ? s->emb : 0);
  s->M1 = (int64_t)s->B * s->N; s->M2 = (int64_t)s->T * s->B;
  s->p = (d->training && d->dropout_p > 0.f) ? d->dropout_p : 0.f;
  if (s->p >= 1.f) { set_error("dropout_p must be < 1"); return -2; }
  if (d->obprop_mode < 0 || d->obprop_mode > 2) { set_error("obprop_mode must be 0 (auto), 1 (tf32) or 2 (3xtf32)"); return -2; }
  s->tc = obprop_tc_supported(s->C) ? 1 : 0;
  s->exact = (s->tc && obprop_tc_exact(s->M1, s->C, d->obprop_mode)) ? 1 : 0;
  return 0;
}

struct Arena {
  int64_t off = 0;  // floats
  int64_t take(int64_t n) { int64_t o = off; off += round_up(n > 0 ? n : 1, 64); return o; }
};

struct WsLayout {
  int64_t rng, cnt, loss_ps, X0, H1, W1r, W2r, W2t, W1lo, W2lo, W2tlo, Z[RD_MAX_LAYERS + 1], feat, hpre, total;
  struct { int64_t qkv, P, Pd, ctx, r1, st1, x1, f, r2, st2, m1, m2; } l[RD_MAX_LAYERS];   // m1, m2: dropout keep bits of r1, r2
  // error-compensation remainders and transposes of the encoder weights (rd_tc_gemm.cuh)
  struct { int64_t in_lo, in_t, in_tlo, out_lo, out_t, out_tlo, l1_lo, l1_t, l1_tlo, l2_lo, l2_t, l2_tlo; } wsp[RD_MAX_LAYERS];
};

WsLayout ws_layout(const Shape& s) {
  WsLayout w;
  Arena a;
  w.rng = a.take(4);
  w.cnt = a.take(64);                   // ticket word of the fused loss reduction (zeroed by the step prologue)
  w.loss_ps = a.take(s.B);              // per-sample cross-entropy terms
  w.X0 = a.take(s.M1 * s.C);
  w.H1 = a.take(s.M1 * s.C);
  w.W1r = a.take((int64_t)s.C * s.C);   // TF32-rounded copies of the two lin_value weights
  w.W2r = a.take((int64_t)s.C * s.C);
  w.W2t = a.take((int64_t)s.C * s.C);   // (rounded) W2^T for the backward d(input) GEMM
  const int64_t nlo = s.exact ? (int64_t)s.C * s.C : 0;     // error-compensated mode: remainders of W1, W2, W2^T
  w.W1lo = a.take(nlo); w.W2lo = a.take(nlo); w.W2tlo = a.take(nlo);
  for (int i = 0; i <= s.L; ++i) w.Z[i] = a.take(s.M2 * s.D);
  // the T x T probabilities only reach HBM on the long-sequence path (the fused short-sequence kernels
  // keep them in shared memory and recompute them in backward)
  const int64_t pp = attn_small_supported(s.T, s.hd) ? 0 : (int64_t)s.B * s.H * s.T * s.T;
  for (int i = 0; i < s.L; ++i) {
    w.l[i].qkv = a.take(s.M2 * 3 * s.D);
    w.l[i].P = a.take(pp);
    w.l[i].Pd = a.take(s.p > 0.f ? pp : 0);
    w.l[i].ctx = a.take(s.M2 * s.D);
    w.l[i].r1 = a.take(s.M2 * s.D);
    w.l[i].st1 = a.take(s.M2 * 2);
    w.l[i].x1 = a.take(s.M2 * s.D);
    w.l[i].f = a.take(s.M2 * s.nhid);
    w.l[i].r2 = a.take(s.M2 * s.D);
    w.l[i].st2 = a.take(s.M2 * 2);
    const int64_t mw = s.p > 0.f ? s.M2 * ((s.D + 31) / 32) : 0;     // one 32-bit word per 32 columns
    w.l[i].m1 = a.take(mw); w.l[i].m2 = a.take(mw);
    const int64_t nin = 3LL * s.D * s.D, nout = (int64_t)s.D * s.D, nff = (int64_t)s.nhid * s.D;
    w.wsp[i].in_lo = a.take(nin); w.wsp[i].in_t = a.take(nin); w.wsp[i].in_tlo = a.take(nin);
    w.wsp[i].out_lo = a.take(nout); w.wsp[i].out_t = a.take(nout); w.wsp[i].out_tlo = a.take(nout);
    w.wsp[i].l1_lo = a.take(nff); w.wsp[i].l1_t = a.take(nff); w.wsp[i].l1_tlo = a.take(nff);
    w.wsp[i].l2_lo = a.take(nff); w.wsp[i].l2_t = a.take(nff); w.wsp[i].l2_tlo = a.take(nff);
  }
  w.feat = a.take((int64_t)s.B * s.Df);
  w.hpre = a.take((int64_t)s.B * s.Df);
  w.total = a.off;
  return w;
}

// Backward scratch.  The weight gradients are DEFERRED: every linear layer's (dY, X) operand pair stays alive in
// its own buffer until one grouped tensor-core launch (tc_wgrad_group) reduces them all, so dY buffers and the
// split-K partial buffers are per layer / per problem instead of ping-pong.
struct BwLayout {
  int64_t dfeat, dhpre, gA, gB, gD, dP, gO2, gO1, partial, total;
  struct { int64_t K2, gF, K1, dqkv, wp[4], ln[2]; } l[RD_MAX_LAYERS];   // wp: linear2, linear1, out_proj, in_proj partials; ln: norm2, norm1
  int64_t wp_ob[2];
  int64_t partial_floats;
};

// Input-gradient scratch (rd_input_grad_scratch_bytes).  The lift backward dX0 = gO1 . W1 runs on the ob-prop tensor-core
// kernel against W1^T and its remainder, derived in the backward (the forward cannot know whether input gradients will
// be asked for); shapes that kernel does not take go through the CUDA-core GEMM into dX0.
struct InLayout { int64_t W1t, W1tlo, dX0, total; };

bool lift_bwd_tc(const Shape& s) { return s.tc && s.dob == 4; }

InLayout in_layout(const Shape& s) {
  InLayout l;
  Arena a;
  const int64_t cc = lift_bwd_tc(s) ? (int64_t)s.C * s.C : 0;
  l.W1t = a.take(cc);
  l.W1tlo = a.take(cc);
  l.dX0 = a.take(lift_bwd_tc(s) ? 0 : s.M1 * s.C);
  l.total = a.off;
  return l;
}

int64_t splitk_partial_floats(int Nout, int Kin, int64_t rows) {
  int ns;
  return gemm_splitk_plan(Nout, Kin, (int)rows, &ns);
}

BwLayout bw_layout(const Shape& s) {
  BwLayout b;
  Arena a;
  b.dfeat = a.take((int64_t)s.B * s.Df);
  b.dhpre = a.take((int64_t)s.B * s.Df);
  b.gA = a.take(s.M2 * s.D);
  b.gB = a.take(s.M2 * s.D);
  b.gD = a.take(s.M2 * s.D);
  b.dP = a.take(attn_small_supported(s.T, s.hd) ? 0 : (int64_t)s.B * s.H * s.T * s.T);
  for (int l = 0; l < s.L; ++l) {
    b.l[l].K2 = a.take(s.M2 * s.D);
    b.l[l].gF = a.take(s.M2 * s.nhid);
    b.l[l].K1 = a.take(s.M2 * s.D);
    b.l[l].dqkv = a.take(s.M2 * 3 * s.D);
    b.l[l].wp[0] = a.take(tc_wgrad_partial_floats(s.D, s.nhid, s.M2));
    b.l[l].wp[1] = a.take(tc_wgrad_partial_floats(s.nhid, s.D, s.M2));
    b.l[l].wp[2] = a.take(tc_wgrad_partial_floats(s.D, s.D, s.M2));
    b.l[l].wp[3] = a.take(tc_wgrad_partial_floats(3 * s.D, s.D, s.M2));
    b.l[l].ln[0] = a.take(ln_bwd_scratch_floats(s.M2, s.D));      // per-CTA dgamma/dbeta partial rows, reduced with the group
    b.l[l].ln[1] = a.take(ln_bwd_scratch_floats(s.M2, s.D));
  }
  b.gO2 = a.take(s.M1 * s.C);
  b.gO1 = a.take(s.M1 * s.C);
  b.wp_ob[0] = a.take(tc_wgrad_partial_floats(s.C, s.C, s.M1));
  b.wp_ob[1] = a.take(tc_wgrad_partial_floats(s.C, s.C, s.M1));
  // shared split-K scratch of the CUDA-core fallback (shapes the tensor-core kernel does not take)
  int64_t pf = 0;
  auto upd = [&](int no, int ki, int64_t rows) { int64_t v = splitk_partial_floats(no, ki, rows); if (v > pf) pf = v; };
  upd(s.C, s.C, s.M1);
  upd(3 * s.D, s.D, s.M2); upd(s.D, s.D, s.M2); upd(s.nhid, s.D, s.M2); upd(s.D, s.nhid, s.M2);
  b.partial_floats = pf;
  b.partial = a.take(pf);
  b.total = a.off;
  return b;
}

// Y[M,N] = epi(X[M,K] . W[N,K]^T)
GemmP nt(const float* X, int64_t ldx, const float* W, int64_t ldw, float* Y, int64_t ldy, int64_t M, int N, int K) {
  GemmP g;
  g.A = X; g.ta = 0; g.sAi = ldx; g.sAk = 1;
  g.B = W; g.tb = 1; g.sBj = ldw; g.sBk = 1;
  g.C = Y; g.sCi = ldy; g.sCj = 1;
  g.M = (int)M; g.N = N; g.K = K;
  return g;
}
// dX[M,Kin] = epi(dY[M,Nout] . W[Nout,Kin])
GemmP nn(const float* dY, int64_t ldy, const float* W, int64_t ldw, float* dX, int64_t ldx, int64_t M, int Kin, int Nout) {
  GemmP g;
  g.A = dY; g.ta = 0; g.sAi = ldy; g.sAk = 1;
  g.B = W; g.tb = 0; g.sBk = ldw; g.sBj = 1;
  g.C = dX; g.sCi = ldx; g.sCj = 1;
  g.M = (int)M; g.N = Kin; g.K = Nout;
  return g;
}
// dW[Nout,Kin] = sum_r dY[r,Nout]^T X[r,Kin], db = sum_r dY[r,:]: queued for the next grouped tensor-core launch when
// the shape fits, else done right away on the CUDA cores (split over rows, deterministic two-stage reduce).
struct WgradQueue {
  WgradItem it[WG_MAX];
  ColsumItem cs[CS_MAX];
  int n = 0, ncs = 0;
  int flush(cudaStream_t st) {
    if (n == 0 && ncs == 0) return 0;
    int rc = tc_wgrad_group(it, n, cs, ncs, st);
    n = 0; ncs = 0;
    return rc;
  }
  // out[c] = sum over the chunks of partial[chunk*stride + c]: reduced by the group's reduction launch
  int colsum(const float* partial, long long stride, int nsplit, int ncols, float* out, cudaStream_t st) {
    if (ncs == CS_MAX) RD_TRY(flush(st));
    cs[ncs++] = ColsumItem{partial, stride, nsplit, ncols, out};
    return 0;
  }
};

int tn(WgradQueue* q, const float* dY, int64_t ldy, const float* X, int64_t ldx, float* dW, float* db, int Nout, int Kin,
       int64_t rows, float* tc_partial, float* partial, cudaStream_t st) {
  if (rows >= 256 && tc_partial && tc_wgrad_supported(Nout, Kin, ldy, ldx, dY, X)) {
    if (q) {
      if (q->n == WG_MAX) RD_TRY(q->flush(st));
      q->it[q->n++] = WgradItem{dY, ldy, X, ldx, rows, Nout, Kin, dW, db, tc_partial};
      return 0;
    }
    return tc_wgrad(dY, ldy, X, ldx, rows, Nout, Kin, dW, db, tc_partial, st);
  }
  GemmP g;
  g.A = dY; g.ta = 1; g.sAk = ldy; g.sAi = 1;
  g.B = X; g.tb = 0; g.sBk = ldx; g.sBj = 1;
  g.C = dW; g.sCi = Kin; g.sCj = 1;
  g.M = Nout; g.N = Kin; g.K = (int)rows;
  int ns;
  gemm_splitk_plan(Nout, Kin, (int)rows, &ns);
  g.nsplit = ns; g.partial = partial;
  g.asum = db;   // db[n] = sum_r dY[r, n] comes out of the same pass
  return gemm(g, st);
}

}  // namespace

// Y[M,N] = epi(X[M,K] . W[N,K]^T): error-compensated tensor-core GEMM when the shape allows it, else CUDA cores.
static int linear_nt(const GemmP& g, const float* W_lo, cudaStream_t st) {
  TcGemmArgs a;
  a.A = g.A; a.lda = g.sAi; a.B = g.B; a.B_lo = W_lo; a.M = g.M; a.N = g.N; a.K = g.K; a.C = g.C;
  a.bias = g.bias; a.relu = g.relu; a.gate = g.gate; a.gate_ld = g.gate_ld; a.gate_scale = g.gate_scale;
  a.drop_p = g.drop_p; a.rng = g.rng; a.drop_site = g.drop_site; a.resid = g.resid; a.resid_ld = g.resid_ld;
  a.drop_mask = g.drop_mask; a.drop_mask_ld = g.drop_mask_ld;
  const bool plain = g.ta == 0 && g.tb == 1 && g.sBj == g.K && g.sCi == g.N && g.sCj == 1 && g.nz == 1 && g.nsplit == 1 &&
                     g.alpha == 1.f && !g.rowscale && !g.perm && !g.asum;
  if (plain && W_lo && tc_gemm_supported(a)) return tc_gemm(a, st);
  return gemm(g, st);
}

// The predicate of linear_nt for a plain y = x W^T GEMM: the backward calls it with the forward's operands to know
// whether the forward's epilogue stored the dropout keep bits (only the tensor-core kernel does).
static bool linear_nt_is_tc(const GemmP& g, const float* W_lo) {
  TcGemmArgs a;
  a.A = g.A; a.lda = g.sAi; a.B = g.B; a.B_lo = W_lo; a.M = g.M; a.N = g.N; a.K = g.K; a.C = g.C;
  a.bias = g.bias; a.relu = g.relu; a.gate = g.gate; a.gate_ld = g.gate_ld; a.gate_scale = g.gate_scale;
  a.drop_p = g.drop_p; a.rng = g.rng; a.drop_site = g.drop_site; a.resid = g.resid; a.resid_ld = g.resid_ld;
  return W_lo && tc_gemm_supported(a);
}

// ---- observation propagation layer (operator level) ---------------------------------------------
// Forward goes to the tcgen05 kernel when the shape fits its tiling, otherwise to the generic
// CUDA-core GEMM (same epilogue).
static int obprop_forward(const ObpropTcArgs& a, cudaStream_t st) {
  if (obprop_tc_supported(a.C) && (!a.perm || a.pdob == 4)) return obprop_tc_fwd(a, st);
  GemmP g = nt(a.x, a.C, a.W, a.C, a.out, a.C, a.rows, a.C, a.C);
  g.bias = a.bias; g.relu = a.relu; g.rowscale = a.scale; g.rowscale_mod = a.scale_mod;
  g.gate = a.gate; g.gate_ld = a.C;
  g.perm = a.perm; g.pB = a.pB; g.pN = a.pN; g.pdob = a.pdob; g.pD = a.pD;
  return gemm(g, st);
}

static int raindrop_fwd(const rd_dims* dims, const rd_params* P, const float* src, const float* statics,
                        const float* times, const int64_t* lengths, const float* nscale, uint64_t* rng_state,
                        float* ws, float* logits, const int64_t* y, float* loss, float* d_logits, int encoder_only,
                        cudaStream_t st) {
  Shape s;
  RD_TRY(make_shape(dims, &s));
  if (!encoder_only && (s.dpe != RD_D_PE || s.emb != s.N)) { set_error("Raindrop_v2 has d_pe = 16 and emb_dim = d_inp"); return -2; }
  if (encoder_only) { s.tc = 0; s.exact = 0; }      // no observation propagation on this entry: no lin_value copies
  if (s.ds > 0 && (!statics || !P->emb_weight || !P->emb_bias)) { set_error("static branch needs statics/emb"); return -2; }
  WsLayout w = ws_layout(s);
  uint64_t* rng = reinterpret_cast<uint64_t*>(ws + w.rng);
  if (s.p > 0.f && !rng_state) { set_error("training with dropout needs rng_state"); return -2; }
  if (y && (!loss || !d_logits)) { set_error("labels given without loss / d_logits outputs"); return -2; }
  // rides along with the first weight-prep launch: dropout-stream capture (+ advance) and the loss ticket reset
  StepPrologue pro;
  if (s.p > 0.f) { pro.rng_state = rng_state; pro.rng_captured = rng; pro.advance = 1; }
  pro.zero_counter = reinterpret_cast<unsigned*>(ws + w.cnt);
  float* X0 = ws + w.X0; float* H1 = ws + w.H1;
  // Fast mode: tensor-core operands are kept exactly TF32-representable by their producers (lift, layer-1 epilogue,
  // rounded weight copies) so the MMA's operand truncation is exact.  Error-compensated mode (latency-bound row
  // counts): operands stay fp32, the weights come with their remainders, nothing is rounded.
  const int tc = s.tc, exact = s.exact;
  const float* W1 = P->ob1_value_weight; const float* W2 = P->ob2_value_weight;
  if (tc && !exact) { W1 = ws + w.W1r; W2 = ws + w.W2r; }   // rounded copies, produced by the weight-prep launch just below
  for (int l0 = 0; l0 < s.L; l0 += 3) {   // every derived weight tensor of the step in one launch (<= 16 tensors each)
    WeightSplit items[16];
    int n = 0;
    if (l0 == 0 && tc && !exact) {
      items[n] = {P->ob1_value_weight, s.C, s.C, nullptr, nullptr, nullptr}; items[n++].rn = ws + w.W1r;
      items[n] = {P->ob2_value_weight, s.C, s.C, nullptr, nullptr, nullptr}; items[n].rn = ws + w.W2r; items[n++].rn_t = ws + w.W2t;
    }
    if (l0 == 0 && exact) {
      items[n++] = {P->ob1_value_weight, s.C, s.C, ws + w.W1lo, nullptr, nullptr};
      items[n++] = {P->ob2_value_weight, s.C, s.C, ws + w.W2lo, ws + w.W2t, ws + w.W2tlo};
    }
    for (int l = l0; l < s.L && l < l0 + 3; ++l) {
      const rd_encoder_layer_params& E = P->layer[l];
      items[n++] = {E.in_proj_weight, 3 * s.D, s.D, ws + w.wsp[l].in_lo, ws + w.wsp[l].in_t, ws + w.wsp[l].in_tlo};
      items[n++] = {E.out_proj_weight, s.D, s.D, ws + w.wsp[l].out_lo, ws + w.wsp[l].out_t, ws + w.wsp[l].out_tlo};
      items[n++] = {E.linear1_weight, s.nhid, s.D, ws + w.wsp[l].l1_lo, ws + w.wsp[l].l1_t, ws + w.wsp[l].l1_tlo};
      items[n++] = {E.linear2_weight, s.D, s.nhid, ws + w.wsp[l].l2_lo, ws + w.wsp[l].l2_t, ws + w.wsp[l].l2_tlo};
    }
    RD_TRY(split_weights(items, n, st, l0 == 0 ? &pro : nullptr));
  }
  float* Z0 = ws + w.Z[0];
  if (!encoder_only) {
  // lift of the raw observations and the positional encoding (written into Z0[..., 4N:]) in one launch
  RD_TRY(lift_posenc(src, P->R_u, s.B, s.T, s.N, s.dob, s.p, rng, tc && !exact, X0, times, s.M2, dims->pe_timescales, RD_D_PE, Z0,
                     s.D, s.Dm, st));
  {
    ObpropTcArgs a;
    a.x = X0; a.W = W1; a.bias = P->ob1_value_bias; a.scale = nscale; a.scale_mod = s.N;
    a.rows = s.M1; a.C = s.C; a.out = H1; a.round_out = tc && !exact;
    a.W_lo = exact ? ws + w.W1lo : nullptr;
    RD_TRY(obprop_forward(a, st));
    a.x = H1; a.W = W2; a.bias = P->ob2_value_bias; a.out = Z0; a.round_out = 0;
    a.W_lo = exact ? ws + w.W2lo : nullptr;
    a.perm = 1; a.pB = s.B; a.pN = s.N; a.pdob = s.dob; a.pD = s.D;
    RD_TRY(obprop_forward(a, st));
  }
  }

  const float scale = 1.f / sqrtf((float)s.hd);
  const int64_t row3 = (int64_t)s.B * 3 * s.D;
  const int64_t TT = (int64_t)s.T * s.T;
  for (int l = 0; l < s.L; ++l) {
    const rd_encoder_layer_params& E = P->layer[l];
    float* x = ws + w.Z[l];
    float* qkv = ws + w.l[l].qkv;
    float* Pm = ws + w.l[l].P;
    float* Pd = s.p > 0.f ? ws + w.l[l].Pd : nullptr;
    {
      GemmP g = nt(x, s.D, E.in_proj_weight, s.D, qkv, 3 * s.D, s.M2, 3 * s.D, s.D);
      g.bias = E.in_proj_bias;
      RD_TRY(linear_nt(g, ws + w.wsp[l].in_lo, st));
    }
    float* ctx = ws + w.l[l].ctx;
    if (attn_tc_supported(s.T, s.hd)) {
      RD_TRY(attn_tc_fwd(qkv, lengths, s.B, s.H, s.T, s.hd, s.p, rng, SITE_ATTN + l, ctx, st));
    } else if (attn_small_supported(s.T, s.hd)) {
      RD_TRY(attn_small_fwd(qkv, lengths, s.B, s.H, s.T, s.hd, s.p, rng, SITE_ATTN + l, ctx, st));
    } else {
      {  // S[b,h] = scale * Q K^T
        GemmP g;
        g.A = qkv; g.ta = 0; g.sAi = row3; g.sAk = 1; g.sAzo = 3 * s.D; g.sAzi = s.hd;
        g.B = qkv + s.D; g.tb = 1; g.sBj = row3; g.sBk = 1; g.sBzo = 3 * s.D; g.sBzi = s.hd;
        g.C = Pm; g.sCi = s.T; g.sCj = 1; g.sCzo = s.H * TT; g.sCzi = TT;
        g.M = s.T; g.N = s.T; g.K = s.hd; g.nz = s.B * s.H; g.nz_inner = s.H; g.alpha = scale;
        RD_TRY(gemm(g, st));
      }
      RD_TRY(attn_softmax_fwd(Pm, lengths, s.B, s.H, s.T, s.p, rng, SITE_ATTN + l, Pd, st));
      {  // ctx[b,h] = P V
        GemmP g;
        g.A = Pd ? Pd : Pm; g.ta = 0; g.sAi = s.T; g.sAk = 1; g.sAzo = s.H * TT; g.sAzi = TT;
        g.B = qkv + 2 * s.D; g.tb = 0; g.sBk = row3; g.sBj = 1; g.sBzo = 3 * s.D; g.sBzi = s.hd;
        g.C = ctx; g.sCi = (int64_t)s.B * s.D; g.sCj = 1; g.sCzo = s.D; g.sCzi = s.hd;
        g.M = s.T; g.N = s.hd; g.K = s.T; g.nz = s.B * s.H; g.nz_inner = s.H;
        RD_TRY(gemm(g, st));
      }
    }
    float* r1 = ws + w.l[l].r1; float* x1 = ws + w.l[l].x1;
    {
      GemmP g = nt(ctx, s.D, E.out_proj_weight, s.D, r1, s.D, s.M2, s.D, s.D);
      g.bias = E.out_proj_bias; g.drop_p = s.p; g.rng = rng; g.drop_site = SITE_RESID1 + l;
      g.resid = x; g.resid_ld = s.D;
      if (s.p > 0.f) { g.drop_mask = reinterpret_cast<uint32_t*>(ws + w.l[l].m1); g.drop_mask_ld = (s.D + 31) / 32; }
      RD_TRY(linear_nt(g, ws + w.wsp[l].out_lo, st));
    }
    RD_TRY(layernorm_fwd(r1, E.norm1_weight, E.norm1_bias, s.M2, s.D, dims->ln_eps, x1, ws + w.l[l].st1, st));
    float* f = ws + w.l[l].f; float* r2 = ws + w.l[l].r2;
    {
      GemmP g = nt(x1, s.D, E.linear1_weight, s.D, f, s.nhid, s.M2, s.nhid, s.D);
      g.bias = E.linear1_bias; g.relu = 1; g.drop_p = s.p; g.rng = rng; g.drop_site = SITE_FFN + l;
      RD_TRY(linear_nt(g, ws + w.wsp[l].l1_lo, st));
    }
    {
      GemmP g = nt(f, s.nhid, E.linear2_weight, s.nhid, r2, s.D, s.M2, s.D, s.nhid);
      g.bias = E.linear2_bias; g.drop_p = s.p; g.rng = rng; g.drop_site = SITE_RESID2 + l;
      g.resid = x1; g.resid_ld = s.D;
      if (s.p > 0.f) { g.drop_mask = reinterpret_cast<uint32_t*>(ws + w.l[l].m2); g.drop_mask_ld = (s.D + 31) / 32; }
      RD_TRY(linear_nt(g, ws + w.wsp[l].l2_lo, st));
    }
    RD_TRY(layernorm_fwd(r2, E.norm2_weight, E.norm2_bias, s.M2, s.D, dims->ln_eps, ws + w.Z[l + 1], ws + w.l[l].st2, st));
  }
  float* feat = ws + w.feat; float* hpre = ws + w.hpre;
  RD_TRY(head_fwd(s.B, s.T, s.D, s.emb, s.ds, s.ncls, ws + w.Z[s.L], lengths, statics, P->emb_weight, P->emb_bias,
                  P->mlp0_weight, P->mlp0_bias, P->mlp2_weight, P->mlp2_bias, feat, hpre, logits, y, ws + w.loss_ps, d_logits,
                  loss, reinterpret_cast<unsigned*>(ws + w.cnt), st));
  return 0;
}

static int raindrop_bwd(const rd_dims* dims, const rd_params* P, const float* statics, const int64_t* lengths,
                        const float* nscale, const float* ws, const float* dlogits, const rd_grads* G, float* sc,
                        int phases, float* d_z0_out, cudaStream_t st, const rd_input_grads* IG = nullptr,
                        float* isc = nullptr) {
  Shape s;
  RD_TRY(make_shape(dims, &s));
  if ((phases & ~3) || phases == 0) { set_error("rd_raindrop_v2_bwd: phases must be 1, 2 or 3"); return -2; }
  WsLayout w = ws_layout(s);
  BwLayout b = bw_layout(s);
  // G == null: input gradients only.  Every weight-gradient enqueue (tn), LayerNorm column sum and the head's parameter
  // outputs are skipped; the input-gradient chain itself is the same launches as with parameter gradients.
  const bool pg = G != nullptr;
  const rd_grads none = {};
  if (!pg) G = &none;
  const bool d_src = IG && IG->src;
  const uint64_t* rng = reinterpret_cast<const uint64_t*>(ws + w.rng);
  float* partial = sc + b.partial;
  const float ik = s.p > 0.f ? 1.f / (1.f - s.p) : 1.f;
  float* gA = sc + b.gA; float* gB = sc + b.gB; float* gD = sc + b.gD; float* dP = sc + b.dP;
  WgradQueue wq;     // weight gradients wait here for ONE grouped tensor-core launch per phase

  if (phases & RD_BWD_ENCODER) {
  // ---- head: logits = mlp2(relu(mlp0(feat))), pooled = masked mean          code/models_rd.py:366-385
  const float* feat = ws + w.feat; const float* hpre = ws + w.hpre;
  float* dfeat = sc + b.dfeat; float* dhpre = sc + b.dhpre;
  RD_TRY(head_bwd(s.B, s.T, s.D, s.emb, s.ds, s.ncls, lengths, statics, P->mlp0_weight, P->mlp2_weight, feat, hpre, dlogits,
                  dhpre, dfeat, gA, G->mlp0_weight, G->mlp0_bias, G->mlp2_weight, G->mlp2_bias, G->emb_weight, G->emb_bias, st));

  const float scale = 1.f / sqrtf((float)s.hd);
  const int64_t row3 = (int64_t)s.B * 3 * s.D;
  const int64_t TT = (int64_t)s.T * s.T;
  // the encoder layers are needed for parameter gradients or d(loss)/d(encoder input); a head-only call for d_statics
  // of a frozen model (rd_encoder_head_bwd_inputs with grads = d_enc_in = NULL) stops at the head
  const bool enc = pg || d_z0_out || (phases & RD_BWD_OBPROP);
  for (int l = enc ? s.L - 1 : -1; l >= 0; --l) {
    const rd_encoder_layer_params& E = P->layer[l];
    const rd_encoder_layer_grads& GE = G->layer[l];
    const float* x = ws + w.Z[l];
    const float* qkv = ws + w.l[l].qkv; const float* Pm = ws + w.l[l].P;
    const float* Pd = s.p > 0.f ? ws + w.l[l].Pd : Pm;
    const float* ctx = ws + w.l[l].ctx; const float* r1 = ws + w.l[l].r1; const float* x1 = ws + w.l[l].x1;
    const float* f = ws + w.l[l].f; const float* r2 = ws + w.l[l].r2;
    float* K2 = sc + b.l[l].K2; float* gF = sc + b.l[l].gF; float* K1 = sc + b.l[l].K1; float* dqkv = sc + b.l[l].dqkv;
    // norm2 + feed-forward block.  K2 = gradient w.r.t. the (dropped) linear2 output: operand of its weight
    // gradient, kept until the grouped launch; res = the undropped residual-path gradient
    float* res = s.p > 0.f ? gB : K2;
    int chunks = 0;
    // did the forward GEMMs of this layer store their dropout keep bits (tensor-core epilogue)?  Same predicate, same operands.
    const uint32_t* m2 = nullptr; const uint32_t* m1 = nullptr;
    const int mld = (s.D + 31) / 32;
    if (s.p > 0.f) {
      GemmP g2 = nt(f, s.nhid, E.linear2_weight, s.nhid, const_cast<float*>(r2), s.D, s.M2, s.D, s.nhid);
      g2.bias = E.linear2_bias; g2.drop_p = s.p; g2.rng = rng; g2.resid = x1; g2.resid_ld = s.D;
      if (linear_nt_is_tc(g2, ws + w.wsp[l].l2_lo)) m2 = reinterpret_cast<const uint32_t*>(ws + w.l[l].m2);
      GemmP g1 = nt(ctx, s.D, E.out_proj_weight, s.D, const_cast<float*>(r1), s.D, s.M2, s.D, s.D);
      g1.bias = E.out_proj_bias; g1.drop_p = s.p; g1.rng = rng; g1.resid = x; g1.resid_ld = s.D;
      if (linear_nt_is_tc(g1, ws + w.wsp[l].out_lo)) m1 = reinterpret_cast<const uint32_t*>(ws + w.l[l].m1);
    }
    RD_TRY(layernorm_bwd(r2, ws + w.l[l].st2, E.norm2_weight, gA, s.M2, s.D, res, GE.norm2_weight, GE.norm2_bias,
                         sc + b.l[l].ln[0], K2, s.p, rng, SITE_RESID2 + l, &chunks, st, m2, mld));
    if (pg) {
      RD_TRY(wq.colsum(sc + b.l[l].ln[0], 2 * s.D, chunks, s.D, GE.norm2_weight, st));
      RD_TRY(wq.colsum(sc + b.l[l].ln[0] + s.D, 2 * s.D, chunks, s.D, GE.norm2_bias, st));
      RD_TRY(tn(&wq, K2, s.D, f, s.nhid, GE.linear2_weight, GE.linear2_bias, s.D, s.nhid, s.M2, sc + b.l[l].wp[0], partial, st));
    }
    {   // gF = (K2 . W2) * [f > 0] / (1-p)   ("NT" against W2^T so that the tensor-core kernel applies)
      GemmP g = nt(K2, s.D, ws + w.wsp[l].l2_t, s.D, gF, s.nhid, s.M2, s.nhid, s.D);
      g.gate = f; g.gate_ld = s.nhid; g.gate_scale = ik;  // relu' and the FFN dropout mask in one
      RD_TRY(linear_nt(g, ws + w.wsp[l].l2_tlo, st));
    }
    if (pg) RD_TRY(tn(&wq, gF, s.nhid, x1, s.D, GE.linear1_weight, GE.linear1_bias, s.nhid, s.D, s.M2, sc + b.l[l].wp[1], partial, st));
    {
      GemmP g = nt(gF, s.nhid, ws + w.wsp[l].l1_t, s.nhid, gA, s.D, s.M2, s.D, s.nhid);
      g.resid = res; g.resid_ld = s.D;
      RD_TRY(linear_nt(g, ws + w.wsp[l].l1_tlo, st));
    }
    // norm1 + self-attention block
    res = s.p > 0.f ? gB : K1;
    RD_TRY(layernorm_bwd(r1, ws + w.l[l].st1, E.norm1_weight, gA, s.M2, s.D, res, GE.norm1_weight, GE.norm1_bias,
                         sc + b.l[l].ln[1], K1, s.p, rng, SITE_RESID1 + l, &chunks, st, m1, mld));
    if (pg) {
      RD_TRY(wq.colsum(sc + b.l[l].ln[1], 2 * s.D, chunks, s.D, GE.norm1_weight, st));
      RD_TRY(wq.colsum(sc + b.l[l].ln[1] + s.D, 2 * s.D, chunks, s.D, GE.norm1_bias, st));
      RD_TRY(tn(&wq, K1, s.D, ctx, s.D, GE.out_proj_weight, GE.out_proj_bias, s.D, s.D, s.M2, sc + b.l[l].wp[2], partial, st));
    }
    RD_TRY(linear_nt(nt(K1, s.D, ws + w.wsp[l].out_t, s.D, gD, s.D, s.M2, s.D, s.D), ws + w.wsp[l].out_tlo, st));
    if (attn_tc_supported(s.T, s.hd)) {
      RD_TRY(attn_tc_bwd(qkv, gD, lengths, s.B, s.H, s.T, s.hd, s.p, rng, SITE_ATTN + l, dqkv, st));
    } else if (attn_small_supported(s.T, s.hd)) {
      RD_TRY(attn_small_bwd(qkv, gD, lengths, s.B, s.H, s.T, s.hd, s.p, rng, SITE_ATTN + l, dqkv, st));
    } else {
      {  // dPd[b,h] = dctx V^T
        GemmP g;
        g.A = gD; g.ta = 0; g.sAi = (int64_t)s.B * s.D; g.sAk = 1; g.sAzo = s.D; g.sAzi = s.hd;
        g.B = qkv + 2 * s.D; g.tb = 1; g.sBj = row3; g.sBk = 1; g.sBzo = 3 * s.D; g.sBzi = s.hd;
        g.C = dP; g.sCi = s.T; g.sCj = 1; g.sCzo = s.H * TT; g.sCzi = TT;
        g.M = s.T; g.N = s.T; g.K = s.hd; g.nz = s.B * s.H; g.nz_inner = s.H;
        RD_TRY(gemm(g, st));
      }
      {  // dV[b,h] = Pd^T dctx
        GemmP g;
        g.A = Pd; g.ta = 1; g.sAk = s.T; g.sAi = 1; g.sAzo = s.H * TT; g.sAzi = TT;
        g.B = gD; g.tb = 0; g.sBk = (int64_t)s.B * s.D; g.sBj = 1; g.sBzo = s.D; g.sBzi = s.hd;
        g.C = dqkv + 2 * s.D; g.sCi = row3; g.sCj = 1; g.sCzo = 3 * s.D; g.sCzi = s.hd;
        g.M = s.T; g.N = s.hd; g.K = s.T; g.nz = s.B * s.H; g.nz_inner = s.H;
        RD_TRY(gemm(g, st));
      }
      RD_TRY(attn_softmax_bwd(Pm, dP, s.B, s.H, s.T, s.p, rng, SITE_ATTN + l, st));
      {  // dQ[b,h] = scale * dS K
        GemmP g;
        g.A = dP; g.ta = 0; g.sAi = s.T; g.sAk = 1; g.sAzo = s.H * TT; g.sAzi = TT;
        g.B = qkv + s.D; g.tb = 0; g.sBk = row3; g.sBj = 1; g.sBzo = 3 * s.D; g.sBzi = s.hd;
        g.C = dqkv; g.sCi = row3; g.sCj = 1; g.sCzo = 3 * s.D; g.sCzi = s.hd;
        g.M = s.T; g.N = s.hd; g.K = s.T; g.nz = s.B * s.H; g.nz_inner = s.H; g.alpha = scale;
        RD_TRY(gemm(g, st));
      }
      {  // dK[b,h] = scale * dS^T Q
        GemmP g;
        g.A = dP; g.ta = 1; g.sAk = s.T; g.sAi = 1; g.sAzo = s.H * TT; g.sAzi = TT;
        g.B = qkv; g.tb = 0; g.sBk = row3; g.sBj = 1; g.sBzo = 3 * s.D; g.sBzi = s.hd;
        g.C = dqkv + s.D; g.sCi = row3; g.sCj = 1; g.sCzo = 3 * s.D; g.sCzi = s.hd;
        g.M = s.T; g.N = s.hd; g.K = s.T; g.nz = s.B * s.H; g.nz_inner = s.H; g.alpha = scale;
        RD_TRY(gemm(g, st));
      }
    }
    if (pg) RD_TRY(tn(&wq, dqkv, 3 * s.D, x, s.D, GE.in_proj_weight, GE.in_proj_bias, 3 * s.D, s.D, s.M2, sc + b.l[l].wp[3], partial, st));
    {
      // the first layer's input gradient is d(loss)/d(encoder input): optionally delivered straight to the caller
      GemmP g = nt(dqkv, 3 * s.D, ws + w.wsp[l].in_t, 3 * s.D, (l == 0 && d_z0_out) ? d_z0_out : gA, s.D, s.M2, s.D, 3 * s.D);
      g.resid = res; g.resid_ld = s.D;
      RD_TRY(linear_nt(g, ws + w.wsp[l].in_tlo, st));
    }
  }
  if (!(phases & RD_BWD_OBPROP)) RD_TRY(wq.flush(st));   // encoder + head gradients complete: the caller may reduce them now
  }

  // with neither parameter gradients nor d_src wanted nothing below the encoder input is needed
  if ((phases & RD_BWD_OBPROP) && (pg || d_src)) {
  // ---- observation propagation: gA = d(loss)/d(Z0) [T,B,D]          code/models_rd.py:322-343
  float* gO2 = sc + b.gO2; float* gO1 = sc + b.gO1;
  const float* X0 = ws + w.X0; const float* H1 = ws + w.H1;
  const int tc = s.tc;
  RD_TRY(obprop_out_grad(gA, ws + w.Z[0], nscale, s.B, s.T, s.N, s.dob, s.D, tc && !s.exact, gO2, st));
  if (pg) RD_TRY(tn(&wq, gO2, s.C, H1, s.C, G->ob2_value_weight, G->ob2_value_bias, s.C, s.C, s.M1, sc + b.wp_ob[0], partial, st));
  if (tc) {
    // dZ1 = (dZ2 . W2) * s * [H1 > 0] on the tensor cores: "NT" form against a transposed, TF32-rounded W2
    const float* W2t = ws + w.W2t;      // written by the forward's weight-prep launch
    ObpropTcArgs a;
    a.x = gO2; a.W = W2t; a.bias = nullptr; a.relu = 0; a.scale = nscale; a.scale_mod = s.N; a.gate = H1;
    a.W_lo = s.exact ? ws + w.W2tlo : nullptr;
    a.rows = s.M1; a.C = s.C; a.out = gO1;
    RD_TRY(obprop_tc_fwd(a, st));
  } else {
    GemmP g = nn(gO2, s.C, P->ob2_value_weight, s.C, gO1, s.C, s.M1, s.C, s.C);
    g.rowscale = nscale; g.rowscale_mod = s.N; g.gate = H1; g.gate_ld = s.C;
    RD_TRY(gemm(g, st));
  }
  if (pg) RD_TRY(tn(&wq, gO1, s.C, X0, s.C, G->ob1_value_weight, G->ob1_value_bias, s.C, s.C, s.M1, sc + b.wp_ob[1], partial, st));
  RD_TRY(wq.flush(st));
  if (d_src) {
    // dX0 = gO1 . W1, gated by X0 != 0 (relu' of the lift and its dropout keep bit at once: X0 is non-zero exactly where
    // both are 1) and scaled by 1/(1-p), then reduced over the d_ob channels against R_u.  Always error-compensated:
    // gO1 is not TF32-rounded (rounding it would change the ob1 weight gradient)
    const float ik = s.p > 0.f ? 1.f / (1.f - s.p) : 1.f;
    const InLayout il = in_layout(s);
    if (lift_bwd_tc(s)) {
      WeightSplit it = {P->ob1_value_weight, s.C, s.C, nullptr, isc + il.W1t, isc + il.W1tlo};
      RD_TRY(split_weights(&it, 1, st));
      ObpropTcArgs a;
      a.x = gO1; a.W = isc + il.W1t; a.W_lo = isc + il.W1tlo; a.bias = nullptr; a.relu = 0; a.gate = X0;
      a.rows = s.M1; a.C = s.C; a.out = IG->src;
      a.pB = s.B; a.pN = s.N; a.pdob = s.dob; a.pD = 2 * s.N;
      a.lift_ru = P->R_u; a.lift_scale = ik;
      RD_TRY(obprop_tc_fwd(a, st));
    } else {
      GemmP g = nn(gO1, s.C, P->ob1_value_weight, s.C, isc + il.dX0, s.C, s.M1, s.C, s.C);
      g.gate = X0; g.gate_ld = s.C; g.gate_scale = ik;
      RD_TRY(gemm(g, st));
    }
  }
  }
  if (IG && (IG->src || IG->times || IG->statics)) {
    RD_TRY(input_grad_tail(s.B, s.T, s.N, s.dob, s.D, gA, ws + w.Z[0], dims->pe_timescales, RD_D_PE, sc + b.dfeat, s.Df,
                           P->emb_weight, s.emb, s.ds, (d_src && !lift_bwd_tc(s)) ? isc + in_layout(s).dX0 : nullptr, P->R_u,
                           IG->src, IG->times, IG->statics, st));
  }
  return 0;
}

}  // namespace rd

// =================================================================================================
// C ABI
// =================================================================================================
using namespace rd;

extern "C" {

int rd_abi_version(void) { return RD_ABI_VERSION; }
const char* rd_last_error_string(void) { return last_error(); }
uint64_t rd_launch_count(void) { return launch_count(); }

int rd_node_scale(const int64_t* edge_tgt, const float* edge_w, int32_t E, int32_t N, float* out, void* stream) {
  if (!edge_tgt || !edge_w || !out || E < 0 || N < 1) { set_error("rd_node_scale: bad arguments"); return -2; }
  return node_scale(edge_tgt, edge_w, E, N, out, (cudaStream_t)stream);
}

size_t rd_obprop_fwd_scratch_bytes(int64_t rows, int32_t C) {
  return (size_t)(round_up(rows * C, 64) + round_up((int64_t)C * C, 64)) * sizeof(float);
}

int rd_obprop_fwd(const float* x, const float* weight, const float* bias, const float* nscale, int32_t mod,
                  int64_t rows, int32_t C, float* out, void* scratch, void* stream) {
  if (!x || !weight || !bias || !nscale || !out || rows < 0 || C < 1 || mod < 1) {
    set_error("rd_obprop_fwd: bad arguments");
    return -2;
  }
  if (rows == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  ObpropTcArgs a;
  a.x = x; a.W = weight; a.bias = bias; a.scale = nscale; a.scale_mod = mod; a.rows = rows; a.C = C; a.out = out;
  if (obprop_tc_supported(C) && scratch) {   // arbitrary caller data
    float* xr = (float*)scratch;
    float* wr = xr + round_up(rows * C, 64);
    if (obprop_tc_exact(rows, C, 0)) {        // latency-bound size: error-compensated kernel, operands as they are
      WeightSplit it = {weight, C, C, wr, nullptr, nullptr};
      RD_TRY(split_weights(&it, 1, st));
      a.W_lo = wr;
    } else {                                  // streaming size: round both operands to TF32 first, single pass
      RD_TRY(round_tf32(x, rows * C, xr, st));
      RD_TRY(round_tf32(weight, (int64_t)C * C, wr, st));
      a.x = xr; a.W = wr;
    }
  }
  return obprop_forward(a, st);
}

size_t rd_obprop_bwd_scratch_bytes(int64_t rows, int32_t C) {
  int64_t tcp = tc_wgrad_partial_floats(C, C, rows), skp = splitk_partial_floats(C, C, rows);
  int64_t a = round_up(rows * C, 64) + round_up(tcp > skp ? tcp : skp, 64);
  return (size_t)a * sizeof(float);
}

int rd_obprop_bwd(const float* x, const float* out, const float* d_out, const float* weight, const float* nscale,
                  int32_t mod, int64_t rows, int32_t C, float* d_x, float* d_weight, float* d_bias, void* scratch,
                  void* stream) {
  if (!x || !out || !d_out || !weight || !nscale || !d_weight || !d_bias || !scratch || rows < 1 || C < 1) {
    set_error("rd_obprop_bwd: bad arguments");
    return -2;
  }
  cudaStream_t st = (cudaStream_t)stream;
  float* dpre = (float*)scratch;
  float* partial = dpre + round_up(rows * C, 64);
  RD_TRY(relu_scale_bwd(d_out, out, nscale, mod, rows, C, dpre, st));
  RD_TRY(tn(nullptr, dpre, C, x, C, d_weight, d_bias, C, C, rows, partial, partial, st));
  if (d_x) RD_TRY(gemm(nn(dpre, C, weight, C, d_x, C, rows, C, C), st));
  return 0;
}

size_t rd_linear_scratch_bytes(int32_t in_features, int32_t out_features) {
  return (size_t)round_up((int64_t)in_features * out_features, 64) * sizeof(float);
}

int rd_linear_fwd(const float* x, const float* weight, const float* bias, int64_t rows, int32_t in_features,
                  int32_t out_features, int32_t relu, float* out, void* scratch, void* stream) {
  if (!x || !weight || !out || !scratch || rows < 0 || in_features < 1 || out_features < 1) {
    set_error("rd_linear_fwd: bad arguments");
    return -2;
  }
  if (rows == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  WeightSplit it = {weight, out_features, in_features, (float*)scratch, nullptr, nullptr};
  RD_TRY(split_weights(&it, 1, st));
  GemmP g = nt(x, in_features, weight, in_features, out, out_features, rows, out_features, in_features);
  g.bias = bias; g.relu = relu;
  return linear_nt(g, (const float*)scratch, st);
}

int rd_debug_attention_timing(uint64_t* buffer) { attn_tc_set_debug((unsigned long long*)buffer); return 0; }
int rd_debug_gemm_timing(uint64_t* buffer) { tc_gemm_set_debug((unsigned long long*)buffer); return 0; }

int rd_temporal_attention_fwd(const float* qkv, const int64_t* lengths, int32_t B, int32_t H, int32_t T, int32_t hd,
                              float drop_p, const uint64_t* rng_captured, uint32_t site, int32_t impl, float* ctx,
                              void* stream) {
  if (!qkv || !lengths || !ctx || B < 1 || H < 1 || T < 1 || hd < 1 || drop_p < 0.f || drop_p >= 1.f || (drop_p > 0.f && !rng_captured)) {
    set_error("rd_temporal_attention_fwd: bad arguments");
    return -2;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if ((impl == 0 || impl == 1) && attn_tc_supported(T, hd)) return attn_tc_fwd(qkv, lengths, B, H, T, hd, drop_p, rng_captured, site, ctx, st);
  if ((impl == 0 || impl == 2) && attn_small_supported(T, hd)) return attn_small_fwd(qkv, lengths, B, H, T, hd, drop_p, rng_captured, site, ctx, st);
  set_error("rd_temporal_attention_fwd: T=%d hd=%d not supported by implementation %d", T, hd, impl);
  return -2;
}

int rd_temporal_attention_bwd(const float* qkv, const float* d_ctx, const int64_t* lengths, int32_t B, int32_t H,
                              int32_t T, int32_t hd, float drop_p, const uint64_t* rng_captured, uint32_t site,
                              int32_t impl, float* d_qkv, void* stream) {
  if (!qkv || !d_ctx || !lengths || !d_qkv || B < 1 || H < 1 || T < 1 || hd < 1 || drop_p < 0.f || drop_p >= 1.f ||
      (drop_p > 0.f && !rng_captured)) {
    set_error("rd_temporal_attention_bwd: bad arguments");
    return -2;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if ((impl == 0 || impl == 1) && attn_tc_supported(T, hd)) return attn_tc_bwd(qkv, d_ctx, lengths, B, H, T, hd, drop_p, rng_captured, site, d_qkv, st);
  if ((impl == 0 || impl == 2) && attn_small_supported(T, hd)) return attn_small_bwd(qkv, d_ctx, lengths, B, H, T, hd, drop_p, rng_captured, site, d_qkv, st);
  set_error("rd_temporal_attention_bwd: T=%d hd=%d not supported by implementation %d", T, hd, impl);
  return -2;
}

size_t rd_linear_wgrad_partial_bytes(int64_t rows, int32_t out_features, int32_t in_features) {
  if (rows < 1 || out_features < 1 || in_features < 1) return 0;
  int64_t a = tc_wgrad_partial_floats(out_features, in_features, rows), b = splitk_partial_floats(out_features, in_features, rows);
  return (size_t)round_up(a > b ? a : b, 64) * sizeof(float);
}

int rd_linear_wgrad_group(const rd_wgrad_item* items, int32_t n, void* stream) {
  if (!items || n < 0) { set_error("rd_linear_wgrad_group: bad arguments"); return -2; }
  cudaStream_t st = (cudaStream_t)stream;
  WgradQueue wq;
  for (int i = 0; i < n; ++i) {
    const rd_wgrad_item& it = items[i];
    if (!it.d_out || !it.x || !it.d_weight || !it.d_bias || !it.partial || it.rows < 1 || it.out_features < 1 || it.in_features < 1) {
      set_error("rd_linear_wgrad_group: problem %d has a NULL pointer or an empty shape", i);
      return -2;
    }
    RD_TRY(tn(&wq, it.d_out, it.out_features, it.x, it.in_features, it.d_weight, it.d_bias, it.out_features, it.in_features,
              it.rows, (float*)it.partial, (float*)it.partial, st));
  }
  return wq.flush(st);
}

size_t rd_workspace_bytes(const rd_dims* dims) {
  Shape s;
  if (make_shape(dims, &s) != 0) return 0;
  return (size_t)ws_layout(s).total * sizeof(float);
}

size_t rd_backward_scratch_bytes(const rd_dims* dims) {
  Shape s;
  if (make_shape(dims, &s) != 0) return 0;
  return (size_t)bw_layout(s).total * sizeof(float);
}

int64_t rd_workspace_offset(const rd_dims* dims, int32_t which, int64_t* n_floats) {
  Shape s;
  if (make_shape(dims, &s) != 0) return -1;
  WsLayout w = ws_layout(s);
  int64_t off = -1, n = 0;
  switch (which) {
    case RD_WS_X0: off = w.X0; n = s.M1 * s.C; break;
    case RD_WS_H1: off = w.H1; n = s.M1 * s.C; break;
    case RD_WS_ENC_IN: off = w.Z[0]; n = s.M2 * s.D; break;
    case RD_WS_ENC_OUT: off = w.Z[s.L]; n = s.M2 * s.D; break;
    case RD_WS_FEAT: off = w.feat; n = (int64_t)s.B * s.Df; break;
    case RD_WS_RNG: off = w.rng; n = 4; break;
    default: set_error("rd_workspace_offset: unknown buffer %d", which); return -1;
  }
  if (n_floats) *n_floats = n;
  return off * (int64_t)sizeof(float);
}

int rd_raindrop_v2_fwd(const rd_dims* dims, const rd_params* params, const float* src, const float* statics,
                       const float* times, const int64_t* lengths, const float* node_scale, uint64_t* rng_state,
                       void* workspace, float* logits, const int64_t* y, float* loss, float* d_logits, void* stream) {
  if (!dims || !params || !src || !times || !lengths || !node_scale || !workspace || !logits) {
    set_error("rd_raindrop_v2_fwd: NULL argument");
    return -2;
  }
  return raindrop_fwd(dims, params, src, statics, times, lengths, node_scale, rng_state, (float*)workspace, logits,
                      y, loss, d_logits, 0, (cudaStream_t)stream);
}

int rd_raindrop_v2_bwd(const rd_dims* dims, const rd_params* params, const float* statics, const int64_t* lengths,
                       const float* node_scale, const void* workspace, const float* d_logits, const rd_grads* grads,
                       void* scratch, int32_t phases, void* stream) {
  if (!dims || !params || !lengths || !node_scale || !workspace || !d_logits || !grads || !scratch) {
    set_error("rd_raindrop_v2_bwd: NULL argument");
    return -2;
  }
  return raindrop_bwd(dims, params, statics, lengths, node_scale, (const float*)workspace, d_logits, grads,
                      (float*)scratch, phases, nullptr, (cudaStream_t)stream);
}

size_t rd_input_grad_scratch_bytes(const rd_dims* dims) {
  Shape s;
  if (make_shape(dims, &s) != 0) return 0;
  return (size_t)in_layout(s).total * sizeof(float);
}

int rd_raindrop_v2_bwd_inputs(const rd_dims* dims, const rd_params* params, const float* statics, const int64_t* lengths,
                              const float* node_scale, const void* workspace, const float* d_logits, const rd_grads* grads,
                              const rd_input_grads* in_grads, void* scratch, void* in_scratch, void* stream) {
  if (!dims || !params || !lengths || !node_scale || !workspace || !d_logits || !scratch) {
    set_error("rd_raindrop_v2_bwd_inputs: NULL argument");
    return -2;
  }
  const bool any_in = in_grads && (in_grads->src || in_grads->statics || in_grads->times);
  if (!grads && !any_in) { set_error("rd_raindrop_v2_bwd_inputs: neither parameter nor input gradients requested"); return -2; }
  if (any_in && in_grads->src && !in_scratch) { set_error("rd_raindrop_v2_bwd_inputs: d_src needs in_scratch"); return -2; }
  if (any_in && in_grads->statics && (dims->d_static < 1 || !statics)) {
    set_error("rd_raindrop_v2_bwd_inputs: a static gradient needs d_static > 0 and statics");
    return -2;
  }
  return raindrop_bwd(dims, params, statics, lengths, node_scale, (const float*)workspace, d_logits, grads, (float*)scratch,
                      RD_BWD_ALL, nullptr, (cudaStream_t)stream, any_in ? in_grads : nullptr, (float*)in_scratch);
}

int rd_positional_encoding(const float* times, int64_t n_tokens, const float* timescales_host, int32_t d_pe, float* out,
                           int64_t ld, int32_t col0, void* stream) {
  if (!times || !timescales_host || !out || n_tokens < 0) { set_error("rd_positional_encoding: bad arguments"); return -2; }
  if (n_tokens == 0) return 0;
  return posenc(times, n_tokens, timescales_host, d_pe, out, ld, col0, (cudaStream_t)stream);
}

int rd_encoder_head_fwd(const rd_dims* dims, const rd_params* params, const float* statics, const int64_t* lengths,
                        uint64_t* rng_state, void* workspace, float* logits, const int64_t* y, float* loss, float* d_logits,
                        void* stream) {
  if (!dims || !params || !lengths || !workspace || !logits) { set_error("rd_encoder_head_fwd: NULL argument"); return -2; }
  return raindrop_fwd(dims, params, nullptr, statics, nullptr, lengths, nullptr, rng_state, (float*)workspace, logits, y, loss,
                      d_logits, 1, (cudaStream_t)stream);
}

int rd_encoder_head_bwd(const rd_dims* dims, const rd_params* params, const float* statics, const int64_t* lengths,
                        const void* workspace, const float* d_logits, const rd_grads* grads, void* scratch, float* d_enc_in,
                        void* stream) {
  if (!dims || !params || !lengths || !workspace || !d_logits || !grads || !scratch || !d_enc_in) {
    set_error("rd_encoder_head_bwd: NULL argument");
    return -2;
  }
  return raindrop_bwd(dims, params, statics, lengths, nullptr, (const float*)workspace, d_logits, grads, (float*)scratch,
                      RD_BWD_ENCODER, d_enc_in, (cudaStream_t)stream);
}

int rd_encoder_head_bwd_inputs(const rd_dims* dims, const rd_params* params, const float* statics, const int64_t* lengths,
                               const void* workspace, const float* d_logits, const rd_grads* grads, float* d_enc_in,
                               float* d_statics, void* scratch, void* stream) {
  if (!dims || !params || !lengths || !workspace || !d_logits || !scratch) {
    set_error("rd_encoder_head_bwd_inputs: NULL argument");
    return -2;
  }
  if (!grads && !d_enc_in && !d_statics) { set_error("rd_encoder_head_bwd_inputs: no gradient requested"); return -2; }
  if (d_statics && (dims->d_static < 1 || !statics || !params->emb_weight)) {
    set_error("rd_encoder_head_bwd_inputs: a static gradient needs d_static > 0, statics and emb_weight");
    return -2;
  }
  rd_input_grads ig = {nullptr, d_statics, nullptr};
  return raindrop_bwd(dims, params, statics, lengths, nullptr, (const float*)workspace, d_logits, grads, (float*)scratch,
                      RD_BWD_ENCODER, d_enc_in, (cudaStream_t)stream, d_statics ? &ig : nullptr);
}

int rd_positional_encoding_bwd(const float* pe, const float* d_pe, int64_t n_tokens, const float* timescales_host,
                               int32_t d_pe_width, int64_t ld, int32_t col0, float* d_times, void* stream) {
  if (!pe || !d_pe || !timescales_host || !d_times || n_tokens < 0 || col0 < 0 || ld < (int64_t)col0 + d_pe_width) {
    set_error("rd_positional_encoding_bwd: bad arguments");
    return -2;
  }
  if (n_tokens == 0) return 0;
  return posenc_bwd(pe, d_pe, n_tokens, timescales_host, d_pe_width, ld, col0, d_times, (cudaStream_t)stream);
}

int rd_dropout(const float* x, int64_t n, float p, const uint64_t* rng_captured, uint32_t site, float* y, void* stream) {
  if (!x || !y || !rng_captured || n < 0 || p < 0.f || p >= 1.f) { set_error("rd_dropout: bad arguments"); return -2; }
  if (n == 0) return 0;
  return apply_dropout(x, n, p, rng_captured, site, y, (cudaStream_t)stream);
}

int rd_gather_batch(const float* src, const int64_t* idx, int64_t T, int64_t n_total, int32_t width, int32_t B, float* out,
                    void* stream) {
  if (!src || !idx || !out || T < 0 || n_total < 1 || width < 1 || B < 0) { set_error("rd_gather_batch: bad arguments"); return -2; }
  return gather_batch(src, idx, T, n_total, width, B, out, (cudaStream_t)stream);
}

int rd_assemble_batch(const float* P, const float* Ptime, const float* Pstatic, const int64_t* y, const int64_t* idx,
                      int32_t T, int64_t n_total, int32_t width, int32_t d_static, int32_t B, float* src, float* times,
                      float* statics, int64_t* y_out, int64_t* lengths, void* stream) {
  if (!P || !Ptime || !idx || !src || !times || !lengths || T < 1 || n_total < 1 || width < 1 || B < 0 || (Pstatic && (!statics || d_static < 1)) ||
      (y && !y_out)) {
    set_error("rd_assemble_batch: bad arguments");
    return -2;
  }
  return assemble_batch(P, Ptime, Pstatic, y, idx, T, n_total, width, d_static, B, src, times, statics, y_out, lengths,
                        (cudaStream_t)stream);
}

size_t rd_feature_stats_scratch_bytes(int64_t n, int32_t T, int32_t F) {
  if (n < 1 || T < 1 || F < 1) return 0;
  return (size_t)feature_stats_scratch_bytes(n, T, F);
}

int rd_feature_stats(const float* raw, int64_t n, int32_t T, int32_t F, float* mean, float* stdv, void* scratch, void* stream) {
  if (!raw || !mean || !stdv || !scratch || n < 1 || T < 1 || F < 1) { set_error("rd_feature_stats: bad arguments"); return -2; }
  return feature_stats(raw, n, T, F, mean, stdv, scratch, (cudaStream_t)stream);
}

int rd_mask_normalize(const float* raw, const float* mean, const float* stdv, int64_t n, int32_t T, int32_t F, float* out,
                      const float* minutes, float* times_out, void* stream) {
  if (!raw || !mean || !stdv || !out || n < 1 || T < 1 || F < 1 || (minutes && !times_out)) {
    set_error("rd_mask_normalize: bad arguments");
    return -2;
  }
  return mask_normalize(raw, mean, stdv, n, T, F, out, minutes, times_out, (cudaStream_t)stream);
}

int rd_zero_features(float* P, int64_t T, int32_t B, int32_t width, const int64_t* idx, int32_t K, int32_t per_sample,
                     void* stream) {
  if (!P || !idx || T < 0 || B < 0 || width < 2 || K < 0) { set_error("rd_zero_features: bad arguments"); return -2; }
  return zero_features(P, T, B, width, idx, K, per_sample, (cudaStream_t)stream);
}

int rd_cross_entropy_fwd_bwd(const float* logits, const int64_t* y, int32_t B, int32_t ncls, float* loss,
                             float* d_logits, void* stream) {
  if (!logits || !y || !loss || B < 1 || ncls < 1) { set_error("rd_cross_entropy_fwd_bwd: bad arguments"); return -2; }
  return cross_entropy(logits, y, B, ncls, loss, d_logits, (cudaStream_t)stream);
}

int rd_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                 const float* lr_dev, float beta1, float beta2, float eps, float grad_scale, int64_t* step, void* stream) {
  if (!param || !grad || !exp_avg || !exp_avg_sq || !step || n < 0) { set_error("rd_adam_step: bad arguments"); return -2; }
  if (n == 0) return 0;
  return adam(param, grad, exp_avg, exp_avg_sq, n, lr, lr_dev, beta1, beta2, eps, grad_scale, step, (cudaStream_t)stream);
}

int rd_debug_dropout_mask(const uint64_t* rng_captured, uint32_t site, int64_t n, float p, float* out, void* stream) {
  if (!rng_captured || !out || n < 0 || p < 0.f || p >= 1.f) { set_error("rd_debug_dropout_mask: bad arguments"); return -2; }
  if (n == 0) return 0;
  return apply_dropout(nullptr, n, p, rng_captured, site, out, (cudaStream_t)stream);
}

}  // extern "C"

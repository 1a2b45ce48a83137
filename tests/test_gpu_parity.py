"""GPU parity tests proper: the CUDA path (through the C ABI) against the reference's outputs
(tests/golden, generated from the reference's own files) and against the CPU oracle on seeded inputs.

Tolerance (BASELINE.json north_star: "forward output within 1e-3 rel-tol of the reference"), defined
normwise as max|delta| / max|ref| (BASELINE.md section 2).  The observation-propagation GEMMs run in
TF32 (expected ~1e-4), everything else in fp32 (expected ~1e-6).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import (build_dropin, case_setup, check_against_golden, load_golden, normwise, rel_l2,
                     sparse_structure, to_dev)
from raindrop_b200.synth import make_batch, model_config, synth_weights, used_param_keys

pytestmark = pytest.mark.gpu

FWD_TOL = 1e-3     # north_star tolerance on forward tensors
# The two observation-propagation GEMMs run in one of two arithmetic modes (rd_dims.obprop_mode):
#   EXACT (2, and what "auto" picks at every latency-bound size incl. the benchmarked P19 B=128): error-compensated
#       3xTF32, fp32-level.  Every one of the 34 gradients must match the fp32 reference to GRAD_TOL_EXACT max-norm
#       and the ob-prop output to 1e-5.
#   FAST (1, what "auto" picks in the HBM-/tensor-bound regime): single-pass TF32 on operands rounded to TF32.
#       Forward error ~3e-4, but the gradient of a ReLU network is DISCONTINUOUS in forward perturbations: a
#       pre-activation within 3e-4 of zero flips its gate and moves a few isolated gradient entries by up to ~10 % of
#       max|grad| while the mean error stays ~0.3 % (DESIGN.md section "Precision").  There we use max-norm GRAD_TOL for
#       every parameter outside the ob-prop layers, relative L2 OBPROP_GRAD_L2 for the two lin_value weights/biases,
#       and a tight check against the oracle evaluated under the kernels' rounding model (`tf32_model=True`).
GRAD_TOL_EXACT = 2e-3
# the widest layers (C = T*d_ob >= 1024: PAM 2400, LARGE 1024) tested at B = 2..3: two fp32 implementations of a
# K = 1024..2400 dot product differ by ~1e-5, which still flips a ReLU gate now and then, and with so few rows one
# flipped gate is visible in max-norm
GRAD_TOL_EXACT_WIDE = 1e-2


def _exact_tol(cfg):
    return GRAD_TOL_EXACT_WIDE if cfg["max_len"] * cfg["d_ob"] >= 1024 else GRAD_TOL_EXACT

GRAD_TOL = 2e-2
OBPROP_GRAD_L2 = 5e-2
MODEL_TOL = 5e-3
EXACT, FAST = 2, 1


def _grad_check_fp32(name, got, ref, mode=FAST, tol=GRAD_TOL_EXACT):
    if mode == EXACT:
        e = normwise(got, ref)
        assert e < tol, (name, "normwise (exact mode)", e)
    elif "lin_value" in name:
        e = rel_l2(got, ref)
        assert e < OBPROP_GRAD_L2, (name, "rel_l2", e)
    else:
        e = normwise(got, ref)
        assert e < GRAD_TOL, (name, "normwise", e)

GOLDEN_CASES = ["tiny_dense", "tiny_t0", "tiny_sparse", "tiny8_nostatic", "p19_b4", "p19_b5_leave10", "p12_b2", "pam_b2"]


def _run_dropin(cfg, batch, weight_seed, train=False, mode=0):
    from raindrop_b200 import functional as RF
    from raindrop_b200 import lib as L
    model = build_dropin(cfg, weight_seed)
    model.train(train)
    model._plan.debug_keep_workspace = True
    model._plan.obprop_mode = mode
    d = to_dev(batch)
    logits, distance, third = model.forward(d["src"], d["static"], d["times"], d["lengths"])
    assert third is None and distance.dim() == 0
    loss = F.cross_entropy(logits, d["y"])
    loss.backward()
    T, B = d["src"].shape[0], d["src"].shape[1]
    D = cfg["d_inp"] * cfg["d_ob"] + 16
    enc_in = RF.workspace_view(model._plan, L.WS_ENC_IN).view(T, B, D)
    enc_out = RF.workspace_view(model._plan, L.WS_ENC_OUT).view(T, B, D)
    return model, logits, distance, loss, enc_in, enc_out


@pytest.mark.parametrize("mode", [EXACT, FAST], ids=["exact", "fast"])
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_golden_fixture(golden_dir, name, mode):
    """CUDA forward + backward vs the outputs of the reference's own unmodified files, in both arithmetic modes of
    the ob-prop GEMMs."""
    z, meta = load_golden(golden_dir, name)
    cfg, batch = case_setup(meta)
    model, logits, distance, loss, enc_in, enc_out = _run_dropin(cfg, batch, meta["weight_seed"], mode=mode)
    errs = {}
    assert normwise(logits, z["logits"]) < (1e-4 if mode == EXACT else FWD_TOL)
    assert abs(loss.item() - float(z["loss"])) < 1e-3 * max(1.0, abs(float(z["loss"])))
    assert float(distance) == float(z["distance"]) == 0.0
    full = meta["full_tensors"]
    D4 = cfg["d_inp"] * cfg["d_ob"]
    check_against_golden(z, full, "obs", enc_in[:, :, :D4], 1e-4 if mode == EXACT else FWD_TOL, errs)   # exact: K <= 2400 products, dropped lo.lo terms
    check_against_golden(z, full, "pe", enc_in[:, :, D4:], 1e-5, errs)
    # the encoder output at padded positions is never used by the reference (masked mean) -> compare valid rows
    lengths = batch["lengths"]
    T = enc_out.shape[0]
    valid = (torch.arange(T)[:, None] < lengths[None, :]).to(enc_out.device)[:, :, None]
    if full:
        ref = torch.from_numpy(z["enc"]).to(enc_out.device)
        e = normwise(enc_out * valid, ref * valid)
        assert e < FWD_TOL, e
    params = dict(model.named_parameters())
    for k in used_param_keys(cfg):
        assert params[k].grad is not None, k
        if mode == EXACT:
            check_against_golden(z, full, "grad." + k, params[k].grad, _exact_tol(cfg), errs)
        elif "lin_value" in k:
            check_against_golden(z, full, "grad." + k, params[k].grad, OBPROP_GRAD_L2 * (1 if full else 2), errs, metric=rel_l2)
        else:
            check_against_golden(z, full, "grad." + k, params[k].grad, GRAD_TOL, errs)
    unused = [k for k, p in params.items() if k not in set(used_param_keys(cfg))]
    assert all(params[k].grad is None for k in unused)     # same 34 tensors get gradient as in the reference
    print(name, "mode", mode, "worst:", max(errs.items(), key=lambda kv: kv[1]))


@pytest.mark.parametrize("cfg_name,B,opts", [
    ("P19", 1, {}), ("P19", 37, {}), ("P19", 100, {"first_time_zero": True}), ("P19", 128, {"zero_sensors": 10}),
    ("P12", 5, {}), ("PAM", 3, {}), ("TINY", 7, {"full_length": True}), ("TINY8", 9, {}),
    ("LARGE", 2, {}),      # BASELINE configs[4] shape: 128 sensors, T=256 (C=1024, D=528, head dim 264)
])
def test_against_oracle(cfg_name, B, opts):
    """Seeded inputs, sizes the dense oracle finishes in seconds (arbitrary B incl. remainder batches)."""
    from oracle.raindrop_oracle import build_oracle_model
    cfg = model_config(cfg_name, dropout=0.2)
    batch = make_batch(cfg, B, seed=100 + B, **opts)
    oracle = build_oracle_model(cfg).eval()
    synth_weights(oracle, cfg, seed=21)
    stages = {}
    ref_logits, _, _ = oracle.forward_dense(batch["src"], batch["static"], batch["times"], batch["lengths"], stages=stages)
    ref_loss = F.cross_entropy(ref_logits, batch["y"])
    ref_loss.backward()
    D4 = cfg["d_inp"] * cfg["d_ob"]
    go = dict(oracle.named_parameters())
    ref_grads = {k: go[k].grad.clone() for k in used_param_keys(cfg)}
    # ---- error-compensated mode: fp32-level agreement with the fp32 oracle, every tensor -------------
    model, logits, _, loss, enc_in, enc_out = _run_dropin(cfg, batch, 21, mode=EXACT)
    assert normwise(enc_in[:, :, :D4], stages["obs"]) < 1e-4
    assert normwise(enc_in[:, :, D4:], stages["pe"]) < 1e-5
    assert normwise(logits, ref_logits) < 1e-4
    gp = dict(model.named_parameters())
    worst = max((normwise(gp[k].grad, ref_grads[k]), k) for k in used_param_keys(cfg))
    print(cfg_name, B, "exact-mode worst gradient error", worst)
    for k in used_param_keys(cfg):
        _grad_check_fp32(k, gp[k].grad, ref_grads[k], EXACT, _exact_tol(cfg))
    # ---- single-pass TF32 mode ----------------------------------------------------------------------
    model, logits, _, loss, enc_in, enc_out = _run_dropin(cfg, batch, 21, mode=FAST)
    assert normwise(enc_in[:, :, :D4], stages["obs"]) < FWD_TOL
    assert normwise(logits, ref_logits) < FWD_TOL
    gp = dict(model.named_parameters())
    for k in used_param_keys(cfg):
        _grad_check_fp32(k, gp[k].grad, ref_grads[k], FAST)
    # same model evaluated under the kernels' TF32 rounding model: everything must agree tightly
    oracle.zero_grad()
    st2 = {}
    m_logits, _, _ = oracle.forward_dense(batch["src"], batch["static"], batch["times"], batch["lengths"], stages=st2,
                                          tf32_model=True)
    F.cross_entropy(m_logits, batch["y"]).backward()
    assert normwise(enc_in[:, :, :D4], st2["obs"].detach()) < 1e-4
    assert normwise(logits, m_logits.detach()) < 1e-4
    for k in used_param_keys(cfg):
        if "lin_value" in k:
            # the CPU model and the tensor core still accumulate in different orders (1e-7), which flips a
            # rare gate: tight in L2, an order of magnitude tighter than vs fp32 in max-norm
            assert rel_l2(gp[k].grad, go[k].grad) < 10 * MODEL_TOL, (k, "rel_l2 vs tf32 precision model")
        else:
            e = normwise(gp[k].grad, go[k].grad)
            assert e < MODEL_TOL, (k, "vs tf32 precision model", e)


@pytest.mark.parametrize("seed", list(range(12)))
def test_random_shapes_against_oracle(seed):
    """Seeded sweep over model shapes the BASELINE configs do not hit: odd sensor counts (head dim not a
    multiple of 4), tiny and ragged T, 1..8 classes, with / without statics, random sparse weighted graphs,
    batch sizes around the 128-row tile edges."""
    from oracle.raindrop_oracle import build_oracle_model
    g = torch.Generator().manual_seed(1000 + seed)
    ri = lambda lo, hi: int(torch.randint(lo, hi + 1, (1,), generator=g))
    N, T, B = ri(1, 13), ri(2, 70), [1, 2, 3, 5, 9, 17, 33, 64, 130][ri(0, 8)]
    static = bool(ri(0, 1))
    cfg = dict(name="RND", d_inp=N, max_len=T, d_static=ri(1, 7) if static else 0, n_classes=ri(2, 8), static=static,
               batch=B, p_obs=0.5, d_ob=4, d_model=4 * N, nhid=8 * N, nlayers=ri(1, 3), nhead=2, dropout=0.2, MAX=100)
    if ri(0, 1):
        a = (torch.rand(N, N, generator=g) < 0.4).float() * torch.rand(N, N, generator=g)
        cfg["global_structure"] = a
    batch = make_batch(cfg, B, seed=seed, first_time_zero=bool(ri(0, 1)))
    oracle = build_oracle_model(cfg).eval()
    synth_weights(oracle, cfg, seed=40 + seed)
    shape = {kk: cfg[kk] for kk in ("d_inp", "max_len", "batch", "nlayers", "n_classes", "static")}
    # single-pass TF32 mode vs the oracle under the kernels' rounding model
    ref, _, _ = oracle.forward_dense(batch["src"], batch["static"], batch["times"], batch["lengths"], tf32_model=True)
    F.cross_entropy(ref, batch["y"]).backward()
    model, logits, _, loss, enc_in, _ = _run_dropin(cfg, batch, 40 + seed, mode=FAST)
    assert normwise(logits, ref.detach()) < 2e-4, (cfg, normwise(logits, ref.detach()))
    gp, go = dict(model.named_parameters()), dict(oracle.named_parameters())
    for k in used_param_keys(cfg):
        e = rel_l2(gp[k].grad, go[k].grad)
        assert e < 5e-2, (k, e, shape)
    # error-compensated mode (what "auto" selects at these sizes) vs the plain fp32 oracle
    oracle.zero_grad()
    ref, _, _ = oracle.forward_dense(batch["src"], batch["static"], batch["times"], batch["lengths"])
    F.cross_entropy(ref, batch["y"]).backward()
    model, logits, _, loss, enc_in, _ = _run_dropin(cfg, batch, 40 + seed, mode=0)
    assert normwise(logits, ref.detach()) < 1e-4, (cfg, normwise(logits, ref.detach()))
    gp = dict(model.named_parameters())
    for k in used_param_keys(cfg):
        e = normwise(gp[k].grad, go[k].grad)
        assert e < GRAD_TOL_EXACT, (k, e, shape)


def test_edge_cases():
    """lengths = 1, a sensor never observed, a sensor always observed, isolated graph node."""
    from oracle.raindrop_oracle import build_oracle_model
    cfg = model_config("TINY", dropout=0.2)
    cfg["global_structure"] = sparse_structure(cfg["d_inp"], 9)
    batch = make_batch(cfg, 6, seed=5)
    batch["lengths"][0] = 1
    batch["times"][1:, 0] = 0
    batch["src"][1:, 0, :] = 0
    N = cfg["d_inp"]
    batch["src"][:, :, 2] = 0; batch["src"][:, :, N + 2] = 0          # never observed
    batch["src"][:, :, N + 3] = (batch["times"] > 0).float()           # always observed
    oracle = build_oracle_model(cfg).eval()
    synth_weights(oracle, cfg, seed=3)
    ref, _, _ = oracle.forward(batch["src"], batch["static"], batch["times"], batch["lengths"])
    model, logits, _, _, _, _ = _run_dropin(cfg, batch, 3)
    assert normwise(logits, ref.detach()) < FWD_TOL


def test_full_size_properties():
    """BASELINE configs[1] at full size (B = 128): size-independent properties."""
    cfg = model_config("P19", dropout=0.2)
    batch = make_batch(cfg, 128, seed=77)
    model = build_dropin(cfg, 4).eval()
    d = to_dev(batch)
    with torch.no_grad():
        a, _, _ = model.forward(d["src"], d["static"], d["times"], d["lengths"])
        b, _, _ = model.forward(d["src"], d["static"], d["times"], d["lengths"])
        assert torch.equal(a, b)                                           # deterministic / idempotent
        h1, _, _ = model.forward(d["src"][:, :64], d["static"][:64], d["times"][:, :64], d["lengths"][:64])
        h2, _, _ = model.forward(d["src"][:, 64:], d["static"][64:], d["times"][:, 64:], d["lengths"][64:])
        assert normwise(torch.cat([h1, h2]), a) < 1e-5                      # samples are independent
        perm = torch.randperm(128, device="cuda")
        p, _, _ = model.forward(d["src"][:, perm], d["static"][perm], d["times"][:, perm], d["lengths"][perm])
        assert normwise(p, a[perm]) < 1e-5                                  # permutation equivariance
    assert torch.isfinite(a).all()


@pytest.mark.parametrize("cfg_name", ["P12", "PAM", "LARGE"])
def test_full_size_other_baseline_configs(cfg_name):
    """BASELINE configs[0], [2] and [4] (per-GPU batch) at FULL size: size-independent properties only
    (finite, deterministic, samples independent, one training step produces finite gradients)."""
    cfg = model_config(cfg_name, dropout=0.2)
    B = cfg["batch"]
    model = build_dropin(cfg, 4).eval()
    model._plan.obprop_mode = FAST     # one arithmetic mode at every batch size (auto switches with the row count)
    d = to_dev(make_batch(cfg, B, seed=31))
    st = lambda sl: None if d["static"] is None else d["static"][sl]
    with torch.no_grad():
        a, _, _ = model.forward(d["src"], d["static"], d["times"], d["lengths"])
        b, _, _ = model.forward(d["src"], d["static"], d["times"], d["lengths"])
        part, _, _ = model.forward(d["src"][:, 5:13], st(slice(5, 13)), d["times"][:, 5:13], d["lengths"][5:13])
    assert a.shape == (B, cfg["n_classes"]) and torch.isfinite(a).all() and torch.equal(a, b)
    assert normwise(part, a[5:13]) < 1e-5
    model.train()
    logits, _, _ = model.forward(d["src"], d["static"], d["times"], d["lengths"])
    F.cross_entropy(logits, d["y"]).backward()
    for p_ in model.used_parameters():
        assert p_.grad is not None and torch.isfinite(p_.grad).all()


def test_whole_validation_set_batch():
    """evaluate_standard pushes the whole validation set through in one batch (code/utils_rd.py:310-320)."""
    cfg = model_config("P19", dropout=0.2)
    model = build_dropin(cfg, 4).eval()
    batch = make_batch(cfg, 3880, seed=9)
    d = to_dev(batch)

    def both():
        with torch.no_grad():
            big, _, _ = model.forward(d["src"], d["static"], d["times"], d["lengths"])
            part, _, _ = model.forward(d["src"][:, 1000:1100], d["static"][1000:1100], d["times"][:, 1000:1100],
                                       d["lengths"][1000:1100])
        return big, part
    model._plan.obprop_mode = FAST           # same arithmetic at every batch size: results are batch-invariant
    big, part = both()
    assert big.shape == (3880, 2) and torch.isfinite(big).all()
    assert normwise(part, big[1000:1100]) < 1e-5
    model._plan.obprop_mode = 0              # auto: B = 3880 streams in single-pass TF32, B = 100 runs error-compensated
    big, part = both()
    assert normwise(part, big[1000:1100]) < 2e-4


# ---- operator level -----------------------------------------------------------------------------
def test_node_scale_and_obprop_operator(golden_dir):
    from raindrop_b200 import functional as RF
    from raindrop_b200.models_rd import Observation_progation
    z = np.load(golden_dir + "/operators.npz")
    x = torch.from_numpy(z["obprop.x"]).cuda()
    ei = torch.from_numpy(z["obprop.edge_index"]).cuda()
    ew = torch.from_numpy(z["obprop.edge_w"]).cuda()
    N, Cc = x.shape
    layer = Observation_progation(in_channels=Cc, out_channels=Cc, heads=1, n_nodes=N, ob_dim=4)
    layer.load_state_dict({k[len("obprop.sd."):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("obprop.sd.")})
    layer = layer.cuda()
    out, (ei2, alpha) = layer(x, p_t=None, edge_index=ei, edge_weights=ew, use_beta=False, edge_attr=None,
                              return_attention_weights=True)
    assert normwise(out, z["obprop.beta0.out"]) < FWD_TOL
    assert torch.equal(ei2.cpu(), torch.from_numpy(z["obprop.beta0.edge_index"]))
    assert np.array_equal(alpha.cpu().numpy(), z["obprop.beta0.alpha"])     # pre-softmax weights, bit exact
    # use_beta=True: pruned edge list (index work: bit exact), alpha and output
    p_t = torch.from_numpy(z["obprop.p_t"]).cuda()
    out_b, (ei_b, alpha_b) = layer(x, p_t=p_t, edge_index=ei, edge_weights=ew, use_beta=True, edge_attr=None,
                                   return_attention_weights=True)
    assert torch.equal(ei_b.cpu(), torch.from_numpy(z["obprop.beta1.edge_index"]))
    assert normwise(alpha_b, z["obprop.beta1.alpha"]) < 1e-5
    assert normwise(out_b, z["obprop.beta1.out"]) < 1e-5
    # rows with no incoming edge are exactly zero, like scatter-add leaves them
    s = RF.node_scale(ei, ew, N).cpu()
    has_in = torch.zeros(N, dtype=torch.bool)
    has_in[ei[1].cpu()] = True
    assert torch.all((s == 0) == ~has_in)
    # operator backward vs autograd of the closed form
    xr = x.clone().requires_grad_(True)
    o = RF.ObPropLayerFunction.apply(xr, layer.lin_value.weight, layer.lin_value.bias, s.cuda(), N)
    w = torch.randn_like(o)
    (o * w).sum().backward()
    from oracle.raindrop_oracle import round_tf32
    xc = round_tf32(x.detach().cpu()).double().requires_grad_(True)          # the operator rounds x and W to TF32
    W = round_tf32(layer.lin_value.weight.detach().cpu()).double().requires_grad_(True)
    bb = layer.lin_value.bias.detach().cpu().double().requires_grad_(True)
    oc = F.relu(xc @ W.T + bb) * s.double()[:, None]
    (oc * w.cpu().double()).sum().backward()
    assert normwise(xr.grad, xc.grad) < MODEL_TOL
    assert normwise(layer.lin_value.weight.grad, W.grad) < MODEL_TOL
    assert normwise(layer.lin_value.bias.grad, bb.grad) < MODEL_TOL


@pytest.mark.parametrize("rows,Cc", [(34 * 3, 240), (500, 860), (129, 16), (257, 1024), (40, 2400), (1000, 64)])
def test_obprop_layer_shapes(rows, Cc):
    """Tensor-core layer kernel on the channel widths of every BASELINE config, ragged row counts."""
    from raindrop_b200 import functional as RF
    g = torch.Generator().manual_seed(rows + Cc)
    x = torch.randn(rows, Cc, generator=g)
    W = torch.randn(Cc, Cc, generator=g) / Cc ** 0.5
    b = torch.randn(Cc, generator=g) * 0.1
    s = torch.rand(17, generator=g)
    ref = F.relu(x.double() @ W.double().T + b.double()) * s.double()[torch.arange(rows) % 17][:, None]
    out = RF.ObPropLayerFunction.apply(x.cuda(), W.cuda(), b.cuda(), s.cuda(), 17)
    assert normwise(out, ref) < FWD_TOL


@pytest.mark.parametrize("rows,in_f,out_f", [(7680, 152, 456), (7680, 152, 152), (7680, 272, 152), (300, 160, 288),
                                              (1000, 84, 252), (129, 528, 1584), (64, 186, 186)])
def test_projection_gemm_is_fp32_accurate(rows, in_f, out_f):
    """Error-compensated tensor-core GEMM (3xTF32) vs fp64: must be at fp32 level, not TF32 level."""
    from raindrop_b200 import functional as RF
    g = torch.Generator().manual_seed(rows + in_f)
    x = torch.randn(rows, in_f, generator=g)
    W = torch.randn(out_f, in_f, generator=g) / in_f ** 0.5
    b = torch.randn(out_f, generator=g)
    ref = F.relu(x.double() @ W.double().T + b.double())
    out = RF.linear(x.cuda(), W.cuda(), b.cuda(), relu=True)
    fp32 = F.relu(x @ W.T + b)
    e, e32 = normwise(out, ref), normwise(fp32, ref)
    assert e < 1e-5 and e < 20 * e32 + 1e-7, (e, e32)   # TF32 alone would be ~5e-4


@pytest.mark.parametrize("rows,Cc", [(1000, 240), (4352, 240), (700, 860), (300, 64)])
def test_obprop_operator_backward_weight_grads(rows, Cc):
    """rd_obprop_bwd at sizes that take the tensor-core weight-gradient kernel (3xTF32, split over rows):
    dW and db must be fp32-accurate given the same forward output."""
    from oracle.raindrop_oracle import round_tf32
    from raindrop_b200 import functional as RF
    g = torch.Generator().manual_seed(rows * 3 + Cc)
    x = round_tf32(torch.randn(rows, Cc, generator=g))
    W = round_tf32(torch.randn(Cc, Cc, generator=g) / Cc ** 0.5)
    b = torch.randn(Cc, generator=g) * 0.1
    s = torch.rand(17, generator=g) + 0.5
    xr, Wr, br = x.cuda().requires_grad_(True), W.cuda().requires_grad_(True), b.cuda().requires_grad_(True)
    out = RF.ObPropLayerFunction.apply(xr, Wr, br, s.cuda(), 17)
    w = torch.randn(rows, Cc, generator=g)
    (out * w.cuda()).sum().backward()
    # reference gradient given the SAME gate pattern (out > 0), in fp64
    gate = (out.detach().cpu() > 0).double()
    dpre = w.double() * s.double()[torch.arange(rows) % 17][:, None] * gate
    assert normwise(Wr.grad, dpre.T @ x.double()) < 1e-5
    assert normwise(br.grad, dpre.sum(0)) < 1e-5
    assert normwise(xr.grad, dpre @ W.double()) < 1e-5      # CUDA-core path for d_x in the operator


def test_positional_encoding():
    from oracle.raindrop_oracle import positional_encoding
    from raindrop_b200.models_rd import PositionalEncodingTF
    for max_len in (60, 215, 600):
        t = torch.rand(max_len, 7) * 50
        pe = PositionalEncodingTF(16, max_len, 100)(t)
        assert pe.is_cuda and normwise(pe, positional_encoding(t, max_len)) < 1e-5


def test_transformer_conv(golden_dir):
    from raindrop_b200.models_rd import TransformerConv
    z = np.load(golden_dir + "/operators.npz")
    x = torch.from_numpy(z["tconv.x"]).cuda()
    ei = torch.from_numpy(z["obprop.edge_index"]).cuda()
    ew = torch.from_numpy(z["obprop.edge_w"]).cuda()
    for tag, heads, w in (("tconv.w.", 1, ew), ("tconv.qk.", 2, None)):
        conv = TransformerConv(in_channels=7, out_channels=5, heads=heads)
        conv.load_state_dict({k[len(tag + "sd."):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(tag + "sd.")})
        conv = conv.cuda()
        out, (_, alpha) = conv(x, edge_index=ei, edge_weights=w, edge_attr=None, return_attention_weights=True)
        assert normwise(out, z[tag + "out"]) < 1e-5
        assert normwise(alpha, z[tag + "alpha"]) < 1e-5


def test_graph_operator_gradients(golden_dir):
    """Backward of Observation_progation (use_beta both ways) and TransformerConv (supplied edge weights / q.k
    attention) against gradient fixtures produced by the reference's own layers (oracle/make_golden.py
    operator_grad_cases): loss = sum(out * G) [+ sum(alpha * g)]."""
    from raindrop_b200.models_rd import Observation_progation, TransformerConv
    z = np.load(golden_dir + "/operators.npz")
    zg = np.load(golden_dir + "/operators_grad.npz")
    ei = torch.from_numpy(z["obprop.edge_index"]).cuda()
    N, Cc = z["obprop.x"].shape
    layer = Observation_progation(in_channels=Cc, out_channels=Cc, heads=1, n_nodes=N, ob_dim=4)
    layer.load_state_dict({k[len("obprop.sd."):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("obprop.sd.")})
    layer = layer.cuda()
    G = torch.from_numpy(zg["obprop.G"]).cuda()
    for ub in (False, True):
        tag = "obprop.beta%d." % int(ub)
        layer.zero_grad()
        x = torch.from_numpy(z["obprop.x"]).cuda().requires_grad_(True)
        p_t = torch.from_numpy(z["obprop.p_t"]).cuda().requires_grad_(True)
        ew = torch.from_numpy(z["obprop.edge_w"]).cuda().requires_grad_(True)
        out, (ei2, alpha) = layer(x, p_t=p_t, edge_index=ei, edge_weights=ew, use_beta=ub, edge_attr=None,
                                  return_attention_weights=True)
        assert normwise(out, z[tag + "out"]) < 1e-5
        loss = (out * G).sum()
        if ub:
            assert torch.equal(ei2.cpu(), torch.from_numpy(z[tag + "edge_index"]))
            loss = loss + (alpha * torch.from_numpy(zg[tag + "g_alpha"]).cuda()).sum()
        loss.backward()
        assert normwise(x.grad, zg[tag + "d_x"]) < 2e-5, (tag, normwise(x.grad, zg[tag + "d_x"]))
        if ub:
            assert normwise(ew.grad, zg[tag + "d_edge_w"]) < 2e-5, normwise(ew.grad, zg[tag + "d_edge_w"])
            assert normwise(p_t.grad, zg[tag + "d_p_t"]) < 2e-5
        else:
            assert np.abs(zg[tag + "d_edge_w"]).max() < 1e-5      # sum of a segment softmax is 1: no gradient to speak of
        params = dict(layer.named_parameters())
        for k in zg.files:
            if k.startswith(tag + "grad."):
                name = k[len(tag + "grad."):]
                assert params[name].grad is not None, name
                assert normwise(params[name].grad, zg[k]) < 2e-5, (tag, name, normwise(params[name].grad, zg[k]))
    xn0 = torch.from_numpy(z["tconv.x"]).cuda()
    for tag, heads, use_w in (("tconv.w.", 1, True), ("tconv.qk.", 2, False)):
        conv = TransformerConv(in_channels=7, out_channels=5, heads=heads)
        conv.load_state_dict({k[len(tag + "sd."):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(tag + "sd.")})
        conv = conv.cuda()
        xn = xn0.clone().requires_grad_(True)
        ew = torch.from_numpy(z["obprop.edge_w"]).cuda().requires_grad_(True)
        out, (_, alpha) = conv(xn, edge_index=ei, edge_weights=ew if use_w else None, edge_attr=None, return_attention_weights=True)
        assert normwise(out, z[tag + "out"]) < 1e-5
        (out * torch.from_numpy(zg[tag + "G"]).cuda()).sum().backward()
        assert normwise(xn.grad, zg[tag + "d_x"]) < 2e-5, (tag, normwise(xn.grad, zg[tag + "d_x"]))
        if use_w:
            assert normwise(ew.grad, zg[tag + "d_edge_w"]) < 2e-5 or np.abs(zg[tag + "d_edge_w"]).max() < 1e-6
        params = dict(conv.named_parameters())
        for k in zg.files:
            if k.startswith(tag + "grad."):
                name = k[len(tag + "grad."):]
                ref = zg[k]
                got = params[name].grad
                if np.abs(ref).max() == 0:
                    assert got is None or float(got.abs().max()) == 0.0, name          # q/k unused when edge weights are supplied
                elif np.abs(ref).max() < 1e-7:
                    assert float(got.abs().max()) < 1e-6, name       # lin_key.bias: a per-target constant shift of the logits, softmax-invariant
                else:
                    assert normwise(got, ref) < 2e-5, (tag, name, normwise(got, ref))
    # batched form: many graphs sharing one edge list == the per-graph loop (legacy Raindrop v1, code/models_rd.py:158-166)
    from raindrop_b200 import functional as RF
    Bn, Tn = 5, 9
    xb = torch.randn(Tn, Bn, 7, generator=torch.Generator().manual_seed(1)).cuda().requires_grad_(True)
    src_e = torch.tensor([0, 1, 2, 2, 3, 0]).cuda(); tgt_e = torch.tensor([1, 2, 0, 2, 0, 0]).cuda()
    eib = torch.stack([src_e, tgt_e]); wb = torch.rand(6, generator=torch.Generator().manual_seed(2)).cuda()
    P = [conv.lin_query.weight, conv.lin_query.bias, conv.lin_key.weight, conv.lin_key.bias, conv.lin_value.weight,
         conv.lin_value.bias, conv.lin_skip.weight, conv.lin_skip.bias]
    for p in P:
        p.grad = None         # (they still hold the gradients of the fixture check above)
    ob, _ = RF.transformer_conv(xb.reshape(Tn * Bn, 7), eib, None, 2, 5, *P, geom=(Tn, Bn, Bn, 1))
    Gb = torch.randn(Tn * Bn, 10, generator=torch.Generator().manual_seed(3)).cuda()
    (ob * Gb).sum().backward()
    gb_batched, xb_grad = [p.grad.clone() for p in P], xb.grad.clone()
    for p in P:
        p.grad = None
    xb.grad = None
    outs = []
    for b_ in range(Bn):
        o1, _ = RF.transformer_conv(xb[:, b_, :], eib, None, 2, 5, *P)
        outs.append(o1)
    ol = torch.stack(outs, 1).reshape(Tn * Bn, 10)
    assert normwise(ob, ol) < 1e-6
    (ol * Gb).sum().backward()
    assert normwise(xb_grad, xb.grad) < 1e-5
    scale = max(float(p.grad.abs().max()) for p in P)
    for a_, p in zip(gb_batched, P):      # lin_key.bias is softmax-invariant: both are rounding noise around zero
        assert normwise(a_, p.grad) < 1e-5 or float((a_ - p.grad).abs().max()) < 1e-6 * scale


def test_legacy_raindrop_v1_against_reference(golden_dir):
    """Legacy `Raindrop` v1 (code/models_rd.py:46-191): logits / loss / distance and all 36 gradients vs the fixture
    produced by the reference's own class (oracle/make_golden.py v1_case; weights from the keyed stream, gradients with
    more than 4096 elements stored as fingerprints)."""
    from raindrop_b200.models_rd import Raindrop
    from raindrop_b200.synth import CONFIGS, keyed_values
    z, meta = load_golden(golden_dir, "v1_p12_b3")
    cfg = dict(CONFIGS["P12"]); cfg["name"] = "P12"
    batch = make_batch(dict(cfg, d_ob=2), 3, seed=77)
    model = Raindrop(36, 72, 2, 144, 2, 0.2, 215, 9, 100, 0.5, "mean", 2, torch.from_numpy(z["global_structure"]))
    sd = model.state_dict()
    assert {k: list(v.shape) for k, v in sd.items()} == meta["state_dict"]
    model.load_state_dict({k: keyed_values(meta["weight_seed"], k, tuple(v.shape)) for k, v in sd.items()})
    model = model.cuda().eval()
    d = to_dev(batch)
    logits, distance, third = model.forward(d["src"], d["static"], d["times"], d["lengths"])
    assert third is None and float(distance) == float(z["distance"]) == 0.0
    assert normwise(logits, z["logits"]) < 1e-4, normwise(logits, z["logits"])
    loss = F.cross_entropy(logits, d["y"])
    assert abs(loss.item() - float(z["loss"])) < 1e-4
    loss.backward()
    params = dict(model.named_parameters())
    with_grad = sorted(meta["with_grad"])
    assert sorted(k for k, p in params.items() if p.grad is not None and float(p.grad.abs().max()) > 0) == with_grad
    errs = {}
    for k in with_grad:
        check_against_golden(z, "grad." + k in z.files, "grad." + k, params[k].grad, 2e-3, errs)
    print("v1 worst gradient error", max(errs.items(), key=lambda kv: kv[1]))
    # train mode runs (dropout on the library's stream) and is reproducible for a fixed (seed, counter)
    model.train()
    a, _, _ = model.forward(d["src"], d["static"], d["times"], d["lengths"])
    assert torch.isfinite(a).all() and not torch.equal(a, logits)


def test_device_dataset_gather_is_bit_exact():
    """rd_gather_batch == torch indexing of the host tensors (index work: bit exact), incl. odd widths."""
    from raindrop_b200.train import DeviceDataset, TrainStep
    cfg = model_config("P19", dropout=0.0)
    full = make_batch(cfg, 300, seed=4)
    ds = DeviceDataset(full["src"], full["static"], full["times"], full["y"], "cuda")
    ts = TrainStep(build_dropin(cfg, 2).train(), 64, use_graph=False)
    idx = torch.randperm(300, generator=torch.Generator().manual_seed(1))[:64]
    ds.fill(ts, idx)
    assert torch.equal(ts.src.cpu(), full["src"][:, idx])
    assert torch.equal(ts.times.cpu(), full["times"][:, idx])
    assert torch.equal(ts.static.cpu(), full["static"][idx])
    assert torch.equal(ts.y.cpu(), full["y"][idx]) and torch.equal(ts.lengths.cpu(), full["lengths"][idx])
    l0 = ts.step().item()
    ts2 = TrainStep(build_dropin(cfg, 2).train(), 64, use_graph=False)
    ts2.load_batch(to_dev({k: (v[:, idx] if k in ("src", "times") else v[idx]) for k, v in full.items()}))
    assert ts2.step().item() == l0


def test_cross_entropy_and_adam():
    import ctypes as C
    from raindrop_b200 import lib as L
    lib = L.load()
    g = torch.Generator().manual_seed(0)
    logits = torch.randn(37, 8, generator=g).cuda()
    y = torch.randint(0, 8, (37,), generator=g).cuda()
    loss = torch.zeros(1, device="cuda"); dl = torch.zeros_like(logits)
    L.check(lib.rd_cross_entropy_fwd_bwd(logits.data_ptr(), y.data_ptr(), 37, 8, loss.data_ptr(), dl.data_ptr(),
                                         L.stream_ptr()), "ce")
    lt = logits.clone().requires_grad_(True)
    ref = F.cross_entropy(lt, y); ref.backward()
    assert abs(loss.item() - ref.item()) < 1e-6 and normwise(dl, lt.grad) < 1e-5
    p = torch.randn(1000, generator=g).cuda(); p_ref = torch.nn.Parameter(p.clone())
    opt = torch.optim.Adam([p_ref], lr=1e-2)
    m = torch.zeros_like(p); v = torch.zeros_like(p); step = torch.zeros(2, dtype=torch.int64, device="cuda")   # {count, ticket}
    lr_dev = torch.full((1,), 1e-2, device="cuda")
    for it in range(5):
        grad = torch.randn(1000, generator=g).cuda()
        p_ref.grad = grad.clone(); opt.step()
        # odd iterations read the learning rate from the device scalar (what a captured graph does)
        L.check(lib.rd_adam_step(p.data_ptr(), grad.data_ptr(), m.data_ptr(), v.data_ptr(), 1000, 1e-2 if it % 2 == 0 else 123.0,
                                 None if it % 2 == 0 else lr_dev.data_ptr(), 0.9, 0.999, 1e-8, 1.0, step.data_ptr(),
                                 L.stream_ptr()), "adam")
    assert step.tolist() == [5, 0] and normwise(p, p_ref.detach()) < 1e-5


def test_fused_head_loss_matches_torch_cross_entropy():
    """rd_raindrop_v2_fwd with labels: loss and d(loss)/d(logits) come out of the head kernel (CrossEntropyLoss,
    mean reduction, code/Raindrop.py:322) -- compared with torch on the kernel's own logits, 2 and 8 classes."""
    from raindrop_b200.train import TrainStep
    for name, B in (("P19", 37), ("TINY8", 5)):
        cfg = model_config(name, dropout=0.0)
        ts = TrainStep(build_dropin(cfg, 3).train(), B, use_graph=False)
        ts.load_batch(to_dev(make_batch(cfg, B, seed=9)))
        ts.step()
        lt = ts.logits.clone().requires_grad_(True)
        ref = F.cross_entropy(lt, ts.y); ref.backward()
        assert abs(ts.loss.item() - ref.item()) < 1e-6 * max(1.0, abs(ref.item())), (name, ts.loss.item(), ref.item())
        assert normwise(ts.d_logits, lt.grad) < 1e-5


def test_flat_adam_matches_torch_adam():
    """raindrop_b200.optim.FlatAdam (flat leaf + CUDA-graph-captured forward/backward + one Adam launch) follows the
    same trajectory as torch.optim.Adam on the general autograd path; dropout 0."""
    from raindrop_b200.optim import FlatAdam
    cfg = model_config("P19", dropout=0.0)
    B = 16
    m1 = build_dropin(cfg, 8).train(); m2 = build_dropin(cfg, 8).train()
    o1 = torch.optim.Adam(m1.parameters(), lr=1e-3); o2 = FlatAdam(m2, lr=1e-3)
    sched = torch.optim.lr_scheduler.StepLR(o2, step_size=2, gamma=0.5)        # it is a torch Optimizer
    sched1 = torch.optim.lr_scheduler.StepLR(o1, step_size=2, gamma=0.5)
    for it in range(5):                 # eager call, capture call, then graph replays
        d = to_dev(make_batch(cfg, B, seed=70 + it))
        losses = []
        for m, o in ((m1, o1), (m2, o2)):
            logits, _, _ = m.forward(d["src"], d["static"], d["times"], d["lengths"])
            loss = F.cross_entropy(logits, d["y"])
            o.zero_grad(); loss.backward(); o.step()
            losses.append(loss.item())
        sched.step(); sched1.step()
        assert abs(losses[0] - losses[1]) < 2e-4 * max(1.0, abs(losses[0])), (it, losses)
    slot = m2._plan._slots[(B, True, 0)]
    assert slot.fwd_graph is not None and slot.bwd_graph is not None      # replays happened
    p1, p2 = dict(m1.named_parameters()), dict(m2.named_parameters())
    for k in used_param_keys(cfg):
        assert rel_l2(p2[k], p1[k]) < 5e-3, k
        assert p2[k].grad is not None and normwise(p2[k].grad, p1[k].grad) < 2e-2, k    # .grad = window of the bucket
    # a no-grad probe between forward and backward must not disturb the pending step
    d = to_dev(make_batch(cfg, B, seed=99))
    logits, _, _ = m2.forward(d["src"], d["static"], d["times"], d["lengths"])
    with torch.no_grad():
        probe, _, _ = m2.forward(d["src"], d["static"], d["times"], d["lengths"])
    assert normwise(probe, logits) < 1e-6
    F.cross_entropy(logits, d["y"]).backward()
    g_a = o2.flat_g.clone()
    logits, _, _ = m2.forward(d["src"], d["static"], d["times"], d["lengths"])
    F.cross_entropy(logits, d["y"]).backward()
    assert torch.equal(g_a, o2.flat_g)
    # checkpoints still round-trip through the module (parameters are views of the flat leaf)
    sd = {k: v.clone() for k, v in m2.state_dict().items()}
    m2.load_state_dict(sd)
    assert all(torch.equal(v, m2.state_dict()[k]) for k, v in sd.items())


def test_default_capture_has_no_side_effects():
    """TrainStep.step() with the DEFAULT implicit capture (3 warm-up iterations) must give the same trajectory as
    the eager loop: warm-up is snapshotted/restored (parameters, Adam moments, step count, dropout stream)."""
    from raindrop_b200.train import TrainStep
    cfg = model_config("P19", dropout=0.2)
    B = 16
    a = TrainStep(build_dropin(cfg, 4).train(), B, lr=1e-3, use_graph=True)
    b = TrainStep(build_dropin(cfg, 4).train(), B, lr=1e-3, use_graph=False)
    for it in range(3):
        d = to_dev(make_batch(cfg, B, seed=30 + it))
        a.load_batch(d); b.load_batch(d)
        la, lb = a.step().item(), b.step().item()
        assert la == lb, (it, la, lb)
    assert torch.equal(a.flat_p, b.flat_p) and a.step_count.tolist() == [3, 0]
    # learning rate lives on the device: changing it after capture takes effect
    a.set_lr(0.0); b.set_lr(0.0)
    before = a.flat_p.clone()
    a.step(); b.step()
    assert torch.equal(a.flat_p, before) and torch.equal(b.flat_p, before)


@pytest.mark.parametrize("shapes", [[(7680, 456, 152), (7680, 152, 152), (7680, 272, 152), (7680, 152, 272), (4352, 240, 240)],
                                    [(300, 16, 64)], [(1000, 288, 160), (5000, 64, 1024), (777, 860, 860)]])
def test_grouped_weight_gradients(shapes):
    """rd_linear_wgrad_group: several dW = dY^T X (+ db) problems in ONE tensor-core launch, fp32-accurate."""
    import ctypes as C
    from raindrop_b200 import lib as L
    lib = L.load()
    g = torch.Generator().manual_seed(3)
    items = (L.RdWgradItem * len(shapes))()
    keep, outs = [], []
    for i, (rows, nout, kin) in enumerate(shapes):
        dY = torch.randn(rows, nout, generator=g).cuda(); X = torch.randn(rows, kin, generator=g).cuda()
        dW = torch.empty(nout, kin, device="cuda"); db = torch.empty(nout, device="cuda")
        part = torch.empty(lib.rd_linear_wgrad_partial_bytes(rows, nout, kin) // 4, device="cuda")
        items[i].d_out, items[i].x, items[i].rows, items[i].out_features, items[i].in_features = dY.data_ptr(), X.data_ptr(), rows, nout, kin
        items[i].d_weight, items[i].d_bias, items[i].partial = dW.data_ptr(), db.data_ptr(), part.data_ptr()
        keep.append((dY, X, part)); outs.append((dW, db))
    L.check(lib.rd_linear_wgrad_group(items, len(shapes), L.stream_ptr()), "rd_linear_wgrad_group")
    for (dY, X, _), (dW, db) in zip(keep, outs):
        ref = dY.double().T @ X.double()
        assert normwise(dW, ref) < 2e-5, normwise(dW, ref)
        assert normwise(db, dY.double().sum(0)) < 2e-5


@pytest.mark.parametrize("B,H,T,hd", [(5, 2, 60, 76), (3, 2, 10, 20), (2, 4, 64, 96), (4, 1, 33, 8), (130, 2, 60, 76)])
def test_temporal_attention_operator(B, H, T, hd):
    """rd_temporal_attention_fwd/_bwd (tcgen05 kernels) vs an fp64 torch restatement of the masked softmax attention
    of nn.TransformerEncoderLayer (code/models_rd.py:358), and vs the CUDA-core kernels under dropout (same
    counter-based masks -> same result)."""
    from raindrop_b200 import lib as L
    lib = L.load()
    g = torch.Generator().manual_seed(B * 1000 + T)
    D = H * hd
    qkv = torch.randn(T, B, 3 * D, generator=g).cuda()
    dctx = torch.randn(T, B, D, generator=g).cuda()
    lengths = torch.randint(1, T + 1, (B,), generator=g).cuda()
    lengths[0] = T
    rng = torch.tensor([12345, 7], dtype=torch.int64, device="cuda")

    def run(impl, p):
        ctx = torch.full((T, B, D), float("nan"), device="cuda"); dq = torch.full((T, B, 3 * D), float("nan"), device="cuda")
        L.check(lib.rd_temporal_attention_fwd(qkv.data_ptr(), lengths.data_ptr(), B, H, T, hd, p, rng.data_ptr(), 16, impl,
                                              ctx.data_ptr(), L.stream_ptr()), "attn fwd")
        L.check(lib.rd_temporal_attention_bwd(qkv.data_ptr(), dctx.data_ptr(), lengths.data_ptr(), B, H, T, hd, p,
                                              rng.data_ptr(), 16, impl, dq.data_ptr(), L.stream_ptr()), "attn bwd")
        torch.cuda.synchronize()
        return ctx, dq

    ctx, dq = run(1, 0.0)
    x = qkv.double().requires_grad_(True)
    q, k, v = (x[:, :, i * D:(i + 1) * D].reshape(T, B, H, hd).permute(1, 2, 0, 3) for i in range(3))
    s = q @ k.transpose(-1, -2) / hd ** 0.5
    mask = torch.arange(T, device="cuda")[None, :] >= lengths[:, None]
    s = s.masked_fill(mask[:, None, None, :], float("-inf"))
    ref = (torch.softmax(s, -1) @ v).permute(2, 0, 1, 3).reshape(T, B, D)
    ref.backward(dctx.double())
    assert normwise(ctx, ref) < 2e-5, normwise(ctx, ref)
    assert normwise(dq, x.grad) < 2e-5, normwise(dq, x.grad)
    if T <= 64 and hd <= 96:
        for p in (0.0, 0.2):
            c1, d1 = run(1, p); c2, d2 = run(2, p)
            assert normwise(c1, c2) < 2e-5 and normwise(d1, d2) < 2e-5, (p, normwise(c1, c2), normwise(d1, d2))


# ---- training mode --------------------------------------------------------------------------------
def test_train_mode_dropout_statistics_and_replay():
    """Dropout cannot match the reference's RNG stream; check keep-rate, determinism under the same
    (seed, counter) and that backward uses exactly the forward's masks (finite-difference free check:
    with p -> masks replayed via rd_debug_dropout_mask the lifted input matches)."""
    import ctypes as C
    from raindrop_b200 import functional as RF
    from raindrop_b200 import lib as L
    cfg = model_config("P19", dropout=0.2)
    batch = make_batch(cfg, 16, seed=1)
    model = build_dropin(cfg, 2).train()
    model._plan.debug_keep_workspace = True
    d = to_dev(batch)
    out1, _, _ = model.forward(d["src"], d["static"], d["times"], d["lengths"])
    x0_train = RF.workspace_view(model._plan, L.WS_X0).clone()
    rng = RF.workspace_view(model._plan, L.WS_RNG).clone()
    out2, _, _ = model.forward(d["src"], d["static"], d["times"], d["lengths"])
    assert not torch.equal(out1, out2)                       # counter advanced -> new masks
    model.eval()
    with torch.no_grad():
        model.forward(d["src"], d["static"], d["times"], d["lengths"])
    x0_eval = RF.workspace_view(model._plan, L.WS_X0).clone()
    nz = x0_eval != 0
    kept = (x0_train[nz] != 0).float().mean().item()
    assert abs(kept - 0.8) < 0.01, kept
    assert torch.allclose(x0_train[nz][x0_train[nz] != 0], (x0_eval[nz] / 0.8)[x0_train[nz] != 0], rtol=2e-3)  # X0 is stored TF32-rounded
    # replay the lift mask through the debug entry point: index space is [T, B, 4N]
    T, B, D4 = 60, 16, cfg["d_inp"] * 4
    mask = torch.empty(T * B * D4, device="cuda")
    lib = L.load()
    L.check(lib.rd_debug_dropout_mask(rng.data_ptr(), L.SITE_LIFT, mask.numel(), C.c_float(0.2), mask.data_ptr(),
                                      L.stream_ptr()), "mask")
    mask = mask.view(T, B, cfg["d_inp"], 4).permute(1, 2, 0, 3).reshape(B * cfg["d_inp"], T * 4)
    assert torch.allclose(x0_train.view_as(mask), x0_eval.view_as(mask) * mask, rtol=2e-3)


def test_train_step_matches_autograd_loop():
    """TrainStep (C ABI + CUDA graph) == the reference-style loop (autograd + torch.optim.Adam), dropout 0."""
    from raindrop_b200.train import TrainStep
    cfg = model_config("P19", dropout=0.0)
    B = 32
    m1 = build_dropin(cfg, 6).train()
    m2 = build_dropin(cfg, 6).train()
    opt = torch.optim.Adam(m1.parameters(), lr=1e-3)
    ts = TrainStep(m2, B, lr=1e-3, use_graph=True)
    with torch.no_grad():   # one-time kernel attribute setup must not happen inside the capture
        d0 = to_dev(make_batch(cfg, B, seed=49))
        m1.forward(d0["src"], d0["static"], d0["times"], d0["lengths"])
    ts.capture(warmup=0)
    for it in range(4):
        batch = make_batch(cfg, B, seed=50 + it)
        d = to_dev(batch)
        logits, _, _ = m1.forward(d["src"], d["static"], d["times"], d["lengths"])
        loss = F.cross_entropy(logits, d["y"])
        opt.zero_grad(); loss.backward(); opt.step()
        ts.load_batch(d)
        l2 = ts.step()
        assert abs(l2.item() - loss.item()) < 2e-4 * max(1.0, abs(loss.item())), (it, l2.item(), loss.item())
    p1, p2 = dict(m1.named_parameters()), dict(m2.named_parameters())
    # Same kernels, but torch.optim.Adam and rd_adam_step round differently (1e-7); a weight that sits on
    # a TF32 rounding boundary then rounds the other way, which Adam's sign-like update amplifies at
    # isolated entries.  The trajectories must still agree in the mean.
    for k in used_param_keys(cfg):
        assert rel_l2(p2[k], p1[k]) < 5e-3, k


def test_dropin_checkpoint_roundtrip():
    """state_dict from the oracle (== reference keys/shapes) loads into the drop-in and back."""
    from oracle.raindrop_oracle import build_oracle_model
    cfg = model_config("P19", dropout=0.2)
    oracle = build_oracle_model(cfg)
    model = build_dropin(cfg, 1)
    model.load_state_dict(oracle.state_dict())
    back = model.state_dict()
    assert list(back.keys()) == list(oracle.state_dict().keys())
    for k, v in oracle.state_dict().items():
        assert torch.equal(back[k].cpu(), v)


def test_two_gpu_equals_one_gpu():
    """N-rank sample-sharded TrainStep (NCCL all-reduce of the flat bucket, eager and CUDA-graph) == 1 rank."""
    import os
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(root, "tools", "ddp_check.py")],
                       capture_output=True, text=True, timeout=600)
    assert "DDP_CHECK_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]

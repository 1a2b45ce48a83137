"""Gradients with respect to the float inputs of Raindrop_v2 (src, static, times) and the attribution helpers built on
them (raindrop_b200.attribution).  References: tests/golden/input_grads.npz (the reference's own files,
tools/make_input_grad_golden.py), the CPU oracle through autograd, and central differences in train mode."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import build_dropin, case_setup, check_against_golden, load_golden, normwise, rel_l2, to_dev
from raindrop_b200.synth import make_batch, model_config, synth_weights, used_param_keys

GOLDEN_CASES = ["tiny_dense", "tiny_t0", "tiny_sparse", "tiny8_nostatic", "p19_b4", "p19_b5_leave10", "p12_b2", "pam_b2"]
EXACT, FAST = 2, 1
# error-compensated ob-prop GEMMs: fp32-level; the widest layers (C >= 1024) at B = 2..3 flip an occasional ReLU gate
GRAD_TOL_EXACT, GRAD_TOL_EXACT_WIDE = 2e-3, 1e-2
# single-pass TF32: a ReLU gate upstream can flip, so the fast mode is checked in relative L2 (as lin_value is)
FAST_SRC_L2, FAST_TOL = 5e-2, 2e-2
# Input gradients are per sample: one ReLU gate that flips between two fp32 implementations (a pre-activation within
# ~1e-6 of zero, which a few thousand rows make likely) moves one (sample, sensor) row of d_src, or one sample's d_times,
# by ~1e-3..1e-2 of max|grad| (parameter gradients average it over the batch).  At the larger batches the oracle
# comparison is therefore relative L2, with a max-norm bound for the isolated rows.
SIZE_L2, SIZE_MAX = 2e-3, 2e-2


def _exact_tol(cfg):
    return GRAD_TOL_EXACT_WIDE if cfg["max_len"] * cfg["d_ob"] >= 1024 else GRAD_TOL_EXACT


def _oracle_input_grads(cfg, batch, weight_seed):
    """Input gradients of the fp32 oracle (autograd through forward_dense) of the batch's cross-entropy loss."""
    from oracle.raindrop_oracle import build_oracle_model
    oracle = build_oracle_model(cfg).eval()
    synth_weights(oracle, cfg, seed=weight_seed)
    src = batch["src"].clone().requires_grad_(True)
    times = batch["times"].clone().requires_grad_(True)
    static = None if batch["static"] is None else batch["static"].clone().requires_grad_(True)
    logits, _, _ = oracle.forward_dense(src, static, times, batch["lengths"])
    F.cross_entropy(logits, batch["y"]).backward()
    return src.grad, (static.grad if static is not None else None), times.grad


def _dropin_input_grads(cfg, batch, weight_seed, mode=0, frozen=False, model=None):
    """(model, logits, d_src, d_static, d_times) of the CUDA path for the batch's cross-entropy loss."""
    if model is None:
        model = build_dropin(cfg, weight_seed).eval()
        model._plan.obprop_mode = mode
    if frozen:
        for p in model.parameters():
            p.requires_grad_(False)
    d = to_dev(batch)
    src = d["src"].clone().requires_grad_(True)
    times = d["times"].clone().requires_grad_(True)
    static = None if d["static"] is None else d["static"].clone().requires_grad_(True)
    logits, _, _ = model.forward(src, static, times, d["lengths"])
    F.cross_entropy(logits, d["y"]).backward()
    return model, logits, src.grad, (static.grad if static is not None else None), times.grad


# ---- CPU -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_oracle_input_grads_match_reference(golden_dir, name):
    """The oracle (autograd through forward_dense) reproduces the reference's own input gradients."""
    z = np.load(golden_dir + "/input_grads.npz")
    _, meta = load_golden(golden_dir, name)
    cfg, batch = case_setup(meta)
    d_src, d_static, d_times = _oracle_input_grads(cfg, batch, meta["weight_seed"])
    errs = {}
    for key, t in (("d_src", d_src), ("d_static", d_static), ("d_times", d_times)):
        if t is None:
            assert not any(k.startswith(name + "/" + key) for k in z.files)
            continue
        check_against_golden(z, meta["full_tensors"], name + "/" + key, t, 1e-5, errs)


# ---- GPU -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", [EXACT, FAST], ids=["exact", "fast"])
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_golden_input_grads(golden_dir, name, mode):
    """d_src, d_static and d_times of the CUDA path against the reference's own files, in both ob-prop modes."""
    z = np.load(golden_dir + "/input_grads.npz")
    _, meta = load_golden(golden_dir, name)
    cfg, batch = case_setup(meta)
    _, _, d_src, d_static, d_times = _dropin_input_grads(cfg, batch, meta["weight_seed"], mode=mode)
    full = meta["full_tensors"]
    errs = {}
    assert (d_static is None) == (not cfg["static"])
    for key, t in (("d_src", d_src), ("d_static", d_static), ("d_times", d_times)):
        if t is None:
            continue
        if mode == EXACT:
            check_against_golden(z, full, name + "/" + key, t, _exact_tol(cfg), errs)
        else:
            tol = FAST_SRC_L2 if key == "d_src" else FAST_TOL
            check_against_golden(z, full, name + "/" + key, t, tol * (1 if full else 2), errs, metric=rel_l2)
    print(name, "mode", mode, errs)


def _check_exact_vs_oracle(cfg, batch, seed, mode=EXACT):
    ref = _oracle_input_grads(cfg, batch, seed)
    _, _, *got = _dropin_input_grads(cfg, batch, seed, mode=mode)
    errs = {}
    for key, g, r in zip(("d_src", "d_static", "d_times"), got, ref):
        assert (g is None) == (r is None), key
        if r is not None:
            errs[key] = (normwise(g, r), rel_l2(g, r))
    assert all(l2 < SIZE_L2 and mx < SIZE_MAX for mx, l2 in errs.values()), (cfg["name"], errs)
    return errs


@pytest.mark.gpu
@pytest.mark.parametrize("cfg_name,B", [("P19", 37), ("P19", 128), ("P12", 5), ("PAM", 3), ("LARGE", 2)])
def test_input_grads_against_oracle(cfg_name, B):
    cfg = model_config(cfg_name, dropout=0.2)
    batch = make_batch(cfg, B, seed=300 + B, zero_sensors=3 if cfg_name == "P19" else 0)
    print(cfg_name, B, _check_exact_vs_oracle(cfg, batch, 31))


@pytest.mark.gpu
@pytest.mark.parametrize("seed", list(range(12)))
def test_input_grads_random_shapes(seed):
    """The random-shape sweep of the parity tests (T <= 3 gives C < 16: the CUDA-core fallback of the lift backward);
    automatic mode, which is error-compensated at these sizes."""
    g = torch.Generator().manual_seed(1000 + seed)
    ri = lambda lo, hi: int(torch.randint(lo, hi + 1, (1,), generator=g))
    N, T, B = ri(1, 13), ri(2, 70), [1, 2, 3, 5, 9, 17, 33, 64, 130][ri(0, 8)]
    static = bool(ri(0, 1))
    cfg = dict(name="RND", d_inp=N, max_len=T, d_static=ri(1, 7) if static else 0, n_classes=ri(2, 8), static=static,
               batch=B, p_obs=0.5, d_ob=4, d_model=4 * N, nhid=8 * N, nlayers=ri(1, 3), nhead=2, dropout=0.2, MAX=100)
    if ri(0, 1):
        cfg["global_structure"] = (torch.rand(N, N, generator=g) < 0.4).float() * torch.rand(N, N, generator=g)
    batch = make_batch(cfg, B, seed=seed, first_time_zero=bool(ri(0, 1)))
    print(dict(N=N, T=T, B=B, static=static), _check_exact_vs_oracle(cfg, batch, 40 + seed, mode=0))


@pytest.mark.gpu
def test_input_grad_fallback_small_C():
    """C = T * 4 < 16: the lift backward runs on the CUDA cores (no tensor-core kernel for that width)."""
    cfg = model_config("TINY", dropout=0.2)
    cfg.update(max_len=3)
    batch = make_batch(cfg, 5, seed=8)
    _check_exact_vs_oracle(cfg, batch, 9, mode=0)


@pytest.mark.gpu
def test_input_grads_exact_zeros():
    """Exactly zero where the reference's are: the mask half of src, values that are 0 (unobserved, padding, left-out
    sensors: relu'(0) = 0) and d_times at padded steps."""
    cfg = model_config("P19", dropout=0.2)
    batch = make_batch(cfg, 24, seed=77, zero_sensors=5)
    for mode in (EXACT, FAST):
        _, _, d_src, _, d_times = _dropin_input_grads(cfg, batch, 5, mode=mode)
        N = cfg["d_inp"]
        src = batch["src"].cuda()
        assert torch.count_nonzero(d_src[..., N:]) == 0
        assert torch.count_nonzero(d_src[..., :N][src[..., :N] == 0]) == 0
        assert torch.count_nonzero(d_src[..., :N]) > 0
        T = cfg["max_len"]
        pad = torch.arange(T)[:, None] >= batch["lengths"][None, :]
        assert torch.count_nonzero(d_times[pad.cuda()]) == 0
        assert torch.count_nonzero(d_times[~pad.cuda()]) > 0


def _grads_bits(model):
    return {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [EXACT, FAST], ids=["exact", "fast"])
def test_parameter_grads_bit_identical_with_input_grads(mode):
    """Asking for input gradients changes neither the logits nor any of the 34 parameter gradients by one bit."""
    cfg = model_config("P19", dropout=0.2)
    d = to_dev(make_batch(cfg, 64, seed=3))
    out = []
    for want in (False, True):
        model = build_dropin(cfg, 4).train()
        model._plan.obprop_mode = mode
        src = d["src"].clone().requires_grad_(want)
        logits, _, _ = model.forward(src, d["static"], d["times"], d["lengths"])
        F.cross_entropy(logits, d["y"]).backward()
        assert (src.grad is not None) == want
        out.append((logits.detach(), _grads_bits(model)))
    assert torch.equal(out[0][0], out[1][0])
    assert sorted(out[0][1]) == sorted(out[1][1]) == sorted(used_param_keys(cfg))
    for k in out[0][1]:
        assert torch.equal(out[0][1][k], out[1][1][k]), k


@pytest.mark.gpu
def test_frozen_model_input_grads_skip_parameter_work():
    """Frozen parameters: the same input gradients, bit for bit, without the parameter-gradient launches."""
    from raindrop_b200 import lib as L
    lib = L.load()
    cfg = model_config("P19", dropout=0.2)
    batch = make_batch(cfg, 128, seed=12)
    res, launches = [], []
    for frozen in (False, True):
        model = build_dropin(cfg, 6).eval()
        model._plan.obprop_mode = EXACT
        _dropin_input_grads(cfg, batch, 6, model=model, frozen=frozen)     # warm-up (one-time kernel set-up)
        d = to_dev(batch)
        src = d["src"].clone().requires_grad_(True)
        times = d["times"].clone().requires_grad_(True)
        static = d["static"].clone().requires_grad_(True)
        logits, _, _ = model.forward(src, static, times, d["lengths"])
        loss = F.cross_entropy(logits, d["y"])
        n0 = lib.rd_launch_count()
        loss.backward()
        launches.append(lib.rd_launch_count() - n0)
        res.append((src.grad, static.grad, times.grad))
        assert all(p.grad is None for p in model.parameters()) == frozen
    for a, b in zip(*res):
        assert torch.equal(a, b)
    print("backward launches: full %d, input-only %d" % tuple(launches))
    # head parameter outputs, the grouped weight-gradient launch and its reduction are gone
    assert launches[0] - launches[1] >= 3, launches


@pytest.mark.gpu
def test_train_mode_dropout_central_difference():
    """Train mode with dropout, error-compensated mode: <d_src, v> against a central difference of the logits with the
    dropout stream rewound before every forward (checks the X0 != 0 gate and the 1 / (1 - p) scale)."""
    cfg = model_config("P19", dropout=0.2)
    d = to_dev(make_batch(cfg, 4, seed=21))
    model = build_dropin(cfg, 2).train()
    model._plan.obprop_mode = EXACT
    with torch.no_grad():
        model.forward(d["src"], d["static"], d["times"], d["lengths"])      # creates the dropout stream state
    rng0 = model._plan.rng_state.clone()

    def f(src, grad=False):
        model._plan.rng_state.copy_(rng0)
        with torch.set_grad_enabled(grad):
            logits, _, _ = model.forward(src, d["static"], d["times"], d["lengths"])
        return logits[:, 0].double().sum() if not grad else logits[:, 0].sum()

    src = d["src"].clone().requires_grad_(True)
    (g,) = torch.autograd.grad(f(src, grad=True), src)
    N = cfg["d_inp"]
    # observed values away from the lift's own kink (relu(v * R_u) at v = 0), so that +-eps v crosses no gate there
    observed = d["src"][..., :N].abs() > 0.05
    gen = torch.Generator(device="cuda").manual_seed(5)
    eps = 1e-3
    for _ in range(3):
        # random magnitudes on a random half of the observed values, signed like the gradient so that <d_src, v> is far
        # above the fp32 rounding of the logits divided by 2 eps (a direction orthogonal to d_src measures only that)
        pick = observed & (torch.rand(observed.shape, generator=gen, device="cuda") < 0.5)
        v = torch.zeros_like(d["src"])
        v[..., :N] = torch.randn(observed.shape, generator=gen, device="cuda").abs() * g[..., :N].sign() * pick
        an = float((g.double() * v.double()).sum())
        fd = float((f(d["src"] + eps * v) - f(d["src"] - eps * v)) / (2 * eps))
        assert abs(an - fd) <= 1e-2 * abs(an), (an, fd)


@pytest.mark.gpu
def test_flat_adam_input_grads():
    """FlatAdam-bound model (graph-captured forward / backward): the same src.grad as the general path, and the same
    parameter update as a step without input gradients."""
    from raindrop_b200.optim import FlatAdam
    cfg = model_config("P19", dropout=0.0)
    B = 16
    general = build_dropin(cfg, 8).train()
    m_in, m_plain = build_dropin(cfg, 8).train(), build_dropin(cfg, 8).train()
    o_in, o_plain = FlatAdam(m_in, lr=1e-3), FlatAdam(m_plain, lr=1e-3)
    for it in range(4):                 # eager call, capture call, then graph replays
        d = to_dev(make_batch(cfg, B, seed=90 + it))
        general.load_state_dict(m_in.state_dict())       # same (updated) parameters on the general path
        grads = []
        for m in (general, m_in):
            src = d["src"].clone().requires_grad_(True)
            logits, _, _ = m.forward(src, d["static"], d["times"], d["lengths"])
            F.cross_entropy(logits, d["y"]).backward()
            assert src.grad is not None
            grads.append(src.grad)
        general.zero_grad()
        assert normwise(grads[1], grads[0]) < 1e-5, it
        logits, _, _ = m_plain.forward(d["src"], d["static"], d["times"], d["lengths"])
        F.cross_entropy(logits, d["y"]).backward()
        o_in.step(); o_plain.step()
        assert torch.equal(o_in.flat_p, o_plain.flat_p), it
    assert m_in._plan._slots[(B, True, 0)].fwd_graph is not None      # the forward ran as a graph replay


@pytest.mark.gpu
def test_autograd_grad_and_saliency():
    """torch.autograd.grad(logits.sum(), src) works; saliency() equals the autograd result on the target logits."""
    from raindrop_b200.attribution import saliency
    cfg = model_config("P19", dropout=0.2)
    d = to_dev(make_batch(cfg, 32, seed=4))
    model = build_dropin(cfg, 3).eval()
    src = d["src"].clone().requires_grad_(True)
    logits, _, _ = model.forward(src, d["static"], d["times"], d["lengths"])
    (g,) = torch.autograd.grad(logits.sum(), src)
    assert g.shape == src.shape and torch.count_nonzero(g) > 0
    src = d["src"].clone().requires_grad_(True)
    times = d["times"].clone().requires_grad_(True)
    static = d["static"].clone().requires_grad_(True)
    logits, _, _ = model.forward(src, static, times, d["lengths"])
    target = logits.detach().argmax(1)
    gs, gst, gt = torch.autograd.grad(logits.gather(1, target[:, None]).sum(), (src, static, times))
    sal = saliency(model, d["src"], d["static"], d["times"], d["lengths"])
    N = cfg["d_inp"]
    assert torch.equal(sal["target"], target)
    assert torch.equal(sal["src"], gs[..., :N])
    assert torch.equal(sal["static"], gst)
    assert torch.equal(sal["times"], gt)
    assert all(p.requires_grad for p in model.parameters())       # restored


def _oracle_ig(cfg, batch, seed, target, steps):
    """The same midpoint Riemann sum as attribution.integrated_gradients, on the fp32 CPU oracle."""
    from oracle.raindrop_oracle import build_oracle_model
    oracle = build_oracle_model(cfg).eval()
    synth_weights(oracle, cfg, seed=seed)
    for p in oracle.parameters():
        p.requires_grad_(False)
    src, static, times, lengths = batch["src"], batch["static"], batch["times"], batch["lengths"]
    T, B, N2 = src.shape
    N = N2 // 2
    x_v = src[..., :N]
    a = (torch.arange(steps, dtype=torch.float32) + 0.5) / steps
    v = (a[None, :, None, None] * x_v[:, None]).requires_grad_(True)                      # zero baseline
    s_k = torch.cat([v, src[:, None, :, N:].expand(T, steps, B, N)], -1).reshape(T, steps * B, N2)
    st = (a[:, None, None] * static[None]).requires_grad_(True)
    logits, _, _ = oracle.forward_dense(s_k, st.reshape(steps * B, -1), times[:, None].expand(T, steps, B).reshape(T, -1),
                                        lengths.repeat(steps))
    gv, gst = torch.autograd.grad(logits.gather(1, target.repeat(steps)[:, None]).sum(), (v, st))
    return x_v * gv.sum(1) / steps, static * gst.sum(0) / steps


@pytest.mark.gpu
def test_integrated_gradients():
    """integrated_gradients at P19 B = 16 matches the same Riemann sum on the CPU oracle (exact mode); its completeness
    residual is small at steps = 64."""
    from raindrop_b200.attribution import integrated_gradients
    cfg = model_config("P19", dropout=0.2)
    batch = make_batch(cfg, 16, seed=55)
    d = to_dev(batch)
    model = build_dropin(cfg, 7).eval()
    model._plan.obprop_mode = EXACT
    ig = integrated_gradients(model, d["src"], d["static"], d["times"], d["lengths"], steps=32, max_batch=200)
    ref_src, ref_static = _oracle_ig(cfg, batch, 7, ig["target"].cpu(), 32)
    e_src, e_static = normwise(ig["src"], ref_src), normwise(ig["static"], ref_static)
    print("IG vs oracle: src %.3e static %.3e" % (e_src, e_static))
    assert e_src < 2e-3 and e_static < 2e-3
    ig64 = integrated_gradients(model, d["src"], d["static"], d["times"], d["lengths"], steps=64)
    # completeness: the Riemann sum of a ReLU network's piecewise-constant gradient; per sample it is reported (a sample
    # whose path crosses many gates needs more steps), the batch as a whole must be within 5e-2
    res, delta = ig64["residual"].abs().cpu(), ig64["delta"].abs().cpu()
    rel = res / delta.clamp_min(1e-6)
    print("IG steps=64 completeness residual / |delta| per sample: max %.3e median %.3e, batch %.3e"
          % (rel.max(), rel.median(), res.sum() / delta.sum()))
    assert float(res.sum() / delta.sum()) <= 5e-2, rel

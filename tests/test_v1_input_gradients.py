"""Gradients with respect to the float inputs of legacy `Raindrop` v1 (src, static, times) and its global_structure, the
differentiable PositionalEncodingTF, and the attribution helpers on a v1 model.  References:
tests/golden/v1_input_grads.npz (the reference's own class, tools/make_v1_input_grad_golden.py), the CPU oracle's
positional encoding through autograd, and central differences in train mode."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import check_against_golden, load_golden, normwise, to_dev
from raindrop_b200.synth import CONFIGS, keyed_values, make_batch

V1_TOL = 2e-3           # the bound the v1 parameter gradients meet against v1_p12_b3.npz
INPUTS = ("d_src", "d_static", "d_times", "d_global_structure")


def _v1_case(golden_dir, B=3, seed=77):
    """The model and batch of v1_p12_b3.npz (keyed weights, the fixture's global_structure), on the device."""
    from raindrop_b200.models_rd import Raindrop
    z, meta = load_golden(golden_dir, "v1_p12_b3")
    cfg = dict(CONFIGS["P12"]); cfg["name"] = "P12"
    batch = make_batch(dict(cfg, d_ob=2), B, seed=seed)
    gs = torch.from_numpy(z["global_structure"]).cuda()
    model = Raindrop(36, 72, 2, 144, 2, 0.2, 215, 9, 100, 0.5, "mean", 2, gs)
    sd = model.state_dict()
    model.load_state_dict({k: keyed_values(meta["weight_seed"], k, tuple(v.shape)) for k, v in sd.items()})
    return model.cuda().eval(), to_dev(batch), meta


def _input_grads(model, d):
    """(logits, d_src, d_static, d_times, d_global_structure) of the batch's cross-entropy loss via torch.autograd.grad."""
    src = d["src"].clone().requires_grad_(True)
    static = d["static"].clone().requires_grad_(True)
    times = d["times"].clone().requires_grad_(True)
    gs0 = model.global_structure
    gs = gs0.detach().clone().requires_grad_(True)
    model.global_structure = gs
    try:
        logits, _, _ = model.forward(src, static, times, d["lengths"])
        grads = torch.autograd.grad(F.cross_entropy(logits, d["y"]), [src, static, times, gs])
    finally:
        model.global_structure = gs0
    return (logits.detach(),) + tuple(grads)


# ---- CPU -------------------------------------------------------------------------------------------------------------
def test_v1_fixture_global_structure_gradient_pattern(golden_dir):
    """The reference's d_global_structure is zero on the diagonal (overwritten in place) and where the graph has no edge
    (the edge list comes from nonzero): the pattern the out-of-place diagonal and the nonzero edge list here reproduce."""
    z = np.load(golden_dir + "/v1_input_grads.npz")
    gs = np.load(golden_dir + "/v1_p12_b3.npz")["global_structure"]
    g = z["d_global_structure"]
    assert g.shape == gs.shape == (36, 36)
    assert not np.diagonal(g).any()
    assert not g[gs == 0].any()
    assert np.count_nonzero(g) > 0


# ---- GPU -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_v1_input_grads_match_reference(golden_dir):
    """torch.autograd.grad(loss, [src, static, times, global_structure]) on v1 against the reference's own gradients."""
    z = np.load(golden_dir + "/v1_input_grads.npz")
    model, d, _ = _v1_case(golden_dir)
    _, *grads = _input_grads(model, d)
    errs = {}
    for key, g in zip(INPUTS, grads):
        assert g is not None and torch.isfinite(g).all(), key
        check_against_golden(z, key in z.files, key, g, V1_TOL, errs)
    N = 36
    assert torch.count_nonzero(grads[0][..., N:]) == 0             # the mask half takes no part in the output
    assert torch.count_nonzero(torch.diagonal(grads[3])) == 0
    print("v1 input gradient errors", errs)


def _param_grads(model):
    return {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}


@pytest.mark.gpu
def test_v1_parameter_grads_bit_identical_with_input_grads(golden_dir):
    """Asking for input gradients (src, static, times, global_structure) changes neither the logits nor any of the 36
    parameter gradients by one bit (train mode: the dropout stream starts from the same state in both runs)."""
    out = []
    for want in (False, True):
        model, d, meta = _v1_case(golden_dir, B=8, seed=5)
        model.train()
        src = d["src"].clone().requires_grad_(want)
        static = d["static"].clone().requires_grad_(want)
        times = d["times"].clone().requires_grad_(want)
        gs0 = model.global_structure
        model.global_structure = gs0.clone().requires_grad_(want)
        logits, _, _ = model.forward(src, static, times, d["lengths"])
        F.cross_entropy(logits, d["y"]).backward()
        for t in (src, static, times, model.global_structure):
            assert (t.grad is not None) == want
        out.append((logits.detach(), _param_grads(model)))
    assert torch.equal(out[0][0], out[1][0])
    assert sorted(out[0][1]) == sorted(out[1][1])
    # lin_query / lin_key get written zeros (supplied edge weights replace their logits); the 36 others are non-zero
    assert sorted(k for k, g in out[0][1].items() if g.abs().max() > 0) == sorted(meta["with_grad"])
    assert len(meta["with_grad"]) == 36
    for k in out[0][1]:
        assert torch.equal(out[0][1][k], out[1][1][k]), k


@pytest.mark.gpu
def test_v1_frozen_model_input_grads_skip_parameter_work(golden_dir):
    """All parameters frozen: the same input gradients, bit for bit, no .grad written, and fewer launches in the backward
    (no weight-gradient GEMMs in the input layer, the TransformerConv and the encoder, no head parameter outputs)."""
    from raindrop_b200 import lib as L
    lib = L.load()
    res, launches = [], []
    for frozen in (False, True):
        model, d, _ = _v1_case(golden_dir, B=16, seed=9)
        for p in model.parameters():
            p.requires_grad_(not frozen)
        _input_grads(model, d)                          # warm-up (one-time kernel set-up)
        src = d["src"].clone().requires_grad_(True)
        static = d["static"].clone().requires_grad_(True)
        times = d["times"].clone().requires_grad_(True)
        gs0 = model.global_structure
        gs = gs0.clone().requires_grad_(True)
        model.global_structure = gs
        logits, _, _ = model.forward(src, static, times, d["lengths"])
        loss = F.cross_entropy(logits, d["y"])
        torch.cuda.synchronize()
        n0 = lib.rd_launch_count()
        res.append(torch.autograd.grad(loss, [src, static, times, gs]))
        launches.append(lib.rd_launch_count() - n0)
        model.global_structure = gs0
        assert all(p.grad is None for p in model.parameters())
    for a, b in zip(*res):
        assert torch.equal(a, b)
    print("v1 backward launches: with parameters %d, frozen %d" % tuple(launches))
    assert launches[1] < launches[0], launches
    # only static asks for a gradient: the backward stops at the head (no d(encoder input)), same d_static
    static = d["static"].clone().requires_grad_(True)
    logits, _, _ = model.forward(d["src"], static, d["times"], d["lengths"])
    loss = F.cross_entropy(logits, d["y"])
    n0 = lib.rd_launch_count()
    (g,) = torch.autograd.grad(loss, static)
    n_static = lib.rd_launch_count() - n0
    assert torch.equal(g, res[1][1])
    assert n_static < launches[1], (n_static, launches)


@pytest.mark.gpu
def test_v1_train_mode_central_difference(golden_dir):
    """Train mode with dropout: <d_times, v> and <d_static, v> against central differences of the logits with the
    dropout stream rewound before every forward."""
    model, d, _ = _v1_case(golden_dir, B=16, seed=21)
    model.train()
    with torch.no_grad():
        model.forward(d["src"], d["static"], d["times"], d["lengths"])      # creates the dropout stream state
    rng0 = model._plan.rng_state.clone()

    def f(static, times, grad=False):
        model._plan.rng_state.copy_(rng0)
        with torch.set_grad_enabled(grad):
            logits, _, _ = model.forward(d["src"], static, times, d["lengths"])
        return logits[:, 0].sum() if grad else logits[:, 0].double().sum()

    static = d["static"].clone().requires_grad_(True)
    times = d["times"].clone().requires_grad_(True)
    g_static, g_times = torch.autograd.grad(f(static, times, grad=True), (static, times))
    T = d["times"].shape[0]
    valid = torch.arange(T, device="cuda")[:, None] < d["lengths"][None, :]
    assert torch.count_nonzero(g_times[~valid]) == 0                    # padded steps take no part in the output
    gen = torch.Generator(device="cuda").manual_seed(5)
    # directions signed like the gradient, so that <g, v> is far above the fp32 rounding of the logits / (2 eps).  d_times
    # is small next to the logits, so its step is larger; a larger step also lets more ReLU gates of the encoder flip
    # inside the interval, hence its looser bound
    for which, g, eps, tol in (("times", g_times, 3e-3, 2e-2), ("static", g_static, 1e-3, 1e-2)):
        for _ in range(2):
            v = torch.rand(g.shape, generator=gen, device="cuda") * g.sign()
            if which == "times":
                v = v * valid
            an = float((g.double() * v.double()).sum())
            if which == "times":
                fd = (f(d["static"], d["times"] + eps * v) - f(d["static"], d["times"] - eps * v)) / (2 * eps)
            else:
                fd = (f(d["static"] + eps * v, d["times"]) - f(d["static"] - eps * v, d["times"])) / (2 * eps)
            print(which, "analytic %.6e central difference %.6e" % (an, float(fd)))
            assert abs(an - float(fd)) <= tol * abs(an), (which, an, float(fd))


@pytest.mark.gpu
@pytest.mark.parametrize("d_pe", [16, 36, 64])
def test_positional_encoding_tf_is_differentiable(d_pe):
    """PositionalEncodingTF: forward bit-identical to RF.positional_encoding; d_times from rd_positional_encoding_bwd
    matches autograd of the oracle's encoding in fp64."""
    from oracle.raindrop_oracle import positional_encoding as pe_oracle
    from raindrop_b200 import functional as RF
    from raindrop_b200.models_rd import PositionalEncodingTF
    T, B, max_len = 50, 7, 215
    g = torch.Generator().manual_seed(d_pe)
    times = torch.cumsum(torch.rand(T, B, generator=g) * 3, 0)
    times[40:, 3] = 0                                                   # padding rows
    G = torch.randn(T, B, d_pe, generator=g)
    mod = PositionalEncodingTF(d_pe, max_len, 100)
    t = times.cuda().requires_grad_(True)
    pe = mod(t)
    assert pe.grad_fn is not None
    assert torch.equal(pe.detach(), RF.positional_encoding(times.cuda(), max_len, d_pe))
    (d_times,) = torch.autograd.grad((pe * G.cuda()).sum(), t)
    t64 = times.double().requires_grad_(True)
    (ref,) = torch.autograd.grad((pe_oracle(t64, max_len, d_pe) * G.double()).sum(), t64)
    e = normwise(d_times, ref)
    print("d_pe", d_pe, "d_times error", e)
    assert e < 1e-5, e


@pytest.mark.gpu
def test_v1_saliency_and_integrated_gradients(golden_dir):
    """saliency() on v1 equals torch.autograd.grad of the target logits; integrated_gradients() equals the midpoint
    Riemann sum of the same model's saliency (v1 has no CPU oracle: a self-consistency check of the chunked path)."""
    from raindrop_b200.attribution import integrated_gradients, saliency
    model, d, _ = _v1_case(golden_dir, B=4, seed=33)
    N = 36
    src = d["src"].clone().requires_grad_(True)
    static = d["static"].clone().requires_grad_(True)
    times = d["times"].clone().requires_grad_(True)
    logits, _, _ = model.forward(src, static, times, d["lengths"])
    target = logits.detach().argmax(1)
    gs_, gst, gt = torch.autograd.grad(logits.gather(1, target[:, None]).sum(), (src, static, times))
    sal = saliency(model, d["src"], d["static"], d["times"], d["lengths"])
    assert torch.equal(sal["target"], target)
    assert torch.equal(sal["src"], gs_[..., :N])
    assert torch.equal(sal["static"], gst)
    assert torch.equal(sal["times"], gt)
    assert all(p.requires_grad for p in model.parameters())            # restored

    steps = 6
    ig = integrated_gradients(model, d["src"], d["static"], d["times"], d["lengths"], target=target, steps=steps,
                              max_batch=3 * d["src"].shape[1])
    x_v = d["src"][..., :N]
    acc_src, acc_static = torch.zeros_like(x_v), torch.zeros_like(d["static"])
    for k in range(steps):
        a = (k + 0.5) / steps
        s = d["src"].clone()
        s[..., :N] *= a
        sk = saliency(model, s, a * d["static"], d["times"], d["lengths"], target=target)
        acc_src += sk["src"]
        acc_static += sk["static"]
    e_src = normwise(ig["src"], x_v * acc_src / steps)
    e_static = normwise(ig["static"], d["static"] * acc_static / steps)
    print("v1 IG vs Riemann sum of saliency: src %.3e static %.3e" % (e_src, e_static))
    assert e_src < 5e-4 and e_static < 5e-4
    assert torch.isfinite(ig["residual"]).all()

"""TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz by running the reference's own,
unmodified files (oracle/ref_harness.py) on CPU:

    RAINDROP_REFERENCE=<checkout of the original project> python -m oracle.make_golden [part]

A fixture stores seeds + the reference's outputs; inputs and weights are regenerated from the
seeds by raindrop_b200.synth (make_batch / synth_weights), so the files stay small.  Stored per
case: logits, distance, the observation-propagation output `obs` [T,B,4N] (input of the temporal
attention, code/models_rd.py:341), the encoder output `enc` [T,B,D] (code/models_rd.py:358), the
cross-entropy loss and the gradient of every parameter that receives one -- in full for tiny
shapes, as fingerprints (sum / abs-sum / l2 / strided sample) for the BASELINE shapes.
"""
import json
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import ref_harness  # noqa: E402
from raindrop_b200.synth import keyed_values, make_batch, model_config, synth_weights, used_param_keys  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
N_SAMPLE = 509


def fingerprint(t):
    """Order-sensitive summary used when the full tensor is too big to commit."""
    f = t.detach().double().flatten()
    step = max(1, f.numel() // N_SAMPLE)
    return dict(sum=float(f.sum()), asum=float(f.abs().sum()), l2=float((f * f).sum().sqrt()),
                sample=f[::step][:N_SAMPLE].float().numpy())


def sparse_structure(n, seed):
    g = torch.Generator().manual_seed(seed)
    a = (torch.rand(n, n, generator=g) < 0.35).float() * torch.rand(n, n, generator=g)
    a[n - 1, :] = 0   # a node with no outgoing edges ...
    a[:, 1] = 0       # ... and one whose only incoming edge is the forced self loop
    return a


CASES = [
    # name, config, batch, data seed, weight seed, options
    ("tiny_dense", "TINY", 3, 11, 7, {}),
    ("tiny_t0", "TINY", 3, 12, 8, {"first_time_zero": True}),
    ("tiny_sparse", "TINY", 4, 13, 9, {"sparse": 5}),
    ("tiny8_nostatic", "TINY8", 4, 14, 10, {}),
    ("p19_b4", "P19", 4, 15, 11, {}),
    ("p19_b5_leave10", "P19", 5, 16, 12, {"zero_sensors": 10}),
    ("p12_b2", "P12", 2, 17, 13, {"first_time_zero": True}),
    ("pam_b2", "PAM", 2, 18, 14, {"first_time_zero": True}),
]


def run_case(name, cfg_name, B, dseed, wseed, opt):
    cfg = model_config(cfg_name, dropout=0.2)
    if "sparse" in opt:
        cfg["global_structure"] = sparse_structure(cfg["d_inp"], opt["sparse"])
    model = ref_harness.build_reference_model(cfg).eval()   # eval: dropout off, parity is exact
    synth_weights(model, cfg, seed=wseed)
    batch = make_batch(cfg, B, seed=dseed, first_time_zero=opt.get("first_time_zero", False),
                       zero_sensors=opt.get("zero_sensors", 0))
    grabbed = {}
    h1 = model.transformer_encoder.register_forward_hook(lambda m, i, o: grabbed.update(enc=o, obs=i[0]))
    logits, distance, _ = model.forward(batch["src"], batch["static"], batch["times"], batch["lengths"])
    h1.remove()
    loss = F.cross_entropy(logits, batch["y"])
    model.zero_grad()
    loss.backward()
    tiny = cfg_name.startswith("TINY")
    out = dict(logits=logits.detach().numpy(), distance=np.float32(distance.item()),
               loss=np.float32(loss.item()))
    D4 = cfg["d_inp"] * cfg["d_ob"]
    tensors = dict(obs=grabbed["obs"][:, :, :D4], pe=grabbed["obs"][:, :, D4:], enc=grabbed["enc"])
    grads = {}
    params = dict(model.named_parameters())
    with_grad = sorted(k for k, p in params.items() if p.grad is not None)
    assert with_grad == sorted(used_param_keys(cfg)), set(with_grad) ^ set(used_param_keys(cfg))
    for k in with_grad:
        grads["grad." + k] = params[k].grad
    tensors.update(grads)
    for k, t in tensors.items():
        if tiny:
            out[k] = t.detach().numpy()
        else:
            fp = fingerprint(t)
            out[k + "#sample"] = fp["sample"]
            out[k + "#stats"] = np.array([fp["sum"], fp["asum"], fp["l2"]], dtype=np.float64)
    meta = dict(case=name, config=cfg_name, batch=B, data_seed=dseed, weight_seed=wseed, options=opt,
                torch=torch.__version__, reference_commit="892eb57",
                generator="oracle/make_golden.py", full_tensors=tiny)
    out["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(GOLDEN, name + ".npz"), **out)
    print("%-18s logits[0]=%s loss=%.6f  %d arrays" % (name, logits[0].tolist(), loss.item(), len(out)))


def operator_cases():
    """Operator-level fixtures: `Observation_progation` with use_beta both ways on a sparse
    weighted graph, and `TransformerConv` with and without supplied edge weights."""
    ref = ref_harness.load_reference()
    from raindrop_b200.synth import _stream
    out = {}
    N, T, d_ob = 6, 5, 4
    C = T * d_ob
    torch.manual_seed(3)
    layer = ref.Observation_progation(in_channels=C, out_channels=C, heads=1, n_nodes=N, ob_dim=d_ob)
    adj = sparse_structure(N, 21)
    adj[torch.arange(N), torch.arange(N)] = 1
    ei = torch.nonzero(adj).T.contiguous()
    ew = adj[ei[0], ei[1]]
    x = torch.from_numpy(_stream(5, "op.x", N * C)).float().view(N, C) - 0.3
    p_t = torch.from_numpy(_stream(5, "op.pt", T * 16)).float().view(T, 16)
    for k, v in layer.state_dict().items():
        out["obprop.sd." + k] = v.numpy()
    for ub in (False, True):
        o, (ei2, al) = layer(x, p_t=p_t, edge_index=ei, edge_weights=ew, use_beta=ub, edge_attr=None,
                             return_attention_weights=True)
        tag = "obprop.beta%d." % int(ub)
        out[tag + "out"] = o.detach().numpy()
        out[tag + "edge_index"] = ei2.numpy()
        out[tag + "alpha"] = al.detach().numpy()
    out["obprop.x"], out["obprop.p_t"] = x.numpy(), p_t.numpy()
    out["obprop.edge_index"], out["obprop.edge_w"] = ei.numpy(), ew.numpy()

    # with supplied edge weights the reference only works for heads == 1 (alpha is [E,1] and is
    # viewed as [-1, heads, 1], code/transformer_conv.py:199-206); the QK path takes any heads.
    xn = torch.from_numpy(_stream(6, "tc.x", N * 7)).float().view(N, 7) - 0.5
    out["tconv.x"] = xn.numpy()
    for tag, heads, w, seed in (("tconv.w.", 1, ew, 4), ("tconv.qk.", 2, None, 5)):
        torch.manual_seed(seed)
        conv = ref.TransformerConv(in_channels=7, out_channels=5, heads=heads)
        for k, v in conv.state_dict().items():
            out[tag + "sd." + k] = v.numpy()
        o, (_, al) = conv(xn, edge_index=ei, edge_weights=w, edge_attr=None, return_attention_weights=True)
        out[tag + "out"] = o.detach().numpy()
        out[tag + "alpha"] = al.detach().numpy()
    np.savez_compressed(os.path.join(GOLDEN, "operators.npz"), **out)
    print("operators          %d arrays" % len(out))


def operator_grad_cases():
    """Gradient fixtures of the two graph operators (reference autograd through code/Ob_propagation.py and
    code/transformer_conv.py under the PyG shim): loss = sum(out * G) [+ sum(alpha * g) for use_beta=True, whose
    returned alpha is differentiable and feeds layer 2 in code/models_rd.py:332-336].  Inputs / weights are the ones
    of operators.npz; written to operators_grad.npz."""
    ref = ref_harness.load_reference()
    from raindrop_b200.synth import _stream
    z = np.load(os.path.join(GOLDEN, "operators.npz"))
    out = {}
    ei = torch.from_numpy(z["obprop.edge_index"])
    N, C = z["obprop.x"].shape
    T, d_ob = z["obprop.p_t"].shape[0], 4
    layer = ref.Observation_progation(in_channels=C, out_channels=C, heads=1, n_nodes=N, ob_dim=d_ob)
    layer.load_state_dict({k[len("obprop.sd."):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("obprop.sd.")})
    G = torch.from_numpy(_stream(9, "opg.G", N * C)).float().view(N, C) - 0.5
    out["obprop.G"] = G.numpy()
    for ub in (False, True):
        layer.zero_grad()
        x = torch.from_numpy(z["obprop.x"]).clone().requires_grad_(True)
        p_t = torch.from_numpy(z["obprop.p_t"]).clone().requires_grad_(True)
        ew = torch.from_numpy(z["obprop.edge_w"]).clone().requires_grad_(True)
        o, (ei2, al) = layer(x, p_t=p_t, edge_index=ei, edge_weights=ew, use_beta=ub, edge_attr=None, return_attention_weights=True)
        loss = (o * G).sum()
        tag = "obprop.beta%d." % int(ub)
        if ub:
            g = torch.from_numpy(_stream(9, "opg.g", al.numel())).float() - 0.5
            out[tag + "g_alpha"] = g.numpy()
            loss = loss + (al * g).sum()
        loss.backward()
        out[tag + "d_x"] = x.grad.numpy()
        out[tag + "d_edge_w"] = (ew.grad if ew.grad is not None else torch.zeros_like(ew)).numpy()
        if ub:
            out[tag + "d_p_t"] = p_t.grad.numpy()
        for k, prm in layer.named_parameters():
            if prm.grad is not None:
                out[tag + "grad." + k] = prm.grad.numpy()
    xn0 = torch.from_numpy(z["tconv.x"])
    for tag, heads, use_w in (("tconv.w.", 1, True), ("tconv.qk.", 2, False)):
        conv = ref.TransformerConv(in_channels=7, out_channels=5, heads=heads)
        conv.load_state_dict({k[len(tag + "sd."):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(tag + "sd.")})
        xn = xn0.clone().requires_grad_(True)
        ew = torch.from_numpy(z["obprop.edge_w"]).clone().requires_grad_(True)
        G2 = torch.from_numpy(_stream(9, tag + "G", N * 5 * heads)).float().view(N, 5 * heads) - 0.5
        o, _ = conv(xn, edge_index=ei, edge_weights=ew if use_w else None, edge_attr=None, return_attention_weights=True)
        (o * G2).sum().backward()
        out[tag + "G"] = G2.numpy()
        out[tag + "d_x"] = xn.grad.numpy()
        if use_w:
            out[tag + "d_edge_w"] = ew.grad.numpy()
        for k, prm in conv.named_parameters():
            out[tag + "grad." + k] = (prm.grad if prm.grad is not None else torch.zeros_like(prm)).numpy()
    np.savez_compressed(os.path.join(GOLDEN, "operators_grad.npz"), **out)
    print("operators_grad     %d arrays: %s" % (len(out), sorted(out)[:60]))


V1_FULL_MAX = 4096      # v1 gradients with more elements are stored as fingerprints (keeps the file small)


def v1_case():
    """Legacy `Raindrop` v1 (code/models_rd.py:46-191; hard-coded to 36 sensors / 215 steps): logits, loss and the
    gradient of every parameter that gets one, B = 3, eval mode.  Weights: every state-dict entry from the keyed
    stream (synth.keyed_values, weight seed 19), so the fixture stores no weights; `encoder` / `emb` thus get a useful
    scale (the reference initialises them to +-1e-10, which would hide the graph layer)."""
    ref = ref_harness.load_reference()
    from raindrop_b200.synth import CONFIGS
    cfg = dict(CONFIGS["P12"]); cfg["name"] = "P12"
    B, wseed = 3, 19
    batch = make_batch(dict(cfg, d_ob=2), B, seed=77)
    torch.manual_seed(5)
    gs = (torch.rand(36, 36) < 0.5).float() * torch.rand(36, 36)
    model = ref.Raindrop(36, 72, 2, 144, 2, 0.2, 215, 9, 100, 0.5, "mean", 2, gs.clone()).eval()
    sd = model.state_dict()
    model.load_state_dict({k: keyed_values(wseed, k, tuple(v.shape)) for k, v in sd.items()})
    logits, distance, _ = model.forward(batch["src"], batch["static"], batch["times"], batch["lengths"])
    loss = F.cross_entropy(logits, batch["y"])
    model.zero_grad()
    loss.backward()
    out = dict(logits=logits.detach().numpy(), loss=np.float32(loss.item()), distance=np.float32(float(distance)),
               global_structure=gs.numpy())
    with_grad = [k for k, prm in model.named_parameters() if prm.grad is not None]
    for k in with_grad:
        g = model.get_parameter(k).grad
        if g.numel() <= V1_FULL_MAX:
            out["grad." + k] = g.numpy()
        else:
            fp = fingerprint(g)
            out["grad." + k + "#sample"] = fp["sample"]
            out["grad." + k + "#stats"] = np.array([fp["sum"], fp["asum"], fp["l2"]], dtype=np.float64)
    meta = dict(case="v1_p12_b3", batch=B, data_seed=77, weight_seed=wseed, torch=torch.__version__,
                reference_commit="892eb57", generator="oracle/make_golden.py v1",
                state_dict={k: list(v.shape) for k, v in sd.items()}, with_grad=with_grad)
    out["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(GOLDEN, "v1_p12_b3.npz"), **out)
    print("v1_p12_b3  logits[0]=%s loss=%.6f distance=%g grads for %d tensors" %
          (logits[0].tolist(), loss.item(), float(distance), len(with_grad)))


def default_init_case():
    """The reference's Raindrop_v2 as code/Raindrop.py:245-251 constructs it (torch.manual_seed(1), the modules' own
    initialisation, TINY shape): its state dict (entries above 1024 elements as fingerprints) and its eval-mode
    logits on make_batch(seed=1)."""
    cfg = model_config("TINY", dropout=0.2)
    ref = ref_harness.build_reference_model(cfg).eval()
    batch = make_batch(cfg, 3, seed=1)
    with torch.no_grad():
        logits = ref.forward(batch["src"], batch["static"], batch["times"], batch["lengths"])[0]
    out = {"logits": logits.numpy()}
    sd = ref.state_dict()
    for k, v in sd.items():
        if v.numel() <= 1024:
            out["sd." + k] = v.numpy()
        else:
            fp = fingerprint(v)
            out["sd." + k + "#sample"] = fp["sample"]
            out["sd." + k + "#stats"] = np.array([fp["sum"], fp["asum"], fp["l2"]], dtype=np.float64)
    out["meta"] = np.frombuffer(json.dumps(dict(keys=list(sd), torch=torch.__version__, reference_commit="892eb57",
                                                generator="oracle/make_golden.py default_init")).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(GOLDEN, "tiny_default_init.npz"), **out)
    print("tiny_default_init  logits[0]=%s  %d state-dict entries" % (logits[0].tolist(), len(sd)))


def data_pipeline_case():
    """The reference's host-side input pipeline (code/utils_rd.py) on the raw arrays of
    tests/test_data_pipeline.py::_raw(seed=4).  getStats is stored only where the installed numpy still accepts it
    (numpy >= 1.24 rejects its `np.max([array, scalar])`); the rest runs on the restatement's statistics."""
    from oracle import data_oracle as DO
    from test_data_pipeline import _raw
    ref_harness.load_reference()
    import utils_rd as U
    P, minutes, static, y = _raw(seed=4)
    out = {}
    mf, stdf = DO.get_stats(P)
    try:
        out["getStats.mf"], out["getStats.stdf"] = U.getStats(P)
    except ValueError:
        pass
    out["mask_normalize"] = U.mask_normalize(P.copy(), mf, stdf)
    ms, ss = U.getStats_static(static, dataset="P12")
    out["getStats_static.ms"], out["getStats_static.ss"] = ms, ss
    out["mask_normalize_static"] = U.mask_normalize_static(static.copy(), ms, ss)
    Plist = [{"arr": P[i], "time": minutes[i][:, None], "extended_static": static[i]} for i in range(len(P))]
    for i, t in enumerate(U.tensorize_normalize(Plist, y, mf, stdf, ms, ss)):
        out["tensorize_normalize.%d" % i] = t.numpy()
    np.savez_compressed(os.path.join(GOLDEN, "data_pipeline.npz"), **out)
    print("data_pipeline      %d arrays: %s" % (len(out), sorted(out)))


if __name__ == "__main__":
    os.makedirs(GOLDEN, exist_ok=True)
    torch.set_num_threads(8)
    if len(sys.argv) > 1 and sys.argv[1] == "operators_grad":      # add-on fixtures: leaves the existing files untouched
        operator_grad_cases()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "v1":
        v1_case()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "default_init":
        default_init_case()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "data_pipeline":
        data_pipeline_case()
        sys.exit(0)
    for case in CASES:
        run_case(*case)
    operator_cases()
    operator_grad_cases()
    v1_case()
    default_init_case()
    data_pipeline_case()

"""CPU: pins the oracle restatement (oracle/raindrop_oracle.py) against the golden fixtures that were
generated from the reference's own unmodified files (oracle/make_golden.py)."""
import json

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import case_setup, check_against_golden, fingerprint, load_golden, normwise
from oracle.raindrop_oracle import (ObPropOracle, TransformerConvOracle, build_oracle_model, encoder_layer_explicit,
                                    graph_from_adjacency, node_scale_from_graph, positional_encoding)
from raindrop_b200.synth import synth_weights, used_param_keys

CASES = ["tiny_dense", "tiny_t0", "tiny_sparse", "tiny8_nostatic", "p19_b4", "p19_b5_leave10", "p12_b2", "pam_b2"]


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("mode", ["edgewise", "dense"])
def test_oracle_matches_reference_outputs(golden_dir, name, mode):
    z, meta = load_golden(golden_dir, name)
    if mode == "edgewise" and meta["config"] in ("P12", "PAM"):
        pytest.skip("per-edge loop at this size is covered by the dense closed form (keeps the CPU suite short)")
    cfg, batch = case_setup(meta)
    torch.set_num_threads(8)
    model = build_oracle_model(cfg).eval()
    synth_weights(model, cfg, seed=meta["weight_seed"])
    stages = {}
    fwd = model.forward if mode == "edgewise" else model.forward_dense
    logits, distance, _ = fwd(batch["src"], batch["static"], batch["times"], batch["lengths"], stages=stages)
    loss = F.cross_entropy(logits, batch["y"])
    loss.backward()
    tol = 1e-6 if mode == "edgewise" else 2e-5
    assert normwise(logits, z["logits"]) < tol
    assert float(distance) == float(z["distance"])
    errs = {}
    full = meta["full_tensors"]
    check_against_golden(z, full, "obs", stages["obs"], tol, errs)
    check_against_golden(z, full, "pe", stages["pe"], 1e-7, errs)
    check_against_golden(z, full, "enc", stages["enc"], tol, errs)
    params = dict(model.named_parameters())
    for k in used_param_keys(cfg):
        check_against_golden(z, full, "grad." + k, params[k].grad, 10 * tol, errs)
    assert sorted(k for k, p in params.items() if p.grad is not None) == sorted(used_param_keys(cfg))


def test_operator_fixtures(golden_dir):
    z = np.load(golden_dir + "/operators.npz")
    x, p_t = torch.from_numpy(z["obprop.x"]), torch.from_numpy(z["obprop.p_t"])
    ei, ew = torch.from_numpy(z["obprop.edge_index"]), torch.from_numpy(z["obprop.edge_w"])
    N, Cc = x.shape
    layer = ObPropOracle(Cc, N, 4)
    layer.load_state_dict({k[len("obprop.sd."):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("obprop.sd.")})
    for ub in (0, 1):
        out, (ei2, alpha) = layer(x, p_t, ei, ew, use_beta=bool(ub))
        tag = "obprop.beta%d." % ub
        assert normwise(out, z[tag + "out"]) < 1e-6
        assert torch.equal(ei2, torch.from_numpy(z[tag + "edge_index"]))
        assert normwise(alpha, z[tag + "alpha"]) < 1e-6
    # closed form == edge-wise on a sparse weighted graph, isolated rows exactly zero
    s = node_scale_from_graph(ei, ew, N)
    assert normwise(layer.forward_dense(x, s[:, None]), z["obprop.beta0.out"]) < 1e-6
    tx = torch.from_numpy(z["tconv.x"])
    for tag, heads, w in (("tconv.w.", 1, ew), ("tconv.qk.", 2, None)):
        conv = TransformerConvOracle(7, 5, heads)
        conv.load_state_dict({k[len(tag + "sd."):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(tag + "sd.")})
        out, alpha = conv(tx, ei, w)
        assert normwise(out, z[tag + "out"]) < 1e-6 and normwise(alpha, z[tag + "alpha"]) < 1e-6


def test_encoder_layer_explicit_matches_torch_module():
    """The written-out encoder layer (used to reason about the CUDA kernels) == nn.TransformerEncoderLayer."""
    torch.manual_seed(0)
    T, B, D, H = 9, 4, 24, 2
    layer = torch.nn.TransformerEncoderLayer(D, H, 40, 0.0).eval()
    x = torch.randn(T, B, D)
    lengths = torch.tensor([9, 3, 1, 6])
    pad = torch.arange(T)[None, :] >= lengths[:, None]
    ref = layer(x, src_key_padding_mask=pad)
    p = {k: v for k, v in layer.state_dict().items()}
    out = encoder_layer_explicit(x, pad, p, H)
    valid = (~pad).T[:, :, None]
    assert normwise(out * valid, ref * valid) < 1e-5


def test_graph_and_pe_conventions():
    adj = torch.tensor([[0., 2., 0.], [0., 0., 0.], [1., 0., 0.5]])
    ei, ew = graph_from_adjacency(adj)
    assert ei.tolist() == [[0, 0, 1, 2, 2], [0, 1, 1, 0, 2]]      # row-major; [0]=source row, [1]=target col
    assert ew.tolist() == [1., 2., 1., 1., 1.]                     # diagonal forced to one (models_rd.py:308)
    pe = positional_encoding(torch.tensor([[0.0, 3.0]]), 60)
    assert pe.shape == (1, 2, 16) and torch.allclose(pe[0, 0], torch.cat([torch.zeros(8), torch.ones(8)]))
    assert abs(pe[0, 1, 7].item() - np.sin(np.float32(3.0) / np.float32(60.0))) < 1e-7


def test_oracle_matches_reference_default_init(golden_dir):
    """Seeded construction (the modules' own initialisation, code/Raindrop.py:245-251) and the eval forward on it
    against the reference's own model (oracle/make_golden.py default_init_case)."""
    from raindrop_b200.synth import make_batch, model_config
    z = np.load(golden_dir + "/tiny_default_init.npz")
    cfg = model_config("TINY", dropout=0.2)
    orc = build_oracle_model(cfg).eval()
    sd = orc.state_dict()
    assert list(sd) == json.loads(bytes(z["meta"]).decode())["keys"]
    for k, v in sd.items():
        if "sd." + k in z.files:
            assert np.array_equal(v.numpy(), z["sd." + k]), k
        else:
            fp = fingerprint(v)
            assert np.array_equal(fp["sample"], z["sd." + k + "#sample"]), k
            assert np.allclose(fp["stats"], z["sd." + k + "#stats"], rtol=1e-12, atol=0), k
    batch = make_batch(cfg, 3, seed=1)
    with torch.no_grad():
        b = orc.forward(batch["src"], batch["static"], batch["times"], batch["lengths"])[0]
    # stored on another machine: CPU GEMM kernels may round the last bit differently there
    assert normwise(b, z["logits"]) < 1e-6


@pytest.mark.parametrize("seed", range(6))
def test_edgewise_equals_closed_form_on_random_graphs(seed):
    """PyG-style gather / segment-softmax / scatter (what the reference executes) == per-node closed form
    (what the CUDA path executes) on random weighted graphs with isolated nodes, both ob-prop layers chained."""
    g = torch.Generator().manual_seed(seed)
    N, T = int(torch.randint(1, 12, (1,), generator=g)), int(torch.randint(1, 9, (1,), generator=g))
    C = 4 * T
    adj = (torch.rand(N, N, generator=g) < 0.3).float() * (torch.rand(N, N, generator=g) * 3 - 1)   # negative weights too
    if N > 2:
        adj[:, 0] = 0                                     # node 0: no incoming edge at all (no forced diagonal here)
    edge_index = torch.nonzero(adj).T.contiguous()
    if edge_index.shape[1] == 0:
        pytest.skip("empty graph")
    w = adj[edge_index[0], edge_index[1]]
    torch.manual_seed(seed)
    l1, l2 = ObPropOracle(C, N, 4), ObPropOracle(C, N, 4)
    x = torch.randn(N, C, generator=g)
    o1, (ei1, a1) = l1(x, None, edge_index, w)
    o2, (_, a2) = l2(o1, None, ei1, a1.reshape(-1))
    s = node_scale_from_graph(edge_index, w, N)[:, None]
    d2 = l2.forward_dense(l1.forward_dense(x, s), s)
    assert torch.equal(a1.reshape(-1), w) and torch.equal(a2.reshape(-1), w)      # alpha is the PRE-softmax weight
    assert normwise(o2, d2) < 1e-6
    no_in = torch.ones(N, dtype=torch.bool)
    no_in[edge_index[1]] = False
    assert torch.all(o2[no_in] == 0) and torch.all(s[no_in] == 0)

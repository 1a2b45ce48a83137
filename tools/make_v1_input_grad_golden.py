"""TEST INFRASTRUCTURE ONLY.  Writes tests/golden/v1_input_grads.npz: the gradients of the reference's own, unmodified
legacy `Raindrop` v1 (code/models_rd.py:46-191, loaded by oracle/ref_harness.py on CPU) with respect to its float inputs
src, static, times and its global_structure, for the case of `oracle/make_golden.py v1` (P12 shape, B = 3, data seed 77,
keyed weights with seed 19, the same global_structure; eval mode, loss = cross entropy of the logits):

    RAINDROP_REFERENCE=<checkout of the original project> python tools/make_v1_input_grad_golden.py

Keys "d_src", "d_static", "d_times", "d_global_structure": full tensors up to 4096 elements, fingerprints
(tests/helpers.fingerprint: "<key>#sample", "<key>#stats") above; "meta" holds the seeds.

The reference writes the diagonal of its global_structure in place (code/models_rd.py:150-151: `.cuda()` is the
identity under the harness), which autograd refuses on a leaf that requires grad.  So the model gets a non-leaf clone
of a leaf `gs`, and d_global_structure is gs.grad: the in-place write makes the diagonal's gradient zero.
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

from helpers import fingerprint  # noqa: E402
from oracle import ref_harness  # noqa: E402
from oracle.make_golden import GOLDEN, V1_FULL_MAX  # noqa: E402
from raindrop_b200.synth import CONFIGS, keyed_values, make_batch  # noqa: E402


def main():
    ref = ref_harness.load_reference()
    cfg = dict(CONFIGS["P12"]); cfg["name"] = "P12"
    B, dseed, wseed = 3, 77, 19
    batch = make_batch(dict(cfg, d_ob=2), B, seed=dseed)
    torch.manual_seed(5)
    gs0 = (torch.rand(36, 36) < 0.5).float() * torch.rand(36, 36)        # as oracle/make_golden.py v1_case
    gs = gs0.clone().requires_grad_(True)
    model = ref.Raindrop(36, 72, 2, 144, 2, 0.2, 215, 9, 100, 0.5, "mean", 2, gs.clone()).eval()
    sd = model.state_dict()
    model.load_state_dict({k: keyed_values(wseed, k, tuple(v.shape)) for k, v in sd.items()})
    src = batch["src"].clone().requires_grad_(True)
    static = batch["static"].clone().requires_grad_(True)
    times = batch["times"].clone().requires_grad_(True)
    logits, _, _ = model.forward(src, static, times, batch["lengths"])
    d_src, d_static, d_times, d_gs = torch.autograd.grad(F.cross_entropy(logits, batch["y"]), (src, static, times, gs))
    out = {}
    for k, g in (("d_src", d_src), ("d_static", d_static), ("d_times", d_times), ("d_global_structure", d_gs)):
        if g.numel() <= V1_FULL_MAX:
            out[k] = g.detach().numpy()
        else:
            fp = fingerprint(g)
            out[k + "#sample"] = fp["sample"]
            out[k + "#stats"] = fp["stats"]
        print("%-20s %-14s |g| %.6e" % (k, tuple(g.shape), float(g.norm())))
    meta = dict(case="v1_p12_b3", batch=B, data_seed=dseed, weight_seed=wseed, torch=torch.__version__,
                reference_commit="892eb57", generator="tools/make_v1_input_grad_golden.py",
                global_structure="oracle/make_golden.py v1_case (torch.manual_seed(5))")
    out["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(GOLDEN, "v1_input_grads.npz"), **out)


if __name__ == "__main__":
    torch.set_num_threads(8)          # as oracle/make_golden.py
    main()

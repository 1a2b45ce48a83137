"""TEST INFRASTRUCTURE ONLY.  Writes tests/golden/input_grads.npz: the gradients of the reference's own, unmodified
Raindrop_v2 (oracle/ref_harness.py, on CPU) with respect to its three float inputs src, static and times, for the eight
cases of oracle/make_golden.py (same seeds, same eval-mode model, loss = cross entropy of the logits):

    RAINDROP_REFERENCE=<checkout of the original project> python tools/make_input_grad_golden.py

Tiny cases store full tensors, the BASELINE-shaped ones fingerprints (tests/helpers.fingerprint), under the keys
"<case>/d_src", "<case>/d_static", "<case>/d_times"; "<case>/meta" holds the case's seeds.
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
from oracle.make_golden import CASES, GOLDEN, sparse_structure  # noqa: E402
from raindrop_b200.synth import make_batch, model_config, synth_weights  # noqa: E402


def main():
    out = {}
    for name, cfg_name, B, dseed, wseed, opt in CASES:
        cfg = model_config(cfg_name, dropout=0.2)
        if "sparse" in opt:
            cfg["global_structure"] = sparse_structure(cfg["d_inp"], opt["sparse"])
        model = ref_harness.build_reference_model(cfg).eval()
        synth_weights(model, cfg, seed=wseed)
        batch = make_batch(cfg, B, seed=dseed, first_time_zero=opt.get("first_time_zero", False),
                           zero_sensors=opt.get("zero_sensors", 0))
        src = batch["src"].clone().requires_grad_(True)
        times = batch["times"].clone().requires_grad_(True)
        static = None if batch["static"] is None else batch["static"].clone().requires_grad_(True)
        logits, _, _ = model.forward(src, static, times, batch["lengths"])
        F.cross_entropy(logits, batch["y"]).backward()
        grads = dict(d_src=src.grad, d_times=times.grad)
        if static is not None:
            grads["d_static"] = static.grad
        tiny = cfg_name.startswith("TINY")
        for k, g in grads.items():
            if tiny:
                out["%s/%s" % (name, k)] = g.detach().numpy()
            else:
                fp = fingerprint(g)
                out["%s/%s#sample" % (name, k)] = fp["sample"]
                out["%s/%s#stats" % (name, k)] = fp["stats"]
        meta = dict(case=name, config=cfg_name, batch=B, data_seed=dseed, weight_seed=wseed, options=opt,
                    torch=torch.__version__, reference_commit="892eb57", generator="tools/make_input_grad_golden.py",
                    full_tensors=tiny)
        out[name + "/meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
        print("%-18s |d_src| %.4e  |d_times| %.4e  %s" % (name, float(src.grad.norm()), float(times.grad.norm()),
                                                      "|d_static| %.4e" % float(static.grad.norm()) if static is not None else ""))
    np.savez_compressed(os.path.join(GOLDEN, "input_grads.npz"), **out)


if __name__ == "__main__":
    main()

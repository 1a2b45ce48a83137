"""Cost of input gradients (rd_raindrop_v2_bwd_inputs) on the drop-in module path, one JSON line per workload.

    python tools/bench_input_grad.py [--steps 50] [--warmup 10] [--configs P19:128,P19:3880,P12:32,PAM:256] [--v1 32,128]

Per workload (train mode, dropout as configured, automatic ob-prop mode, seeded inputs and weights):
  step_ms / step_in_ms   forward + cross entropy + backward without / with src.requires_grad (all 34 parameter
                         gradients in both), and our kernel launches per step (rd_launch_count)
  bwd_full_ms / bwd_in_ms  the backward alone: parameter gradients only vs frozen parameters with d_src, d_static, d_times
  ig_attr_per_s          integrated_gradients(steps=32) attributions (samples) per second, eval mode
Medians over --steps CUDA-event-timed repetitions after --warmup untimed ones (IG: 5 timed calls).  Workloads are
the benchmark's P19 batch, the P19 validation-set batch (3880) and the P12 / PAM batches.
Legacy Raindrop v1 (--v1 batch sizes; "" skips it): the P12-shaped model of tests/golden/v1_p12_b3.npz (keyed weights,
its global_structure) in eval mode, "model": "v1" in the JSON line:
  step_ms / step_in_ms     forward + cross entropy + backward without / with src, static, times .requires_grad
  bwd_full_ms / bwd_in_ms  the backward alone: parameter gradients only vs frozen parameters with the three input gradients
The card's name and power limit are printed first: every number belongs to them.
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from raindrop_b200 import lib as L  # noqa: E402
from raindrop_b200.attribution import integrated_gradients  # noqa: E402
from raindrop_b200.models_rd import Raindrop, Raindrop_v2  # noqa: E402
from raindrop_b200.synth import CONFIGS, keyed_values, make_batch, model_config, synth_weights  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def build(cfg):
    torch.manual_seed(1)
    gs = torch.ones(cfg["d_inp"], cfg["d_inp"])
    kw = {} if cfg["static"] else {"static": False}
    m = Raindrop_v2(cfg["d_inp"], cfg["d_model"], cfg["nhead"], cfg["nhid"], cfg["nlayers"], cfg["dropout"],
                    cfg["max_len"], cfg["d_static"], cfg["MAX"], 0.5, "mean", cfg["n_classes"], gs, **kw)
    synth_weights(m, cfg, seed=5)
    return m.cuda()


def timed(fn, steps, warmup, pre=None):
    """median ms of fn() over `steps` CUDA-event-timed calls; pre() runs untimed before each call"""
    for _ in range(warmup):
        fn(pre()) if pre else fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(steps):
        state = pre() if pre else None
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn(state) if pre else fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2]


def workload(name, B, steps, warmup):
    lib = L.load()
    cfg = model_config(name)
    m = build(cfg).train()
    d = {k: (v.cuda() if v is not None else None) for k, v in make_batch(cfg, B, seed=3).items()}

    def step(want_src):
        src = d["src"].clone().requires_grad_(want_src)
        logits, _, _ = m.forward(src, d["static"], d["times"], d["lengths"])
        F.cross_entropy(logits, d["y"]).backward()

    out = {"config": name, "B": B}
    for key, want in (("step", False), ("step_in", True)):
        out[key + "_ms"] = round(timed(lambda: step(want), steps, warmup), 4)
        n0 = lib.rd_launch_count()
        step(want)
        torch.cuda.synchronize()
        out[key + "_launches"] = int(lib.rd_launch_count() - n0)
    out["step_overhead_pct"] = round(100.0 * (out["step_in_ms"] / out["step_ms"] - 1.0), 2)

    def fwd(frozen):
        def pre():
            for p in m.parameters():
                p.requires_grad_(not frozen)
            src = d["src"].clone().requires_grad_(frozen)
            times = d["times"].clone().requires_grad_(frozen)
            static = None if d["static"] is None else d["static"].clone().requires_grad_(frozen)
            logits, _, _ = m.forward(src, static, times, d["lengths"])
            return F.cross_entropy(logits, d["y"])
        return pre

    out["bwd_full_ms"] = round(timed(lambda loss: loss.backward(), steps, warmup, pre=fwd(False)), 4)
    out["bwd_in_ms"] = round(timed(lambda loss: loss.backward(), steps, warmup, pre=fwd(True)), 4)
    for p in m.parameters():
        p.requires_grad_(True)
    m.eval()
    ig_ms = timed(lambda: integrated_gradients(m, d["src"], d["static"], d["times"], d["lengths"], steps=32), 5, 1)
    out["ig_ms"] = round(ig_ms, 3)
    out["ig_attr_per_s"] = round(B / (ig_ms / 1e3), 1)
    return out


def build_v1():
    """The v1 model of oracle/make_golden.py v1_case (weight seed 19, global_structure from torch.manual_seed(5))."""
    torch.manual_seed(5)
    gs = (torch.rand(36, 36) < 0.5).float() * torch.rand(36, 36)
    m = Raindrop(36, 72, 2, 144, 2, 0.2, 215, 9, 100, 0.5, "mean", 2, gs.cuda())
    sd = m.state_dict()
    m.load_state_dict({k: keyed_values(19, k, tuple(v.shape)) for k, v in sd.items()})
    return m.cuda().eval()


def workload_v1(B, steps, warmup):
    lib = L.load()
    m = build_v1()
    cfg = dict(CONFIGS["P12"], name="P12", d_ob=2)
    d = {k: (v.cuda() if v is not None else None) for k, v in make_batch(cfg, B, seed=3).items()}

    def loss_of(want_in):
        src = d["src"].clone().requires_grad_(want_in)
        static = d["static"].clone().requires_grad_(want_in)
        times = d["times"].clone().requires_grad_(want_in)
        logits, _, _ = m.forward(src, static, times, d["lengths"])
        return F.cross_entropy(logits, d["y"])

    out = {"model": "v1", "config": "P12", "B": B, "mode": "eval"}
    for key, want in (("step", False), ("step_in", True)):
        out[key + "_ms"] = round(timed(lambda: loss_of(want).backward(), steps, warmup), 4)
        n0 = lib.rd_launch_count()
        loss_of(want).backward()
        torch.cuda.synchronize()
        out[key + "_launches"] = int(lib.rd_launch_count() - n0)
    out["step_overhead_pct"] = round(100.0 * (out["step_in_ms"] / out["step_ms"] - 1.0), 2)

    def pre(frozen):
        def fn():
            for p in m.parameters():
                p.requires_grad_(not frozen)
            return loss_of(frozen)
        return fn

    for key, frozen in (("bwd_full", False), ("bwd_in", True)):
        out[key + "_ms"] = round(timed(lambda loss: loss.backward(), steps, warmup, pre=pre(frozen)), 4)
        loss = pre(frozen)()
        torch.cuda.synchronize()
        n0 = lib.rd_launch_count()
        loss.backward()
        torch.cuda.synchronize()
        out[key + "_launches"] = int(lib.rd_launch_count() - n0)
    for p in m.parameters():
        p.requires_grad_(True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--configs", default="P19:128,P19:3880,P12:32,PAM:256")
    ap.add_argument("--v1", default="32,128", help="batch sizes of the legacy Raindrop v1 leg (empty: skip)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_input_grad.py needs a GPU")
    print(json.dumps({"card": card(), "torch": torch.__version__}), flush=True)
    for item in filter(None, args.configs.split(",")):
        name, B = item.split(":")
        print(json.dumps(workload(name, int(B), args.steps, args.warmup)), flush=True)
    for B in filter(None, args.v1.split(",")):
        print(json.dumps(workload_v1(int(B), args.steps, args.warmup)), flush=True)


if __name__ == "__main__":
    main()

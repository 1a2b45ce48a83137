#!/usr/bin/env python
"""Benchmark of the Raindrop hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NAME] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

`--dump-outputs DIR` writes, after the timed steps, what the last timed TrainStep computed on rank 0 as float32
DIR/<name>.npy: `loss`, `logits`, and per used parameter its updated value `param.<key>` and its gradient
`grad.<key>` (state-dict keys).  Inputs and weights are seeded, so two builds run with the same arguments can be
compared output for output.  Above 64 MiB in all, arrays larger than an even share are replaced by a fixed, seeded
sample of their elements.

A "step" is one training step of Raindrop_v2 (forward + CrossEntropy + backward + Adam, dropout 0.2,
code/Raindrop.py:311-324) on one batch of synthetic data of the named configuration.  The default
configuration is the one BASELINE.json's metric is quoted on (configs[1]: P19 shape, B = 128 samples per
GPU, 34 sensors, T_max = 60); `--config` selects the other BASELINE configurations:

    P12      configs[0]  B = 32,  36 sensors, T = 215   (the reference's CPU-runnable case)
    P19      configs[1]  B = 128, 34 sensors, T = 60    (default)
    PAM      configs[2]  B = 256, 17 sensors, T = 600, 8 classes, no static branch
    P19x4    configs[3]  B = 256 per GPU (1024 over 4 GPUs), leave-10-sensors-out mask
    LARGEx8  configs[4]  B = 512 per GPU (4096 over 8 GPUs), 128 sensors, T = 256

Weak scaling: every rank owns its own per-GPU batch; the only collective is the NCCL all-reduce of the
flat gradient bucket (two buckets, the first overlapped with the observation-propagation backward).

Timing protocol: W >= 3 warm-up steps; K timed steps, each bracketed by CUDA events on the launching stream
with an L2 flush (256 MiB write + read-back) before it, outside the event pair; the per-step times of all
ranks are all-gathered, each step counts as the MAX over ranks, `ms_per_step` is the MEDIAN over steps
(p90 / max / mean and the per-rank medians are reported next to it); value = global batch / median.

Printed JSON line (rank 0):
  value     samples/s, whole job, inputs resident in HBM, step = one CUDA-graph replay of TrainStep
  e2e       samples/s through the drop-in nn.Module API (model.forward -> CrossEntropyLoss -> backward ->
            FlatAdam.step) with pinned HOST batches; one batch upload (H2D, on a copy stream, overlapping the
            previous step) and the loss read-back (D2H) inside every timed step
  roofline  the observation-propagation (message-passing) layer kernel: algorithmic bytes
            8*N*C per (sample, layer) / CUDA-event time, at a row count with >= 1 GiB of traffic
            (`rows`) and at the configuration's own batch (`at_config`)
  cpu_baseline  the CPU restatement of the reference (oracle/, same per-sample loop and per-edge
            GEMMs as code/models_rd.py:322-343) timed on this box's host cores
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import warnings  # noqa: E402

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from raindrop_b200.synth import make_batch, model_config  # noqa: E402
from raindrop_b200.synth import synth_weights  # noqa: E402

warnings.filterwarnings("ignore")
L2_FLUSH_BYTES = 256 << 20   # > 126 MB L2

# name -> (synthetic model config, per-GPU batch, GPUs the BASELINE config names, make_batch options, workload string)
BENCH_CONFIGS = {
    "P12": ("P12", 32, 1, {}, "P12 synthetic (batch=32 per GPU, 36 sensors, T_max=215)"),
    "P19": ("P19", 128, 1, {}, "P19 synthetic (batch=128 per GPU, 34 sensors, T_max=60)"),
    "PAM": ("PAM", 256, 1, {}, "PAM synthetic (batch=256 per GPU, 17 sensors, T_max=600, 8-class, no static)"),
    "P19x4": ("P19", 256, 4, {"zero_sensors": 10},
              "P19 synthetic batch=1024 over 4 GPUs (256 per GPU), 34 sensors, leave-10-sensors-out mask"),
    "LARGEx8": ("LARGE", 512, 8, {}, "Synthetic large batch=4096 over 8 GPUs (512 per GPU), 128 sensors, T_max=256, dense sensor graph"),
}
STEP_DESC = "Raindrop_v2 training step: fwd + CrossEntropy + bwd + Adam, dropout 0.2"


def workload_string(name):
    return "%s %s" % (BENCH_CONFIGS[name][4], STEP_DESC)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        p = json.load(open(path))
        return float(p["hbm_gbs"]), float(p.get("bf16_tflops", 0.0)) or None, "measured (MEASURED_PEAKS.json)"
    return 6650.0, None, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs (rank 0)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc, self.lines, self.index = None, [], index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def mark(self):
        """Samples before this point are warm-up / idle, not the timed region."""
        self.skip = len(self.lines)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm, mx, reasons = [], None, set()
        for ln in self.lines[getattr(self, "skip", 0):]:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def dist_setup(n_gpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    elif n_gpus > 1:
        raise SystemExit("--gpus %d needs torchrun (one process per GPU)" % n_gpus)
    return world, rank, local


def build_model(cfg, device):
    from raindrop_b200.models_rd import Raindrop_v2
    torch.manual_seed(1)   # code/Raindrop.py:58
    gs = torch.ones(cfg["d_inp"], cfg["d_inp"])
    kw = {} if cfg["static"] else {"static": False}
    m = Raindrop_v2(cfg["d_inp"], cfg["d_model"], cfg["nhead"], cfg["nhid"], cfg["nlayers"], cfg["dropout"],
                    cfg["max_len"], cfg["d_static"], cfg["MAX"], 0.5, "mean", cfg["n_classes"], gs, **kw)
    synth_weights(m, cfg, seed=7)      # random-init weights of the named architecture, same on every rank
    return m.to(device).train()


def flush_l2(buf):
    """Write a buffer larger than L2, then read it back: the write evicts everything, the read leaves the
    cache full of CLEAN lines (otherwise the timed kernel pays for writing back ~126 MB of dirty zeros)."""
    buf.zero_()
    buf.sum()


def timed_steps(step_fn, steps, flush_buf):
    """Per-step CUDA-event timing; the L2 flush between steps sits outside the event pairs."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for s, e in ev:
        flush_l2(flush_buf)
        s.record()
        step_fn()
        e.record()
    torch.cuda.synchronize()
    return [s.elapsed_time(e) for s, e in ev]


def summarize(per_step, world, device):
    """per_step: this rank's CUDA-event times (ms).  All ranks' lists are gathered; a step costs what its
    slowest rank took; the headline is the MEDIAN over steps."""
    t = torch.tensor(per_step, dtype=torch.float64, device=device)
    if world > 1:
        allt = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        allt = torch.stack(allt)                      # [world, steps]
    else:
        allt = t[None]
    step_max = allt.max(dim=0).values.cpu().tolist()
    srt = sorted(step_max)
    n = len(srt)
    return {"median": statistics.median(srt), "mean": sum(srt) / n, "p90": srt[min(n - 1, int(0.9 * n))],
            "max": srt[-1], "min": srt[0],
            "per_rank_median": [round(statistics.median(r), 4) for r in allt.cpu().tolist()]}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """name -> tensor, written as out_dir/<name>.npy in float32.  If they exceed DUMP_LIMIT_BYTES in all, every array
    larger than an even share of the limit is replaced by that many elements at fixed, seeded positions."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_LIMIT_BYTES // 4 // len(arrays)
    over = sum(t.numel() for t in arrays.values()) * 4 > DUMP_LIMIT_BYTES
    for name, t in arrays.items():
        a = t.detach().float().cpu()
        if over and a.numel() > share:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:share].sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def _round_tf32(t):
    """RN to TF32 with integer ops (bench-side data prep, so the timed launch is the GEMM kernel alone)."""
    i = t.contiguous().view(torch.int32)
    return ((i + 0x1000) & ~0x1FFF).view(torch.float32)


def roofline_leg(cfg, batch, device):
    """Message-passing layer kernel alone (rd_obprop_fwd on TF32-exact operands, no rounding pre-pass):
    algorithmic bytes = read x[rows,C] + write out[rows,C]; algorithmic flops = 2*rows*C^2."""
    from raindrop_b200 import lib as L
    lib = L.load()
    N, C = cfg["d_inp"], cfg["max_len"] * cfg["d_ob"]
    hbm_peak, bf16_peak, how = peaks()
    tf32_peak = bf16_peak / 2 if bf16_peak else None       # TF32 issues at half the bf16 rate
    big_rows = max(batch * N, ((1 << 30) // (C * 8) // N + 1) * N)     # >= 1 GiB of activation traffic
    out = {}
    for tag, rows in (("large", big_rows), ("at_config", batch * N)):
        x = _round_tf32(torch.randn(rows, C, device=device))
        W = _round_tf32(torch.randn(C, C, device=device) / C ** 0.5)
        b = torch.zeros(C, device=device)
        s = torch.ones(N, device=device)
        y = torch.empty_like(x)

        def fn():
            L.check(lib.rd_obprop_fwd(x.data_ptr(), W.data_ptr(), b.data_ptr(), s.data_ptr(), N, rows, C, y.data_ptr(),
                                      None, L.stream_ptr()), "rd_obprop_fwd")
        for _ in range(3):
            fn()
        flush = torch.empty(L2_FLUSH_BYTES // 4, dtype=torch.float32, device=device)
        ts = timed_steps(fn, 20, flush)
        ms = sum(ts) / len(ts)
        gb = rows * C * 8 / 1e9
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms_b2b = e0.elapsed_time(e1) / 10
        out[tag] = dict(rows=rows, ms=ms, achieved=gb / (ms * 1e-3), frac=gb / (ms * 1e-3) / hbm_peak,
                        tflops=2.0 * rows * C * C / (ms * 1e-3) / 1e12, ms_b2b=ms_b2b, frac_b2b=gb / (ms_b2b * 1e-3) / hbm_peak)
        del x, y
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "obprop_tc_traffic.json")
    if os.path.isfile(tpath) and C == 240:
        traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
    big = out["large"]
    tensor_frac = (big["tflops"] / tf32_peak) if tf32_peak else None
    # C/4 flop per byte against the TF32 ridge: HBM binds at C=240, both are close at 860/1024, tensor at 2400
    bound = "tensor" if (tensor_frac is not None and tensor_frac > big["frac"]) else "hbm"
    r = {"kernel": "obprop_tc_kernel (tcgen05 TF32 + TMA, one ob-prop layer, C=%d)" % C, "bound": bound,
         "peak_source": how, "rows": big["rows"], "ms_per_launch": round(big["ms"], 5), "traffic": traffic,
         "algorithmic_bytes_per_launch": big["rows"] * C * 8, "algorithmic_flops_per_launch": 2 * big["rows"] * C * C,
         "hbm": {"achieved": round(big["achieved"], 1), "peak": hbm_peak, "unit": "GB/s", "frac": round(big["frac"], 4)},
         "tensor": {"achieved": round(big["tflops"], 1), "peak": tf32_peak, "unit": "TFLOP/s (tf32 = measured bf16 peak / 2)",
                    "frac": round(tensor_frac, 4) if tensor_frac is not None else None},
         "back_to_back": {"ms_per_launch": round(big["ms_b2b"], 5), "frac": round(big["frac_b2b"], 4),
                          "note": "no L2 flush between launches (same protocol as the measured copy peak)"},
         "at_config": {"rows": out["at_config"]["rows"], "ms_per_launch": round(out["at_config"]["ms"], 5),
                       "achieved": round(out["at_config"]["achieved"], 1), "frac": round(out["at_config"]["frac"], 4),
                       "tflops": round(out["at_config"]["tflops"], 1),
                       "note": "the configuration's own batch: %d rows" % out["at_config"]["rows"]}}
    if bound == "hbm":
        r.update(achieved=r["hbm"]["achieved"], peak=hbm_peak, unit="GB/s", frac=r["hbm"]["frac"])
    else:
        r.update(achieved=r["tensor"]["achieved"], peak=tf32_peak, unit="TFLOP/s", frac=r["tensor"]["frac"])
    return r


def cpu_reference_leg(name, steps, warmup, budget_s=25.0):
    """The CPU restatement of the reference (oracle/): same per-sample Python loop with per-edge
    lin_value GEMMs and torch.nn.TransformerEncoder as code/models_rd.py:322-358, train mode
    (dropout 0.2), CrossEntropy + backward + Adam(lr=1e-4) like code/Raindrop.py:319-324.
    A step is a BOUNDED sample of the workload: the first `b_cpu` samples of the per-GPU batch (all of it
    for P12 / P19; per-sample cost is independent of B in the reference's per-sample loop)."""
    from oracle.raindrop_oracle import build_oracle_model       # the checker, timed as the baseline
    cfg_name, batch, _, opts, _ = BENCH_CONFIGS[name]
    cfg = model_config(cfg_name, dropout=0.2)
    b_cpu = {"P12": 32, "P19": 128, "PAM": 16, "P19x4": 128, "LARGEx8": 4}[name]
    b_cpu = min(b_cpu, batch)
    model = build_oracle_model(cfg).train()
    synth_weights(model, cfg, seed=7)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    full = make_batch(cfg, b_cpu, seed=1000 * 2, **opts)

    def one(b):
        logits, _, _ = model.forward(b["src"], b["static"], b["times"], b["lengths"])
        loss = F.cross_entropy(logits, b["y"])
        opt.zero_grad()
        loss.backward()
        opt.step()
        return loss.item()

    # the path is thousands of tiny ops: more threads is not always faster.  Probe thread counts on the SAME
    # kind of step that is timed (train step on a slice of the batch) and keep the best.
    ncpu = os.cpu_count() or 1
    pb = max(1, min(8, b_cpu))
    probe = {k: (v[:, :pb] if k in ("src", "times") else (v[:pb] if v is not None else None)) for k, v in full.items()}
    best_t, threads = None, 1
    for cand in sorted({c for c in (4, 8, 16, 32, 64, ncpu) if c <= ncpu}):
        torch.set_num_threads(cand)
        one(probe)
        t0 = time.perf_counter()
        one(probe)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best_t, threads = dt, cand
    torch.set_num_threads(threads)
    for _ in range(max(1, warmup)):
        one(full)
    ts = []
    t_begin = time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        one(full)
        ts.append(time.perf_counter() - t0)
        if time.perf_counter() - t_begin > budget_s:
            break
    sec = statistics.median(ts)
    return {"value": round(b_cpu / sec, 2), "unit": "samples/s", "cores": threads, "kind": "port",
            "sample": "%d train steps (fwd+CE+bwd+Adam, dropout 0.2) on %d of the %d samples of a %s batch after %d warm-up, "
                      "median %.2f s/step; torch %s CPU, %d threads (best of a probe over thread counts on the same "
                      "train step; host has %d logical CPUs)"
                      % (len(ts), b_cpu, batch, name, max(1, warmup), sec, torch.__version__, threads, ncpu),
            "sec_per_step": sec, "steps": len(ts), "samples_per_step": b_cpu}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.config
    batch = BENCH_CONFIGS[name][1]
    cb = cpu_reference_leg(name, steps=max(1, min(args.steps, 20)), warmup=max(1, min(args.warmup, 3)), budget_s=150.0)
    line = {"impl": "reference", "metric": "samples/sec (%s-shape synthetic) training step" % BENCH_CONFIGS[name][0],
            "value": cb["value"],
            "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(cb["sec_per_step"] * 1e3, 2), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(name), "global_batch": batch * args.gpus, "per_gpu_batch": batch,
                       "note": "reference is CPU-only here: single process on rank 0's host cores, %d timed steps of %d samples"
                               % (cb["steps"], cb["samples_per_step"])},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="P19", choices=sorted(BENCH_CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    if args.warmup < 3:
        args.warmup = 3

    from raindrop_b200 import lib as L
    from raindrop_b200.optim import FlatAdam
    from raindrop_b200.train import TrainStep, allreduce_gradients
    world, rank, local = dist_setup(args.gpus)
    device = torch.device("cuda", local if world > 1 else 0)
    torch.cuda.set_device(device)
    cfg_name, BATCH, named_gpus, opts, _ = BENCH_CONFIGS[args.config]
    cfg = model_config(cfg_name, dropout=0.2)
    lib = L.load()
    flush = torch.empty(L2_FLUSH_BYTES // 4, dtype=torch.float32, device=device)
    # clock sampler runs on rank 0 from BEFORE the first barrier (so starting it never sits between a barrier and
    # the timed loop); samples taken before `mark()` are discarded
    sampler = ClockSampler(device.index or 0)
    if rank == 0:
        sampler.start()

    # ---- leg 1: device-resident TrainStep, one CUDA graph per step ------------------------------
    model = build_model(cfg, device)
    ts = TrainStep(model, BATCH, lr=1e-4, use_graph=True)
    host_batches = [make_batch(cfg, BATCH, seed=1000 * 2 + 17 * rank + i, pin=True, **opts) for i in range(4)]
    ts.load_batch(host_batches[0])
    n0 = lib.rd_launch_count()
    ts._enqueue()                      # eager once: counts our launches per step
    launches_per_step = int(lib.rd_launch_count() - n0)
    graph_note = "one CUDA-graph replay (TrainStep)"
    try:
        ts.capture(warmup=2)
    except Exception as exc:  # noqa: BLE001  (e.g. NCCL refusing stream capture): run the same step eagerly
        ts.use_graph, ts.graph = False, None
        graph_note = "eager TrainStep (graph capture failed: %r)" % (exc,)
        torch.cuda.synchronize()
    for _ in range(args.warmup):
        ts.step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.mark()
    t_wall = time.perf_counter()
    per_step = timed_steps(ts.step, args.steps, flush)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall = time.perf_counter() - t_wall
    clocks = sampler.stop() if rank == 0 else None
    dev = summarize(per_step, world, device)
    ms_per_step = dev["median"]
    value = world * BATCH / (ms_per_step * 1e-3)
    loss_graph = float(ts.loss.item())
    if args.dump_outputs and rank == 0:
        outs = {"loss": ts.loss, "logits": ts.logits}
        for (key, _), p, off in zip(ts.plan.fields, model.used_parameters(), ts.offsets):
            outs["param." + key] = p.data
            outs["grad." + key] = ts.flat_g[off:off + p.numel()].view(p.shape)
        dump_outputs(args.dump_outputs, outs)

    # ---- leg 2: end to end through the drop-in module API, host batches ---------------------------
    model2 = build_model(cfg, device)
    opt = FlatAdam(model2, lr=1e-4)
    crit = torch.nn.CrossEntropyLoss()
    keys = [k for k in ("src", "times", "static", "y") if host_batches[0][k] is not None]
    h2d = sum(host_batches[0][k].numel() * host_batches[0][k].element_size() for k in keys)
    copy_stream = torch.cuda.Stream(device=device)
    slots = [{k: torch.empty_like(host_batches[0][k], device=device) for k in keys} for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    state = {"i": 0, "loss": 0.0}

    def upload(i):
        """pinned host batch i -> device slot i % 2 on the copy stream (overlaps the step that is running)"""
        hb, slot = host_batches[i % len(host_batches)], slots[i % 2]
        with torch.cuda.stream(copy_stream):
            for k in keys:
                slot[k].copy_(hb[k], non_blocking=True)
            ready[i % 2].record(copy_stream)

    def e2e_step():
        i = state["i"]
        state["i"] += 1
        upload(i + 1)                                              # H2D of the NEXT batch, inside this timed step
        torch.cuda.current_stream().wait_event(ready[i % 2])
        d = slots[i % 2]
        lengths = torch.sum(d["times"] > 0, dim=0)                 # code/Raindrop.py:317
        outputs, _, _ = model2.forward(d["src"], d.get("static"), d["times"], lengths)   # code/Raindrop.py:319
        opt.zero_grad()
        loss = crit(outputs, d["y"])
        loss.backward()
        allreduce_gradients(model2)
        opt.step()
        state["loss"] = loss.item()                                # D2H read of the step's result

    upload(0)
    for _ in range(args.warmup):
        e2e_step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e2e_times = timed_steps(e2e_step, args.steps, flush)
    if world > 1:
        dist.barrier()
    e2e = summarize(e2e_times, world, device)
    e2e_value = world * BATCH / (e2e["median"] * 1e-3)

    # ---- leg 3: device-resident training set (raindrop_b200.data): no batch bytes over PCIe ---------------
    # the whole (synthetic) training split lives in HBM; per step ONE kernel assembles the batch from the epoch's
    # index matrix (uploaded once per epoch, code/Raindrop.py:292-309) straight into the TrainStep buffers
    from raindrop_b200.data import DeviceDataset, EpochSampler
    n_train = 16 * BATCH
    pool = make_batch(cfg, n_train, seed=777 + rank, **opts)
    dds = DeviceDataset(pool["src"], pool["static"], pool["times"], pool["y"], device=device)
    import numpy as _np
    _np.random.seed(1234 + rank)
    sampler = EpochSampler(pool["y"].numpy(), batch_size=BATCH, strategy=2 if cfg["n_classes"] == 2 else 3, device=device)
    epoch_idx = sampler.epoch()
    dd_state = {"i": 0}

    def dd_step():
        dds.fill(ts, epoch_idx[dd_state["i"] % epoch_idx.shape[0]])
        dd_state["i"] += 1
        ts.step()

    for _ in range(args.warmup):
        dd_step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    dd = summarize(timed_steps(dd_step, args.steps, flush), world, device)
    dd_value = world * BATCH / (dd["median"] * 1e-3)

    # ---- leg 4: whole-validation-set evaluation (evaluate_standard, code/utils_rd.py:310-320), sharded ----------
    from raindrop_b200.train import evaluate_sharded
    n_val = {"P19": 3880, "P12": 1199, "PAM": 533}.get(cfg_name, 4 * BATCH)          # SURVEY.md section 3.2
    val = make_batch(cfg, n_val, seed=4242, **opts)
    val_dev = {k: (v.to(device) if v is not None else None) for k, v in val.items()}
    model2.eval()

    def eval_step():
        evaluate_sharded(model2, val_dev["src"], val_dev["static"], val_dev["times"])

    for _ in range(3):
        eval_step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ev = summarize(timed_steps(eval_step, 10, flush), world, device)
    model2.train()

    if rank != 0:
        _finish(world)
        return
    line = {
        "metric": "samples/sec (%s-shape synthetic) training step" % cfg_name, "value": round(value, 1), "unit": "samples/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (tf32 operands in the ob-prop GEMMs, 3xTF32 error-compensated encoder GEMMs)",
        "data": "synthetic",
        "config": {"workload": workload_string(args.config), "global_batch": world * BATCH, "per_gpu_batch": BATCH,
                   "bench_config": args.config, "baseline_config_gpus": named_gpus,
                   "precision": "fp32 storage and accumulation; ob-prop GEMM operands rounded to TF32 (forward error 3e-4), "
                                "encoder GEMMs error-compensated 3xTF32 (fp32-level)",
                   "parallelism": "sample-sharded dp%d, NCCL all-reduce of the flat grad bucket in 2 pieces (first overlaps the ob-prop backward)" % world,
                   "l2": "flushed between timed steps (256 MiB write + read-back, outside the per-step CUDA-event pairs)",
                   "step": graph_note, "wall_ms_per_step_incl_flush": round(wall / args.steps * 1e3, 4)},
        "timing": {"statistic": "median over steps of (max over ranks of the per-step CUDA-event time)",
                   "ms_median": round(dev["median"], 4), "ms_mean": round(dev["mean"], 4), "ms_p90": round(dev["p90"], 4),
                   "ms_max": round(dev["max"], 4), "ms_min": round(dev["min"], 4), "per_rank_median_ms": dev["per_rank_median"]},
        "clocks": clocks,
        "e2e": {"value": round(e2e_value, 1), "unit": "samples/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
                "ms_per_step": round(e2e["median"], 4), "ms_mean": round(e2e["mean"], 4), "ms_p90": round(e2e["p90"], 4),
                "ms_max": round(e2e["max"], 4), "per_rank_median_ms": e2e["per_rank_median"],
                "path": "pinned host batch -> H2D (copy stream, one batch ahead) -> models_rd.Raindrop_v2.forward -> "
                        "CrossEntropyLoss -> backward -> raindrop_b200.optim.FlatAdam.step -> loss.item()"},
        "device_dataset": {"value": round(dd_value, 1), "unit": "samples/s", "ms_per_step": round(dd["median"], 4),
                           "note": "training split resident in HBM (%d samples per rank), batch assembled on the device by "
                                   "rd_assemble_batch from the epoch's balanced index matrix (1 launch) + TrainStep graph replay; "
                                   "0 batch bytes over PCIe per step" % n_train},
        "eval": {"value": round(n_val / (ev["median"] * 1e-3), 1), "unit": "samples/s", "batch": n_val,
                 "ms_per_pass": round(ev["median"], 4),
                 "note": "evaluate_sharded: the whole validation set as one batch per pass (code/utils_rd.py:310-320), "
                         "samples sharded over %d rank(s), logits all-gathered; eval mode, no_grad" % world},
        "gpu_launches": launches_per_step * args.steps,
        "gpu_launches_per_step": launches_per_step,
        "final_loss": {"graph": round(loss_graph, 5), "e2e": round(state["loss"], 5)},
    }
    if not args.no_roofline:
        line["roofline"] = roofline_leg(cfg, BATCH, device)
    if world == 1 and not args.no_cpu_baseline:
        # separate process (own thread pool, hard time limit) so a slow host cannot stall the bench
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "5",
                                "--warmup", "1", "--config", args.config], capture_output=True, text=True, timeout=300)
            ref = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
            line["cpu_baseline"] = ref["cpu_baseline"]
        except Exception as exc:  # noqa: BLE001
            line["cpu_baseline"] = {"value": None, "unit": "samples/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": "cpu leg failed or timed out: %r" % (exc,)}
    print(json.dumps(line), flush=True)
    _finish(world)


def _finish(world):
    """destroy_process_group() was observed to hang on this pool after NCCL work has been captured in a
    CUDA graph; every rank is done and synchronised here, so leave without tearing the communicator down."""
    if world > 1:
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()

"""Input attributions of a trained Raindrop_v2 (drop-in module): saliency and integrated gradients over sensors x time,
the static features and the timestamps.

Both go through torch.autograd.grad on the inputs with the model's parameters frozen for the call, so the backward is
rd_raindrop_v2_bwd_inputs without any parameter work (no weight-gradient GEMMs, no LayerNorm column sums).
"""
import contextlib
import ctypes as C

import torch

from . import lib as L


@contextlib.contextmanager
def _frozen(model):
    """requires_grad off for every parameter (and the flat leaf of a bound FlatAdam) for the duration of the call."""
    flat = model._flat_optim() if getattr(model, "_flat_optim", None) is not None else None
    params = list(model.parameters()) + ([flat.flat_p] if flat is not None else [])
    before = [p.requires_grad for p in params]
    try:
        for p in params:
            p.requires_grad_(False)
        yield
    finally:
        for p, r in zip(params, before):
            p.requires_grad_(r)


def _device(model):
    return next(model.parameters()).device


def _input_grads(model, src, static, times, lengths, target):
    """logits of (src, static, times) and d logits[b, target[b]] / d (src, static, times), summed over b."""
    src = src.detach().requires_grad_(True)
    times = times.detach().requires_grad_(True)
    static = None if static is None else static.detach().requires_grad_(True)
    with _frozen(model), torch.enable_grad():
        logits, _, _ = model(src, static, times, lengths)
        if target is None:
            target = logits.detach().argmax(1)
        sel = logits.gather(1, target.view(-1, 1)).sum()
        inputs = [src, times] + ([static] if static is not None else [])
        grads = torch.autograd.grad(sel, inputs)
    return logits.detach(), target, grads[0], (grads[2] if static is not None else None), grads[1]


def _prep(model, src, static, times, lengths, target):
    dev = _device(model)
    f32 = dict(device=dev, dtype=torch.float32)
    src = src.to(**f32).contiguous()
    times = times.to(**f32).contiguous()
    static = None if static is None else static.to(**f32).contiguous()
    lengths = lengths.to(device=dev, dtype=torch.int64).contiguous()
    target = None if target is None else torch.as_tensor(target, device=dev, dtype=torch.int64).reshape(-1)
    return src, static, times, lengths, target


def saliency(model, src, static, times, lengths, target=None):
    """Gradient of logits[b, target[b]] (default target: the argmax class) with respect to the inputs.

    Returns {"src": [T, B, N] (the value half of src; the mask half takes no part in the output), "static": [B, d_static]
    or None, "times": [T, B], "target": [B], "logits": [B, n_classes]}."""
    src, static, times, lengths, target = _prep(model, src, static, times, lengths, target)
    N = src.shape[2] // 2
    logits, target, d_src, d_static, d_times = _input_grads(model, src, static, times, lengths, target)
    return {"src": d_src[..., :N], "static": d_static, "times": d_times, "target": target, "logits": logits}


def _default_max_batch(model):
    """Samples per chunk: activation workspace + backward scratch (rd_workspace_bytes, rd_backward_scratch_bytes) of
    the chunk within a quarter of the free device memory."""
    lib = L.load()
    plan = model._plan
    dims = plan._make_dims(64, model.training)
    per64 = lib.rd_workspace_bytes(C.byref(dims)) + lib.rd_backward_scratch_bytes(C.byref(dims))
    if per64 == 0:
        L.check(-2, "rd_workspace_bytes")
    free, _ = torch.cuda.mem_get_info(_device(model))
    return max(1, int((free // 4) * 64 // per64))


def integrated_gradients(model, src, static, times, lengths, target=None, baseline=None, steps=32, max_batch=None):
    """Integrated gradients of logits[b, target[b]] over the value half of src and over static, along the straight
    path from `baseline` (dict with optional "src" [T, B, N] and "static" [B, d_static]; zeros by default) to the input.
    The mask half of src, times and lengths are held fixed.  Midpoint Riemann sum with `steps` points
    alpha_k = (k + 0.5) / steps; the B * steps interpolated samples run as batches of at most `max_batch` samples
    (default: sized from the activation workspace, see _default_max_batch; a chunk holds at least one whole step).

    Returns {"src": [T, B, N], "static": [B, d_static] or None, "target": [B],
             "delta": logit(x) - logit(baseline) [B], "residual": sum of the attributions - delta [B]}."""
    src, static, times, lengths, target = _prep(model, src, static, times, lengths, target)
    T, B, N2 = src.shape
    N = N2 // 2
    if steps < 1:
        raise ValueError("steps must be >= 1")
    baseline = baseline or {}
    x_v = src[..., :N]
    b_v = baseline.get("src")
    b_v = torch.zeros_like(x_v) if b_v is None else b_v.to(x_v).reshape(x_v.shape)
    b_s = None
    if static is not None:
        b_s = baseline.get("static")
        b_s = torch.zeros_like(static) if b_s is None else b_s.to(static).reshape(static.shape)
    with torch.no_grad(), _frozen(model):
        logits_x, _, _ = model(src, static, times, lengths)
        if target is None:
            target = logits_x.argmax(1)
        base_src = torch.cat([b_v, src[..., N:]], dim=-1)
        logits_b, _, _ = model(base_src, b_s, times, lengths)
    delta = (logits_x.gather(1, target.view(-1, 1)) - logits_b.gather(1, target.view(-1, 1))).view(-1)
    if max_batch is None:
        max_batch = _default_max_batch(model)
    alphas = (torch.arange(steps, device=src.device, dtype=torch.float32) + 0.5) / steps
    g_src = torch.zeros_like(x_v)
    g_static = None if static is None else torch.zeros_like(static)
    per = max(1, int(max_batch) // B)            # whole interpolation steps per chunk (at least one)
    for k0 in range(0, steps, per):
        a = alphas[k0:k0 + per]
        K = a.numel()
        # sample (k, b) of the chunk is column k * B + b
        v = b_v[:, None] + a[None, :, None, None] * (x_v - b_v)[:, None]                 # [T, K, B, N]
        s_k = torch.cat([v, src[:, None, :, N:].expand(T, K, B, N)], dim=-1).reshape(T, K * B, N2)
        t_k = times[:, None, :].expand(T, K, B).reshape(T, K * B)
        l_k = lengths.repeat(K)
        st_k = None
        if static is not None:
            st_k = (b_s[None] + a[:, None, None] * (static - b_s)[None]).reshape(K * B, -1)
        _, _, d_src, d_static, _ = _input_grads(model, s_k, st_k, t_k, l_k, target.repeat(K))
        g_src += d_src.view(T, K, B, N2)[..., :N].sum(1)
        if static is not None:
            g_static += d_static.view(K, B, -1).sum(0)
    attr_src = (x_v - b_v) * g_src / steps
    attr_static = None if static is None else (static - b_s) * g_static / steps
    total = attr_src.sum(dim=(0, 2)) + (attr_static.sum(1) if attr_static is not None else 0.0)
    return {"src": attr_src, "static": attr_static, "target": target, "delta": delta, "residual": total - delta}

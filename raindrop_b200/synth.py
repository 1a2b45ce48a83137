"""Synthetic irregularly-sampled time series of P12 / P19 / PAM shape (SURVEY.md section 8d).

The real `PTdict_list.npy` files are not shipped with the reference (README.md:239-253), so every
benchmark and parity test runs on seeded synthetic tensors that follow the conventions of the
reference's host-side tensorisation:

  * `src[T, B, 2N]  = cat([values * mask, mask], -1)`   (code/utils_rd.py:164-175, 221-257)
  * `times[T, B]`   strictly increasing positive hours on valid rows, zero padding afterwards
  * `lengths[B]     = sum(times > 0, dim=0)`            (code/Raindrop.py:317)
  * `static[B, d_static]` or None (PAM)                 (code/Raindrop.py:311-315)
  * labels balanced (code/Raindrop.py:303-305)

Weights for full-size parity cases are generated per state-dict key from a counter-based stream
(`synth_state_dict`) so a fixture only has to store seeds and outputs, not megabytes of weights.
"""
import zlib

import numpy as np
import torch

# hyper-parameters exactly as code/Raindrop.py:105-148 derives them (d_ob = 4, d_model = 4 N,
# nhid = 2 d_model, nlayers = 2, nhead = 2, dropout = 0.2, MAX = 100)
CONFIGS = {
    # BASELINE.json configs[0]: reference CPU-runnable correctness case
    "P12": dict(d_inp=36, max_len=215, d_static=9, n_classes=2, static=True, batch=32, p_obs=0.2),
    # BASELINE.json configs[1]: the configuration the metric is quoted on
    "P19": dict(d_inp=34, max_len=60, d_static=6, n_classes=2, static=True, batch=128, p_obs=0.2),
    # BASELINE.json configs[2]
    "PAM": dict(d_inp=17, max_len=600, d_static=0, n_classes=8, static=False, batch=256, p_obs=0.4),
    # BASELINE.json configs[4] (per-GPU batch 512)
    "LARGE": dict(d_inp=128, max_len=256, d_static=6, n_classes=2, static=True, batch=512, p_obs=1.0),
    # tiny shapes for exhaustive parity / golden fixtures
    "TINY": dict(d_inp=5, max_len=12, d_static=3, n_classes=2, static=True, batch=3, p_obs=0.5),
    "TINY8": dict(d_inp=6, max_len=10, d_static=0, n_classes=8, static=False, batch=4, p_obs=0.6),
}


def model_config(name, dropout=0.2):
    c = dict(CONFIGS[name])
    c["name"] = name
    c["d_ob"] = 4
    c["d_model"] = c["d_inp"] * 4
    c["nhid"] = 2 * c["d_model"]
    c["nlayers"] = 2
    c["nhead"] = 2
    c["dropout"] = dropout
    c["MAX"] = 100
    return c


def make_batch(cfg, batch=None, seed=0, first_time_zero=False, full_length=False,
               zero_sensors=0, device="cpu", pin=False):
    """Returns dict(src, static, times, lengths, y) on `device` (float32 / int64).

    `first_time_zero` reproduces real P12/PAM data where the first timestamp is 0 so that
    `lengths = #(t > 0)` undercounts by one (code/utils_rd.py:248, SURVEY.md section 7).
    `zero_sensors=k` zeroes the value columns of k random sensors per sample, mask columns
    untouched -- the "leave-k-sensors-out" setting of code/Raindrop.py:216-223.
    """
    B = int(batch or cfg["batch"])
    T, N = cfg["max_len"], cfg["d_inp"]
    g = torch.Generator().manual_seed(int(seed))
    if full_length or cfg["name"] == "PAM":
        n_obs = torch.full((B,), T, dtype=torch.int64)
    else:
        lo = 20 if cfg["name"] == "P12" else 2
        n_obs = torch.randint(min(lo, T), T + 1, (B,), generator=g)
    t_idx = torch.arange(T)[:, None]
    valid = (t_idx < n_obs[None, :])                                   # [T, B]
    gaps = torch.rand(T, B, generator=g) + 0.05
    times = torch.cumsum(gaps, 0)
    if first_time_zero:
        times = times - times[0:1]
    times = (times * valid).float()
    m = (torch.rand(T, B, N, generator=g) < cfg["p_obs"]) & valid[:, :, None]
    v = torch.randn(T, B, N, generator=g) * m
    if zero_sensors:
        for b in range(B):
            idx = torch.randperm(N, generator=g)[:zero_sensors]
            v[:, b, idx] = 0.0
    src = torch.cat([v, m.float()], -1).float().contiguous()
    static = torch.randn(B, cfg["d_static"], generator=g).float() if cfg["static"] else None
    y = (torch.arange(B) % cfg["n_classes"])[torch.randperm(B, generator=g)].long()
    lengths = torch.sum(times > 0, dim=0)
    out = dict(src=src, static=static, times=times.contiguous(), lengths=lengths, y=y)
    for k, t in out.items():
        if t is None:
            continue
        if pin:
            t = t.pin_memory()
        out[k] = t.to(device) if device != "cpu" else t
    return out


def _stream(seed, key, n):
    """Counter-based uniform(0,1) stream: depends only on (seed, key), not on call order."""
    ss = np.random.SeedSequence([int(seed), zlib.crc32(key.encode())])
    return np.random.Generator(np.random.PCG64(ss)).random(n, dtype=np.float64)


# state-dict keys that receive gradient on the live path (SURVEY.md section 0.2 / 8a18)
def used_param_keys(cfg):
    keys = []
    if cfg["static"]:
        keys += ["emb.weight", "emb.bias"]
    for l in range(cfg["nlayers"]):
        p = "transformer_encoder.layers.%d." % l
        keys += [p + s for s in ("self_attn.in_proj_weight", "self_attn.in_proj_bias",
                                 "self_attn.out_proj.weight", "self_attn.out_proj.bias",
                                 "linear1.weight", "linear1.bias", "linear2.weight", "linear2.bias",
                                 "norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias")]
    for ob in ("ob_propagation", "ob_propagation_layer2"):
        keys += [ob + ".lin_value.weight", ob + ".lin_value.bias"]
    keys += ["mlp_static.0.weight", "mlp_static.0.bias", "mlp_static.2.weight", "mlp_static.2.bias"]
    return keys


def keyed_values(seed, key, shape, scale=1.0):
    """Values of state-dict entry `key` from the keyed stream: fan-in scaled uniform for matrices, LayerNorm
    weights near one, other vectors near zero (perturbed so that every term is exercised)."""
    u = torch.from_numpy(_stream(seed, key, int(np.prod(shape)))).view(shape).float()
    if key.endswith("norm1.weight") or key.endswith("norm2.weight"):
        return 1.0 + 0.2 * (u - 0.5)
    if len(shape) == 1:
        return 0.2 * (u - 0.5)
    return (2 * u - 1) * (scale * (3.0 / shape[1]) ** 0.5)


def synth_weights(model, cfg, seed=7, scale=1.0):
    """Overwrites the USED parameters of `model` (reference, oracle or drop-in: same keys) and its
    `R_u` attribute with values from the keyed stream (`keyed_values`).  Returns R_u."""
    sd = model.state_dict()
    with torch.no_grad():
        for key in used_param_keys(cfg):
            t = sd[key]
            t.copy_(keyed_values(seed, key, tuple(t.shape), scale))
        Dm = cfg["d_inp"] * cfg["d_ob"]
        r = torch.from_numpy(_stream(seed, "R_u", Dm)).float().view(1, Dm)
        r_u = (2 * r - 1) * 1.2
    model.load_state_dict(sd)
    ru = getattr(model, "R_u")
    with torch.no_grad():
        ru.copy_(r_u.to(ru.device))
    return r_u

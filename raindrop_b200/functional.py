"""torch.autograd bindings over the C ABI (librd_b200.so).  PyTorch is plumbing here: it owns the
device memory, the stream and the autograd graph; every number is produced by our CUDA kernels."""
import ctypes as C

import numpy as np
import torch

from . import lib as L

# parameters that take part in the live path, in the order they are passed to the autograd
# Function (state-dict keys of the reference model, SURVEY.md section 8b / 8a18)
_LAYER_KEYS = ["self_attn.in_proj_weight", "self_attn.in_proj_bias", "self_attn.out_proj.weight",
               "self_attn.out_proj.bias", "linear1.weight", "linear1.bias", "linear2.weight",
               "linear2.bias", "norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias"]
_HEAD_FIELDS = [("emb.weight", "emb_weight"), ("emb.bias", "emb_bias"),
                ("mlp_static.0.weight", "mlp0_weight"), ("mlp_static.0.bias", "mlp0_bias"),
                ("mlp_static.2.weight", "mlp2_weight"), ("mlp_static.2.bias", "mlp2_bias")]
_OBPROP_FIELDS = [("ob_propagation.lin_value.weight", "ob1_value_weight"),
                  ("ob_propagation.lin_value.bias", "ob1_value_bias"),
                  ("ob_propagation_layer2.lin_value.weight", "ob2_value_weight"),
                  ("ob_propagation_layer2.lin_value.bias", "ob2_value_bias")]


def used_param_fields(nlayers, static):
    """[(state-dict key, struct field path)] in Function-argument = flat-bucket order.  The order is the order
    in which the backward FINISHES gradients (head, encoder, then the two lin_value pairs), so that the bucket
    splits into a front part that can be all-reduced while the observation-propagation backward still runs
    (SURVEY.md section 8e) and a tail part (`n_obprop_fields` entries)."""
    out = []
    for key, field in _HEAD_FIELDS:
        if not static and key.startswith("emb."):
            continue
        out.append((key, (field,)))
    for l in range(nlayers):
        for k, f in zip(_LAYER_KEYS, L._LAYER_FIELDS):
            out.append(("transformer_encoder.layers.%d.%s" % (l, k), ("layer", l, f)))
    for key, field in _OBPROP_FIELDS:
        out.append((key, (field,)))
    return out


N_OBPROP_FIELDS = len(_OBPROP_FIELDS)


def _set_field(struct, path, value):
    if len(path) == 1:
        setattr(struct, path[0], value)
    else:
        setattr(getattr(struct, path[0])[path[1]], path[2], value)


def pe_timescales(max_len, d_pe=16):
    """max_len ** linspace(0, 1, d_pe/2) in fp64, cast to fp32 (code/models_rd.py:31,34)."""
    return (float(max_len) ** np.linspace(0, 1, d_pe // 2)).astype(np.float32)


class Plan:
    """Everything about one model instance that the kernels need besides the tensors."""

    def __init__(self, d_inp, d_ob, nhead, nhid, nlayers, d_static, n_classes, max_len, dropout, static, d_pe=16, emb_dim=0,
                 obprop=True):
        self.N, self.d_ob, self.nhead, self.nhid, self.nlayers = d_inp, d_ob, nhead, nhid, nlayers
        self.d_pe, self.emb_dim = d_pe, emb_dim
        self.d_static = d_static if static else 0
        self.n_classes, self.T, self.dropout = n_classes, max_len, float(dropout)
        self.static = static
        self.fields = used_param_fields(nlayers, static)
        if not obprop:          # legacy v1: no observation-propagation layers
            self.fields = self.fields[:-N_OBPROP_FIELDS]
        self.timescales = pe_timescales(max_len)
        self.node_scale = None      # [N] device tensor (rd_node_scale)
        self.R_u = None             # [1, N*d_ob] device tensor
        self.rng_state = None       # int64[2] device tensor {seed, counter}
        self.owner = None           # weakref to the module (receives the flat gradient bucket)
        self.obprop_mode = 0        # 0 auto, 1 single-pass TF32, 2 error-compensated 3xTF32 (rd_dims.obprop_mode)
        self.debug_keep_workspace = False   # tests: keep the last forward's workspace for workspace_view()
        self.last_workspace = None
        self.last_dims = None

    def dims(self, B, training):
        key = (B, bool(training), self.obprop_mode)
        cache = self.__dict__.setdefault("_dims_cache", {})
        d = cache.get(key)
        if d is not None:
            return d
        d = cache[key] = self._make_dims(B, training)
        return d

    def _make_dims(self, B, training):
        d = L.RdDims()
        d.B, d.T, d.N, d.d_ob = B, self.T, self.N, self.d_ob
        d.nhead, d.nhid, d.nlayers = self.nhead, self.nhid, self.nlayers
        d.d_static, d.n_classes = self.d_static, self.n_classes
        d.training = 1 if training else 0
        d.dropout_p = self.dropout
        d.ln_eps = 1e-5
        d.obprop_mode = int(self.obprop_mode)
        d.d_pe = 0 if self.d_pe == 16 else int(self.d_pe)
        d.emb_dim = int(self.emb_dim)
        for i, v in enumerate(self.timescales):
            d.pe_timescales[i] = float(v)
        return d


def _as_f32(t):
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


class RaindropV2Function(torch.autograd.Function):
    """logits = Raindrop_v2.forward(...) (code/models_rd.py:278-387) as ONE autograd node:
    rd_raindrop_v2_fwd in forward, rd_raindrop_v2_bwd in backward."""

    @staticmethod
    def forward(ctx, plan, training, src, static, times, lengths, *params):
        lib = L.load()
        if not src.is_cuda:
            raise L.RaindropB200Error("raindrop_b200 runs on CUDA tensors only (no CPU fallback)")
        T, B = src.shape[0], src.shape[1]
        if T != plan.T or src.shape[2] != 2 * plan.N:
            raise ValueError("src must be [max_len=%d, B, 2*d_inp=%d], got %s" % (plan.T, 2 * plan.N, tuple(src.shape)))
        dims = plan.dims(B, training)
        keep = [t if (t.dtype == torch.float32 and t.is_contiguous()) else _as_f32(t) for t in params]
        ptrs = (plan.R_u.data_ptr(),) + tuple(t.data_ptr() for t in keep)
        cached = plan.__dict__.get("_param_struct")
        if cached is not None and cached[0] == ptrs:
            P = cached[1]
        else:
            P = L.RdParams()
            P.R_u = ptrs[0]
            for (key, path), ptr_ in zip(plan.fields, ptrs[1:]):
                _set_field(P, path, ptr_)
            plan.__dict__["_param_struct"] = (ptrs, P)
        sizes = plan.__dict__.setdefault("_ws_bytes", {})
        ws_bytes = sizes.get((B, bool(training), plan.obprop_mode))
        if ws_bytes is None:
            ws_bytes = sizes[(B, bool(training), plan.obprop_mode)] = (lib.rd_workspace_bytes(C.byref(dims)),
                                                     lib.rd_backward_scratch_bytes(C.byref(dims)))
        ws_bytes, sc_bytes = ws_bytes
        if ws_bytes == 0:
            L.check(-2, "rd_workspace_bytes")
        # activation workspace: recycled through a small per-(B, mode) pool (a forward whose backward has not run
        # yet keeps its workspace; everything else reuses the last one instead of a fresh multi-MB allocation)
        pool = plan.__dict__.setdefault("_ws_pool", {}).setdefault((B, bool(training), src.device.index, plan.obprop_mode), [])
        ws = pool.pop() if pool else torch.empty(ws_bytes // 4, dtype=torch.float32, device=src.device)
        logits = torch.empty(B, plan.n_classes, dtype=torch.float32, device=src.device)
        rng = plan.rng_state
        rc = lib.rd_raindrop_v2_fwd(C.byref(dims), C.byref(P), src.data_ptr(), L.ptr(static), times.data_ptr(),
                                    lengths.data_ptr(), plan.node_scale.data_ptr(), L.ptr(rng), ws.data_ptr(),
                                    logits.data_ptr(), None, None, None, L.stream_ptr(src.device))
        L.check(rc, "rd_raindrop_v2_fwd")
        ctx.plan, ctx.dims, ctx.P, ctx.ws, ctx.pool = plan, dims, P, ws, pool
        ctx.keep = (keep, static, lengths, plan.node_scale, plan.R_u)
        ctx.sc_bytes = sc_bytes
        ctx.src_shape = tuple(src.shape)
        if plan.debug_keep_workspace:      # parity tests read named activation buffers (workspace_view)
            plan.last_workspace = ws
            plan.last_dims = dims
        elif not any(ctx.needs_input_grad):
            pool.append(ws)                # no backward will come: hand the workspace straight back
            ctx.ws = None
        return logits

    @staticmethod
    def backward(ctx, d_logits):
        lib = L.load()
        plan, dims = ctx.plan, ctx.dims
        if ctx.ws is None:
            raise L.RaindropB200Error("backward called twice (or after a no-grad forward): the activation workspace of "
                                      "this forward has been released; retain_graph is not supported")
        keep, static, lengths, node_scale, _ = ctx.keep
        d_logits = _as_f32(d_logits)
        dev = d_logits.device
        params = keep
        need = ctx.needs_input_grad
        want_in = (need[2], need[3] and static is not None, need[4])      # src, static, times
        want_params = any(need[6:])
        if any(want_in) or not want_params:
            return _backward_with_inputs(ctx, d_logits, want_in, want_params)
        owner = plan.owner() if plan.owner is not None else None
        flat, G = _grad_bucket(plan, params, dev)
        scratch = _cached_buffer(plan, "bwd", ctx.sc_bytes, dev)
        rc = lib.rd_raindrop_v2_bwd(C.byref(dims), C.byref(ctx.P), L.ptr(static), lengths.data_ptr(),
                                    node_scale.data_ptr(), ctx.ws.data_ptr(), d_logits.data_ptr(), C.byref(G),
                                    scratch.data_ptr(), L.BWD_ALL, L.stream_ptr(dev))
        L.check(rc, "rd_raindrop_v2_bwd")
        grads = torch._utils._unflatten_dense_tensors(flat, params)      # views, one C++ call
        if owner is not None:
            owner._flat_grad = flat          # the DDP bucket: one all-reduce covers every gradient
        if not plan.debug_keep_workspace:
            ctx.pool.append(ctx.ws)
        ctx.ws = None
        return (None, None, None, None, None, None) + tuple(grads)


def _grad_bucket(plan, params, dev):
    """Fresh flat gradient bucket and the rd_grads struct pointing into it (cached by base address)."""
    layout = plan.__dict__.get("_grad_layout")
    if layout is None:      # tightly packed flat bucket, one offset per used parameter
        offs, total = [], 0
        for t in params:
            offs.append(total)
            total += t.numel()
        layout = plan.__dict__["_grad_layout"] = (offs, total)
    offs, total = layout
    flat = torch.empty(total, dtype=torch.float32, device=dev)
    base = flat.data_ptr()
    cachedG = plan.__dict__.get("_grad_struct")
    if cachedG is not None and cachedG[0] == base:
        return flat, cachedG[1]
    G = L.RdGrads()
    for (key, path), off in zip(plan.fields, offs):
        _set_field(G, path, base + 4 * off)
    plan.__dict__["_grad_struct"] = (base, G)
    return flat, G


def _cached_buffer(plan, name, n_bytes, dev):
    """Device scratch that holds nothing across calls: one buffer per (name, size, device)."""
    bufs = plan.__dict__.setdefault("_scratch", {})
    key = (name, n_bytes, dev.index)
    buf = bufs.get(key)
    if buf is None:
        buf = bufs[key] = torch.empty(max(1, n_bytes // 4), dtype=torch.float32, device=dev)
    return buf


def _input_grad_buffers(shape_src, static, want_in, dev):
    """d_src / d_static / d_times tensors (None where not wanted) and the rd_input_grads struct over them."""
    T, B, N2 = shape_src
    f32 = dict(dtype=torch.float32, device=dev)
    outs = (torch.empty(T, B, N2, **f32) if want_in[0] else None,
            torch.empty(static.shape, **f32) if want_in[1] else None,
            torch.empty(T, B, **f32) if want_in[2] else None)
    ig = L.RdInputGrads()
    ig.src, ig.statics, ig.times = L.ptr(outs[0]), L.ptr(outs[1]), L.ptr(outs[2])
    return outs, ig


def _backward_with_inputs(ctx, d_logits, want_in, want_params):
    """RaindropV2Function.backward when an input needs a gradient or no parameter does: rd_raindrop_v2_bwd_inputs
    (parameter gradients bit-identical to rd_raindrop_v2_bwd; none at all, and none of their launches, for a frozen
    model)."""
    lib = L.load()
    plan, dims = ctx.plan, ctx.dims
    keep, static, lengths, node_scale, _ = ctx.keep
    dev = d_logits.device
    flat, G = _grad_bucket(plan, keep, dev) if want_params else (None, None)
    scratch = _cached_buffer(plan, "bwd", ctx.sc_bytes, dev)
    in_scratch = _cached_buffer(plan, "in", lib.rd_input_grad_scratch_bytes(C.byref(dims)), dev)
    (d_src, d_static, d_times), ig = _input_grad_buffers(ctx.src_shape, static, want_in, dev)
    rc = lib.rd_raindrop_v2_bwd_inputs(C.byref(dims), C.byref(ctx.P), L.ptr(static), lengths.data_ptr(),
                                       node_scale.data_ptr(), ctx.ws.data_ptr(), d_logits.data_ptr(),
                                       C.byref(G) if G is not None else None, C.byref(ig), scratch.data_ptr(),
                                       in_scratch.data_ptr(), L.stream_ptr(dev))
    L.check(rc, "rd_raindrop_v2_bwd_inputs")
    need = ctx.needs_input_grad
    if want_params:
        grads = torch._utils._unflatten_dense_tensors(flat, keep)
        grads = tuple(g if n else None for g, n in zip(grads, need[6:]))
        owner = plan.owner() if plan.owner is not None else None
        if owner is not None:
            owner._flat_grad = flat
    else:
        grads = (None,) * len(keep)
    if not plan.debug_keep_workspace:
        ctx.pool.append(ctx.ws)
    ctx.ws = None
    return (None, None, d_src, d_static, d_times, None) + grads


class _StepSlot:
    """Static buffers + captured CUDA graphs of one (batch size, mode, device) for the flat-bucket fast path."""

    def __init__(self, plan, B, training, dev, flat):
        lib = L.load()
        self.B, self.training, self.dev = B, training, dev
        self.dims = plan.dims(B, training)
        f32 = dict(dtype=torch.float32, device=dev)
        self.src = torch.zeros(plan.T, B, 2 * plan.N, **f32)
        self.times = torch.zeros(plan.T, B, **f32)
        self.lengths = torch.ones(B, dtype=torch.int64, device=dev)
        self.static = torch.zeros(B, plan.d_static, **f32) if plan.static else None
        self.logits = torch.zeros(B, plan.n_classes, **f32)
        self.d_logits = torch.zeros(B, plan.n_classes, **f32)
        ws_bytes = lib.rd_workspace_bytes(C.byref(self.dims))
        if ws_bytes == 0:
            L.check(-2, "rd_workspace_bytes")
        self.ws = torch.empty(ws_bytes // 4, **f32)
        self.scratch = None
        self.P, self.G = L.RdParams(), L.RdGrads()
        self.P.R_u = plan.R_u.data_ptr()
        for (key, path), off in zip(plan.fields, flat.offsets):
            _set_field(self.P, path, flat.flat_p.data_ptr() + 4 * off)
            _set_field(self.G, path, flat.flat_g.data_ptr() + 4 * off)
        self.key = (flat.flat_p.data_ptr(), flat.flat_g.data_ptr(), plan.R_u.data_ptr(), plan.node_scale.data_ptr(),
                    plan.rng_state.data_ptr())
        self.fwd_calls = self.bwd_calls = 0
        self.fwd_graph = self.bwd_graph = None
        self.pending = False          # a forward whose backward has not run yet owns the buffers
        self.in_scratch = None


def _run_or_capture(slot, which, fn):
    """1st call eager (one-time kernel attribute setup must not happen inside a capture), 2nd call captured,
    afterwards one graph launch per call."""
    graph = getattr(slot, which + "_graph")
    if graph is not None:
        graph.replay()
        return
    calls = getattr(slot, which + "_calls")
    setattr(slot, which + "_calls", calls + 1)
    if calls == 0 or not GRAPHS_ENABLED or torch.cuda.is_current_stream_capturing():
        fn()
        return
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    setattr(slot, which + "_graph", g)
    g.replay()


GRAPHS_ENABLED = True


class RaindropV2FlatFunction(torch.autograd.Function):
    """Same arithmetic as RaindropV2Function for a model whose used parameters live in ONE flat leaf tensor
    (raindrop_b200.optim.FlatAdam).  Inputs are staged into static buffers so that the forward and the backward are
    each ONE CUDA-graph launch; the gradient bucket is written in place (flat_p.grad IS the bucket), so autograd
    has a single leaf to visit and nothing to copy."""

    @staticmethod
    def forward(ctx, plan, training, slot, flat, src, static, times, lengths, flat_p):
        lib = L.load()
        slot.src.copy_(src); slot.times.copy_(times); slot.lengths.copy_(lengths)
        if slot.static is not None:
            slot.static.copy_(static)

        def fwd():
            rc = lib.rd_raindrop_v2_fwd(C.byref(slot.dims), C.byref(slot.P), slot.src.data_ptr(), L.ptr(slot.static),
                                        slot.times.data_ptr(), slot.lengths.data_ptr(), plan.node_scale.data_ptr(),
                                        L.ptr(plan.rng_state), slot.ws.data_ptr(), slot.logits.data_ptr(), None, None, None,
                                        L.stream_ptr(slot.dev))
            L.check(rc, "rd_raindrop_v2_fwd")
        _run_or_capture(slot, "fwd", fwd)
        ctx.plan, ctx.slot, ctx.flat = plan, slot, flat
        slot.pending = any(ctx.needs_input_grad)
        if plan.debug_keep_workspace:
            plan.last_workspace, plan.last_dims = slot.ws, slot.dims
        return slot.logits.clone()

    @staticmethod
    def backward(ctx, d_logits):
        lib = L.load()
        plan, slot, flat = ctx.plan, ctx.slot, ctx.flat
        if not slot.pending:
            raise L.RaindropB200Error("backward called twice for one forward (retain_graph is not supported)")
        slot.d_logits.copy_(d_logits)
        if slot.scratch is None:
            slot.scratch = torch.empty(lib.rd_backward_scratch_bytes(C.byref(slot.dims)) // 4, dtype=torch.float32,
                                       device=slot.dev)

        need = ctx.needs_input_grad
        want_in = (need[4], need[5] and slot.static is not None, need[6])      # src, static, times
        want_params = need[8]
        if not any(want_in):
            def bwd():
                rc = lib.rd_raindrop_v2_bwd(C.byref(slot.dims), C.byref(slot.P), L.ptr(slot.static), slot.lengths.data_ptr(),
                                            plan.node_scale.data_ptr(), slot.ws.data_ptr(), slot.d_logits.data_ptr(),
                                            C.byref(slot.G), slot.scratch.data_ptr(), L.BWD_ALL, L.stream_ptr(slot.dev))
                L.check(rc, "rd_raindrop_v2_bwd")
            _run_or_capture(slot, "bwd", bwd)
            d_in = (None, None, None)
        else:
            # run eagerly (not graph-captured): the forward stays one graph replay, parameter gradients are still written
            # in place into the bucket
            d_in, ig = _input_grad_buffers(slot.src.shape, slot.static, want_in, slot.dev)
            if slot.in_scratch is None:
                slot.in_scratch = torch.empty(max(1, lib.rd_input_grad_scratch_bytes(C.byref(slot.dims)) // 4),
                                              dtype=torch.float32, device=slot.dev)

            rc = lib.rd_raindrop_v2_bwd_inputs(C.byref(slot.dims), C.byref(slot.P), L.ptr(slot.static),
                                               slot.lengths.data_ptr(), plan.node_scale.data_ptr(), slot.ws.data_ptr(),
                                               slot.d_logits.data_ptr(), C.byref(slot.G) if want_params else None,
                                               C.byref(ig), slot.scratch.data_ptr(), slot.in_scratch.data_ptr(),
                                               L.stream_ptr(slot.dev))
            L.check(rc, "rd_raindrop_v2_bwd_inputs")
        slot.pending = False
        if want_params:
            flat.grads_ready = True
            owner = plan.owner() if plan.owner is not None else None
            if owner is not None:
                owner._flat_grad = flat.flat_g
        # flat_p.grad already IS flat_g (written in place by the kernels): nothing for autograd to accumulate
        return (None, None, None, None) + d_in + (None, None)


def flat_forward(plan, training, flat, src, static, times, lengths):
    """Entry of the flat-bucket fast path (models_rd.Raindrop_v2.forward when a FlatAdam is bound)."""
    dev = src.device
    B = src.shape[1]
    if src.shape[0] != plan.T or src.shape[2] != 2 * plan.N:
        raise ValueError("src must be [max_len=%d, B, 2*d_inp=%d], got %s" % (plan.T, 2 * plan.N, tuple(src.shape)))
    slots = plan.__dict__.setdefault("_slots", {})
    k = (B, bool(training), dev.index)
    slot = slots.get(k)
    if slot is not None and slot.dims.obprop_mode != plan.obprop_mode:
        slot = None                      # arithmetic mode changed: new workspace layout, new graphs
    key = (flat.flat_p.data_ptr(), flat.flat_g.data_ptr(), plan.R_u.data_ptr(), plan.node_scale.data_ptr(),
           plan.rng_state.data_ptr())
    if slot is None or slot.key != key:      # pointers changed (graph / R_u / optimiser re-created): rebuild
        slot = slots[k] = _StepSlot(plan, B, bool(training), dev, flat)
    if slot.pending:
        if torch.is_grad_enabled():
            raise L.RaindropB200Error("a FlatAdam-bound model keeps ONE forward in flight per batch size: call "
                                      "loss.backward() before the next training forward (for gradient accumulation "
                                      "use torch.optim.Adam)")
        return None      # caller falls back to the general path (e.g. a no-grad probe between forward and backward)
    return RaindropV2FlatFunction.apply(plan, training, slot, flat, src, static, times, lengths, flat.flat_p)


class ObPropLayerFunction(torch.autograd.Function):
    """One observation-propagation layer on `rows` node rows at once (rd_obprop_fwd / _bwd)."""

    @staticmethod
    def forward(ctx, x, weight, bias, node_scale, mod):
        lib = L.load()
        x, weight, bias = _as_f32(x), _as_f32(weight), _as_f32(bias)
        rows, Cc = x.shape
        out = torch.empty_like(x)
        sc = torch.empty(lib.rd_obprop_fwd_scratch_bytes(rows, Cc) // 4, dtype=torch.float32, device=x.device)
        rc = lib.rd_obprop_fwd(x.data_ptr(), weight.data_ptr(), bias.data_ptr(), node_scale.data_ptr(), int(mod),
                               rows, Cc, out.data_ptr(), sc.data_ptr(), L.stream_ptr())
        L.check(rc, "rd_obprop_fwd")
        ctx.save_for_backward(x, weight, out, node_scale)
        ctx.mod = int(mod)
        return out

    @staticmethod
    def backward(ctx, d_out):
        lib = L.load()
        x, weight, out, node_scale = ctx.saved_tensors
        d_out = _as_f32(d_out)
        rows, Cc = x.shape
        d_x = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        d_w = torch.empty_like(weight)
        d_b = torch.empty(Cc, dtype=torch.float32, device=x.device)
        sc = torch.empty(lib.rd_obprop_bwd_scratch_bytes(rows, Cc) // 4, dtype=torch.float32, device=x.device)
        rc = lib.rd_obprop_bwd(x.data_ptr(), out.data_ptr(), d_out.data_ptr(), weight.data_ptr(),
                               node_scale.data_ptr(), ctx.mod, rows, Cc, L.ptr(d_x), d_w.data_ptr(), d_b.data_ptr(),
                               sc.data_ptr(), L.stream_ptr())
        L.check(rc, "rd_obprop_bwd")
        return d_x, d_w, d_b, None, None


class ObPropBetaFunction(torch.autograd.Function):
    """Observation_progation.forward(use_beta=True) for one sample (code/Ob_propagation.py:161-211) with gradients:
    rd_obprop_beta_fwd / rd_obprop_beta_bwd.  Returns (out [N, C], alpha [K], pruned edge list [2, K] (data))."""

    @staticmethod
    def forward(ctx, x, p_t, edge_weights, src_i, tgt_i, d_ob, inc_w, inc_b, map_w, val_w, val_b):
        lib = L.load()
        x, p_t, w = _as_f32(x), _as_f32(p_t), _as_f32(edge_weights)
        N, Cc = x.shape
        T = Cc // d_ob
        E = src_i.numel()
        K = E // 2
        out = torch.empty(N, Cc, dtype=torch.float32, device=x.device)
        ei = torch.empty(2, K, dtype=torch.int64, device=x.device)
        alpha = torch.empty(K, dtype=torch.float32, device=x.device)
        sc = torch.empty(lib.rd_obprop_beta_scratch_bytes(N, T, d_ob, E) // 4, dtype=torch.float32, device=x.device)
        ps = [_as_f32(t) for t in (inc_w, inc_b, map_w, val_w, val_b)]
        rc = lib.rd_obprop_beta_fwd(x.data_ptr(), p_t.data_ptr(), src_i.data_ptr(), tgt_i.data_ptr(), w.data_ptr(), E, N, T,
                                    d_ob, *[p.data_ptr() for p in ps], out.data_ptr(), ei[0].data_ptr(), ei[1].data_ptr(),
                                    alpha.data_ptr(), sc.data_ptr(), L.stream_ptr(x.device))
        L.check(rc, "rd_obprop_beta_fwd")
        ctx.save_for_backward(x, p_t, w, src_i, tgt_i, *ps)
        ctx.d_ob = d_ob
        ctx.mark_non_differentiable(ei)
        return out, alpha, ei

    @staticmethod
    def backward(ctx, d_out, d_alpha, _d_ei):
        lib = L.load()
        x, p_t, w, src_i, tgt_i, inc_w, inc_b, map_w, val_w, val_b = ctx.saved_tensors
        N, Cc = x.shape
        d_ob = ctx.d_ob
        T, E = Cc // d_ob, src_i.numel()
        dev = x.device
        d_out = _as_f32(d_out) if d_out is not None else torch.zeros(N, Cc, dtype=torch.float32, device=dev)
        d_alpha = None if d_alpha is None else _as_f32(d_alpha)
        f32 = dict(dtype=torch.float32, device=dev)
        d_x = torch.empty(N, Cc, **f32)
        d_w = torch.empty(E, **f32); d_pt = torch.empty(T, 16, **f32)
        g_iw = torch.empty_like(inc_w); g_ib = torch.empty_like(inc_b); g_mw = torch.empty_like(map_w)
        g_vw = torch.empty_like(val_w); g_vb = torch.empty_like(val_b)
        sc = torch.empty(lib.rd_obprop_beta_bwd_scratch_bytes(N, T, d_ob, E) // 4, **f32)
        rc = lib.rd_obprop_beta_bwd(x.data_ptr(), p_t.data_ptr(), src_i.data_ptr(), tgt_i.data_ptr(), w.data_ptr(), E, N, T, d_ob,
                                    inc_w.data_ptr(), inc_b.data_ptr(), map_w.data_ptr(), val_w.data_ptr(), val_b.data_ptr(),
                                    d_out.data_ptr(), L.ptr(d_alpha), d_x.data_ptr(), d_w.data_ptr(), d_pt.data_ptr(),
                                    g_iw.data_ptr(), g_ib.data_ptr(), g_mw.data_ptr(), g_vw.data_ptr(), g_vb.data_ptr(),
                                    sc.data_ptr(), L.stream_ptr(dev))
        L.check(rc, "rd_obprop_beta_bwd")
        return d_x, d_pt, d_w, None, None, None, g_iw, g_ib, g_mw, g_vw, g_vb


def obprop_beta(x, p_t, edge_index, edge_weights, d_ob, inc_w, inc_b, map_w, val_w, val_b):
    """Observation_progation.forward(use_beta=True) for one sample.  Returns (out [N, C], edge_index_pruned [2, K],
    alpha [K]); differentiable w.r.t. x, p_t, edge_weights and the five parameters."""
    src_i, tgt_i = edge_index[0].contiguous().long(), edge_index[1].contiguous().long()

    out, alpha, ei = ObPropBetaFunction.apply(x, p_t, edge_weights, src_i, tgt_i, d_ob, inc_w, inc_b, map_w, val_w, val_b)
    return out, ei, alpha


def node_scale(edge_index, edge_weights, n_nodes):
    """s[n] = sum over incoming edges of the segment softmax (rd_node_scale)."""
    lib = L.load()
    tgt = edge_index[1].contiguous().long()
    w = _as_f32(edge_weights)
    s = torch.empty(n_nodes, dtype=torch.float32, device=w.device)
    L.check(lib.rd_node_scale(tgt.data_ptr(), w.data_ptr(), tgt.numel(), n_nodes, s.data_ptr(), L.stream_ptr()),
            "rd_node_scale")
    return s


def _pe_timescales_c(max_len, d_pe):
    return (C.c_float * (d_pe // 2))(*[float(v) for v in pe_timescales(max_len, d_pe)])


def positional_encoding(times, max_len, d_pe=16):
    """[T, B] -> [T, B, d_pe] on the device (rd_positional_encoding); d_pe even, <= 64.  No autograd node: see
    PositionalEncodingFunction for the differentiable version."""
    lib = L.load()
    t = _as_f32(times)
    out = torch.empty(t.shape + (d_pe,), dtype=torch.float32, device=t.device)
    L.check(lib.rd_positional_encoding(t.data_ptr(), t.numel(), _pe_timescales_c(max_len, d_pe), d_pe, out.data_ptr(), d_pe, 0,
                                       L.stream_ptr(t.device)), "rd_positional_encoding")
    return out


class PositionalEncodingFunction(torch.autograd.Function):
    """pe = [sin(times / ts), cos(times / ts)] (code/models_rd.py:28-37) with d(pe)/d(times): the forward is
    positional_encoding; the backward (rd_positional_encoding_bwd) forms d_times from the saved sin / cos columns."""

    @staticmethod
    def forward(ctx, times, max_len, d_pe):
        pe = positional_encoding(times, max_len, d_pe)
        ctx.max_len, ctx.d_pe, ctx.shape = max_len, d_pe, times.shape
        ctx.save_for_backward(pe)
        return pe

    @staticmethod
    def backward(ctx, d_pe):
        lib = L.load()
        (pe,) = ctx.saved_tensors
        d_pe = _as_f32(d_pe)
        d_times = torch.empty(ctx.shape, dtype=torch.float32, device=pe.device)
        n = d_times.numel()
        L.check(lib.rd_positional_encoding_bwd(pe.data_ptr(), d_pe.data_ptr(), n, _pe_timescales_c(ctx.max_len, ctx.d_pe),
                                               ctx.d_pe, ctx.d_pe, 0, d_times.data_ptr(), L.stream_ptr(pe.device)),
                "rd_positional_encoding_bwd")
        return d_times, None, None


def linear(x, weight, bias=None, relu=False):
    """x [rows, in] -> [rows, out] through the encoder's projection GEMM (rd_linear_fwd); inference only."""
    lib = L.load()
    x, weight = _as_f32(x), _as_f32(weight)
    rows, in_f = x.shape
    out_f = weight.shape[0]
    out = torch.empty(rows, out_f, dtype=torch.float32, device=x.device)
    sc = torch.empty(lib.rd_linear_scratch_bytes(in_f, out_f) // 4, dtype=torch.float32, device=x.device)
    b = None if bias is None else _as_f32(bias)
    L.check(lib.rd_linear_fwd(x.data_ptr(), weight.data_ptr(), L.ptr(b), rows, in_f, out_f, int(relu), out.data_ptr(),
                              sc.data_ptr(), L.stream_ptr()), "rd_linear_fwd")
    return out


class TransformerConvFunction(torch.autograd.Function):
    """TransformerConv.forward (code/transformer_conv.py:139-207) with gradients: rd_transformer_conv_fwd / _bwd.
    x [rows, in] holds `n_graphs` graphs of `n_nodes` nodes sharing one edge list; row(node i, graph g) =
    i * node_stride + g * graph_stride.  Returns (out [rows, H*F], alpha [n_graphs, E, H])."""

    @staticmethod
    def forward(ctx, x, edge_index, edge_weights, geom, heads, out_channels, wq, bq, wk, bk, wv, bv, ws, bs):
        lib = L.load()
        n_nodes, n_graphs, node_stride, graph_stride = geom
        x = _as_f32(x)
        rows, in_ch = x.shape
        src_i = edge_index[0].contiguous().long()
        tgt_i = edge_index[1].contiguous().long()
        E = src_i.numel()
        ew = None if edge_weights is None else _as_f32(edge_weights)
        out = torch.empty(rows, heads * out_channels, dtype=torch.float32, device=x.device)
        alpha = torch.empty(n_graphs, E, heads, dtype=torch.float32, device=x.device)
        sc = torch.empty(max(1, lib.rd_transformer_conv_scratch_bytes(n_nodes, n_graphs, in_ch, heads, out_channels, E, 0) // 4),
                         dtype=torch.float32, device=x.device)
        ps = [_as_f32(t) for t in (wq, bq, wk, bk, wv, bv, ws, bs)]
        rc = lib.rd_transformer_conv_fwd(x.data_ptr(), n_nodes, n_graphs, node_stride, graph_stride, in_ch, heads, out_channels,
                                         src_i.data_ptr(), tgt_i.data_ptr(), L.ptr(ew), E, *[p.data_ptr() for p in ps],
                                         out.data_ptr(), alpha.data_ptr(), sc.data_ptr(), L.stream_ptr(x.device))
        L.check(rc, "rd_transformer_conv_fwd")
        ctx.save_for_backward(x, src_i, tgt_i, alpha, *ps)
        ctx.ew = ew
        ctx.geom, ctx.heads, ctx.out_channels = geom, heads, out_channels
        ctx.mark_non_differentiable(alpha)       # the reference only ever uses the returned alpha as data (detached by cdist/mean)
        return out, alpha

    @staticmethod
    def backward(ctx, d_out, _d_alpha):
        lib = L.load()
        x, src_i, tgt_i, alpha, wq, bq, wk, bk, wv, bv, ws, bs = ctx.saved_tensors
        n_nodes, n_graphs, node_stride, graph_stride = ctx.geom
        heads, F_ = ctx.heads, ctx.out_channels
        rows, in_ch = x.shape
        E = src_i.numel()
        d_out = _as_f32(d_out)
        dev = x.device
        d_x = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        if any(ctx.needs_input_grad[6:]):
            gw = [torch.empty(heads * F_, in_ch, dtype=torch.float32, device=dev) for _ in range(4)]
            gb = [torch.empty(heads * F_, dtype=torch.float32, device=dev) for _ in range(4)]
        else:       # frozen layer: NULL weight / bias gradients, no weight-gradient launch
            gw, gb = [None] * 4, [None] * 4
        d_ew = torch.zeros(E, dtype=torch.float32, device=dev) if (ctx.ew is not None and ctx.needs_input_grad[2]) else None
        sc = torch.empty(max(1, lib.rd_transformer_conv_scratch_bytes(n_nodes, n_graphs, in_ch, heads, F_, E, 1) // 4),
                         dtype=torch.float32, device=dev)
        rc = lib.rd_transformer_conv_bwd(x.data_ptr(), n_nodes, n_graphs, node_stride, graph_stride, in_ch, heads, F_,
                                         src_i.data_ptr(), tgt_i.data_ptr(), L.ptr(ctx.ew), E, wq.data_ptr(), bq.data_ptr(),
                                         wk.data_ptr(), bk.data_ptr(), wv.data_ptr(), bv.data_ptr(), ws.data_ptr(),
                                         alpha.data_ptr(), d_out.data_ptr(), L.ptr(d_x), L.ptr(gw[0]), L.ptr(gb[0]),
                                         L.ptr(gw[1]), L.ptr(gb[1]), L.ptr(gw[2]), L.ptr(gb[2]), L.ptr(gw[3]),
                                         L.ptr(gb[3]), L.ptr(d_ew), sc.data_ptr(), L.stream_ptr(dev))
        L.check(rc, "rd_transformer_conv_bwd")
        return (d_x, None, d_ew, None, None, None, gw[0], gb[0], gw[1], gb[1], gw[2], gb[2], gw[3], gb[3])


def transformer_conv(x, edge_index, edge_weights, heads, out_channels, wq, bq, wk, bk, wv, bv, ws, bs, geom=None):
    """TransformerConv forward with autograd (code/transformer_conv.py:139-207).  Returns (out, alpha); alpha is
    [E, heads] for a single graph, [n_graphs, E, heads] when `geom` = (n_nodes, n_graphs, node_stride, graph_stride)."""
    single = geom is None
    if single:
        geom = (x.shape[0], 1, 1, 0)
    out, alpha = TransformerConvFunction.apply(x, edge_index, edge_weights, geom, heads, out_channels, wq, bq, wk, bk, wv, bv, ws, bs)
    return out, (alpha[0] if single else alpha)


class LinearFunction(torch.autograd.Function):
    """y = x W^T + b on the error-compensated tensor-core GEMM (rd_linear_fwd); backward: dX through the same kernel
    against W^T, dW / db through the grouped weight-gradient kernel (rd_linear_wgrad_group)."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return linear(x, weight, bias)

    @staticmethod
    def backward(ctx, dy):
        lib = L.load()
        x, weight = ctx.saved_tensors
        dy = _as_f32(dy)
        dx = linear(dy, weight.t().contiguous()) if ctx.needs_input_grad[0] else None
        if not (ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2])):
            return dx, None, None           # frozen layer: no weight-gradient launch
        rows, out_f = dy.shape
        in_f = x.shape[1]
        dW = torch.empty_like(weight)
        db = torch.empty(out_f, dtype=torch.float32, device=dy.device)
        part = torch.empty(max(1, lib.rd_linear_wgrad_partial_bytes(rows, out_f, in_f) // 4), dtype=torch.float32, device=dy.device)
        it = (L.RdWgradItem * 1)()
        it[0].d_out, it[0].x, it[0].rows, it[0].out_features, it[0].in_features = dy.data_ptr(), _as_f32(x).data_ptr(), rows, out_f, in_f
        it[0].d_weight, it[0].d_bias, it[0].partial = dW.data_ptr(), db.data_ptr(), part.data_ptr()
        L.check(lib.rd_linear_wgrad_group(it, 1, L.stream_ptr(dy.device)), "rd_linear_wgrad_group")
        return dx, dW, (db if ctx.has_bias else None)


class DropoutFunction(torch.autograd.Function):
    """nn.Dropout on the library's counter-based stream (rd_dropout); the backward re-applies the same mask."""

    @staticmethod
    def forward(ctx, x, p, rng, site):
        lib = L.load()
        x = _as_f32(x)
        y = torch.empty_like(x)
        L.check(lib.rd_dropout(x.data_ptr(), x.numel(), p, rng.data_ptr(), site, y.data_ptr(), L.stream_ptr(x.device)), "rd_dropout")
        ctx.p, ctx.site = p, site
        ctx.save_for_backward(rng)
        return y

    @staticmethod
    def backward(ctx, dy):
        lib = L.load()
        (rng,) = ctx.saved_tensors
        dy = _as_f32(dy)
        dx = torch.empty_like(dy)
        L.check(lib.rd_dropout(dy.data_ptr(), dy.numel(), ctx.p, rng.data_ptr(), ctx.site, dx.data_ptr(), L.stream_ptr(dy.device)),
                "rd_dropout")
        return dx, None, None, None


class EncoderHeadFunction(torch.autograd.Function):
    """Temporal encoder + masked-mean pooling + mlp_static on a given encoder input z0 [T, B, D] (rd_encoder_head_fwd /
    _bwd): the part of the model that legacy Raindrop v1 shares with Raindrop_v2 (code/models_rd.py:168-191)."""

    @staticmethod
    def forward(ctx, plan, training, z0, static, lengths, *params):
        lib = L.load()
        z0 = _as_f32(z0)
        T, B, D = z0.shape
        dims = plan.dims(B, training)
        keep = [_as_f32(t) for t in params]
        P = L.RdParams()
        for (key, path), t in zip(plan.fields, keep):
            _set_field(P, path, t.data_ptr())
        ws = torch.empty(lib.rd_workspace_bytes(C.byref(dims)) // 4, dtype=torch.float32, device=z0.device)
        n = C.c_int64(0)
        off = lib.rd_workspace_offset(C.byref(dims), L.WS_ENC_IN, C.byref(n))
        if off < 0 or n.value != z0.numel():
            raise L.RaindropB200Error("encoder input must be [T=%d, B, D=%d], got %s" % (plan.T, n.value // max(1, T * B), tuple(z0.shape)))
        ws[off // 4: off // 4 + n.value].copy_(z0.reshape(-1))
        logits = torch.empty(B, plan.n_classes, dtype=torch.float32, device=z0.device)
        rc = lib.rd_encoder_head_fwd(C.byref(dims), C.byref(P), L.ptr(static), lengths.data_ptr(), L.ptr(plan.rng_state),
                                     ws.data_ptr(), logits.data_ptr(), None, None, None, L.stream_ptr(z0.device))
        L.check(rc, "rd_encoder_head_fwd")
        ctx.plan, ctx.dims, ctx.P, ctx.ws, ctx.keep = plan, dims, P, ws, (keep, static, lengths)
        ctx.shape = (T, B, D)
        return logits

    @staticmethod
    def backward(ctx, d_logits):
        lib = L.load()
        plan, dims = ctx.plan, ctx.dims
        keep, static, lengths = ctx.keep
        d_logits = _as_f32(d_logits)
        dev = d_logits.device
        need = ctx.needs_input_grad
        want_static = need[3] and static is not None
        want_params = any(need[5:])
        flat, G = None, None
        if want_params:
            offs, total = [], 0
            for t in keep:
                offs.append(total)
                total += t.numel()
            flat = torch.empty(total, dtype=torch.float32, device=dev)
            G = L.RdGrads()
            for (key, path), off in zip(plan.fields, offs):
                _set_field(G, path, flat.data_ptr() + 4 * off)
        sc = torch.empty(lib.rd_backward_scratch_bytes(C.byref(dims)) // 4, dtype=torch.float32, device=dev)
        dz = torch.empty(ctx.shape, dtype=torch.float32, device=dev) if (need[2] or not want_static) else None
        d_static = torch.empty(static.shape, dtype=torch.float32, device=dev) if want_static else None
        if want_params and not want_static:
            rc = lib.rd_encoder_head_bwd(C.byref(dims), C.byref(ctx.P), L.ptr(static), lengths.data_ptr(), ctx.ws.data_ptr(),
                                         d_logits.data_ptr(), C.byref(G), sc.data_ptr(), dz.data_ptr(), L.stream_ptr(dev))
            L.check(rc, "rd_encoder_head_bwd")
        else:
            rc = lib.rd_encoder_head_bwd_inputs(C.byref(dims), C.byref(ctx.P), L.ptr(static), lengths.data_ptr(),
                                                ctx.ws.data_ptr(), d_logits.data_ptr(), C.byref(G) if G is not None else None,
                                                L.ptr(dz), L.ptr(d_static), sc.data_ptr(), L.stream_ptr(dev))
            L.check(rc, "rd_encoder_head_bwd_inputs")
        if want_params:
            grads = torch._utils._unflatten_dense_tensors(flat, keep)
            grads = tuple(g if n else None for g, n in zip(grads, need[5:]))
        else:
            grads = (None,) * len(keep)
        ctx.ws = None
        return (None, None, dz if need[2] else None, d_static, None) + grads


def workspace_view(plan, which):
    """Named activation buffer of the most recent forward (parity tests)."""
    lib = L.load()
    n = C.c_int64(0)
    off = lib.rd_workspace_offset(C.byref(plan.last_dims), which, C.byref(n))
    if off < 0:
        L.check(-2, "rd_workspace_offset")
    return plan.last_workspace[off // 4: off // 4 + n.value]

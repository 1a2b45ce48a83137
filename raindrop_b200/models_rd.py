"""Drop-in replacement for the reference's `code/models_rd.py`.

`from models_rd import *` in code/Raindrop.py:19 must find `Raindrop_v2`, `Raindrop`,
`PositionalEncodingTF`, `Observation_progation`, `TransformerConv` with the reference's constructor
signatures, forward signatures and state-dict keys (SURVEY.md section 8b).  Everything numeric is
done by librd_b200.so (hand-written sm_100a CUDA) through `raindrop_b200.functional`; the torch
modules below only hold parameters so that `.cuda()`, `.parameters()`, `state_dict()` and
`load_state_dict()` behave exactly like the reference's.
"""
import math
import weakref

import torch
import torch.nn as nn
from torch.nn.parameter import Parameter

from . import functional as RF

__all__ = ["PositionalEncodingTF", "Raindrop", "Raindrop_v2", "Observation_progation", "TransformerConv"]


def _glorot(t):
    """torch_geometric.nn.inits.glorot (code/models_rd.py:276, code/Ob_propagation.py:85,90-91)."""
    if t is not None:
        a = math.sqrt(6.0 / (t.size(-2) + t.size(-1)))
        t.data.uniform_(-a, a)


def _device_of(*tensors):
    for t in tensors:
        if torch.is_tensor(t) and t.is_cuda:
            return t.device
    if not torch.cuda.is_available():
        raise RF.L.RaindropB200Error("raindrop_b200 needs a CUDA device (no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device())


class PositionalEncodingTF(nn.Module):
    """code/models_rd.py:20-43.  The reference builds the encoding on the host with numpy and
    copies it to the GPU (two syncs per forward); here it is one kernel on the device.  Differentiable with respect
    to P_time, as the reference's torch ops are (RF.PositionalEncodingFunction)."""

    def __init__(self, d_model, max_len=500, MAX=10000):
        super().__init__()
        self.max_len = max_len
        self.d_model = d_model
        self.MAX = MAX
        self._num_timescales = d_model // 2

    def getPE(self, P_time):
        dev = _device_of(P_time)
        return RF.PositionalEncodingFunction.apply(P_time.to(dev), self.max_len, self.d_model)

    def forward(self, P_time):
        return self.getPE(P_time)


class Observation_progation(nn.Module):
    """code/Ob_propagation.py:17-233 (parameter names and shapes kept, :39-70).

    forward(x [n_nodes, C], p_t, edge_index [2,E], edge_weights [E], use_beta=False, ...) ->
    out [n_nodes, C] or (out, (edge_index, alpha)) when return_attention_weights is a bool.
    On the live path the message is relu(lin_value(x_i)) of the TARGET node (:200), the logits are
    the supplied edge weights (:187) and the returned alpha is PRE-softmax (:193)."""

    def __init__(self, in_channels, out_channels, n_nodes, ob_dim, heads=1, concat=True, beta=False,
                 dropout=0., edge_dim=None, bias=True, root_weight=True, **kwargs):
        super().__init__()
        if isinstance(in_channels, int):
            in_channels = (in_channels, in_channels)
        if heads != 1 or edge_dim is not None or beta or not concat or dropout != 0.:
            raise NotImplementedError("only the configuration used by Raindrop_v2 (heads=1, concat, no edge "
                                      "features, no beta gate, dropout 0) is built")
        self.in_channels, self.out_channels, self.heads = in_channels[0], out_channels, heads
        self.n_nodes, self.ob_dim = n_nodes, ob_dim
        self.lin_key = nn.Linear(in_channels[0], heads * out_channels)
        self.lin_query = nn.Linear(in_channels[1], heads * out_channels)
        self.lin_value = nn.Linear(in_channels[0], heads * out_channels)
        self.lin_skip = nn.Linear(in_channels[1], heads * out_channels, bias=bias)
        self.weight = Parameter(torch.Tensor(in_channels[1], heads * out_channels))
        self.bias = Parameter(torch.Tensor(heads * out_channels))
        self.nodewise_weights = Parameter(torch.Tensor(n_nodes, heads * out_channels))
        self.increase_dim = nn.Linear(in_channels[1], heads * out_channels * 8)
        self.map_weights = Parameter(torch.Tensor(n_nodes, heads * 16))
        self.reset_parameters()

    def reset_parameters(self):
        for lin in (self.lin_key, self.lin_query, self.lin_value, self.lin_skip):
            lin.reset_parameters()
        _glorot(self.weight)
        bound = 1 / math.sqrt(self.weight.size(0))
        nn.init.uniform_(self.bias, -bound, bound)
        _glorot(self.nodewise_weights)
        _glorot(self.map_weights)
        self.increase_dim.reset_parameters()

    def forward(self, x, p_t, edge_index, edge_weights=None, use_beta=False, edge_attr=None,
                return_attention_weights=None):
        if edge_weights is None:
            raise ValueError("edge_weights is required (the reference fails without it, code/Ob_propagation.py:195)")
        if isinstance(x, (tuple, list)):
            x = x[1]
        n = x.shape[0]
        if use_beta:
            # dormant in Raindrop_v2 (code/models_rd.py:317) but part of the operator; differentiable (rd_obprop_beta_bwd)
            out, ei, alpha = RF.obprop_beta(x, p_t, edge_index, edge_weights, self.ob_dim, self.increase_dim.weight,
                                            self.increase_dim.bias, self.map_weights, self.lin_value.weight,
                                            self.lin_value.bias)
            if isinstance(return_attention_weights, bool):
                return out, (ei, alpha)
            return out
        s = RF.node_scale(edge_index, edge_weights, n)
        out = RF.ObPropLayerFunction.apply(x, self.lin_value.weight, self.lin_value.bias, s, n)
        if isinstance(return_attention_weights, bool):
            return out, (edge_index, edge_weights.unsqueeze(-1))
        return out

    def __repr__(self):
        return "{}({}, {}, heads={})".format(self.__class__.__name__, self.in_channels, self.out_channels, self.heads)


class TransformerConv(nn.Module):
    """code/transformer_conv.py:13-212 (concat=True, root_weight=True, beta=False, edge_dim=None), forward and
    backward on the device (rd_transformer_conv_fwd / _bwd); `forward_batched` applies the layer to many graphs that
    share one edge list in one call (what legacy `Raindrop` v1 does per sample in a Python loop)."""

    def __init__(self, in_channels, out_channels, heads=1, concat=True, beta=False, dropout=0., edge_dim=None,
                 bias=True, root_weight=True, **kwargs):
        super().__init__()
        if isinstance(in_channels, int):
            in_channels = (in_channels, in_channels)
        if not concat or beta or dropout != 0. or edge_dim is not None or not root_weight or not bias:
            raise NotImplementedError("only concat=True, root_weight=True, beta=False, edge_dim=None is built")
        self.in_channels, self.out_channels, self.heads = in_channels[0], out_channels, heads
        self.lin_key = nn.Linear(in_channels[0], heads * out_channels)
        self.lin_query = nn.Linear(in_channels[1], heads * out_channels)
        self.lin_value = nn.Linear(in_channels[0], heads * out_channels)
        self.lin_skip = nn.Linear(in_channels[1], heads * out_channels, bias=bias)

    def reset_parameters(self):
        for lin in (self.lin_key, self.lin_query, self.lin_value, self.lin_skip):
            lin.reset_parameters()

    def forward(self, x, edge_index, edge_weights=None, edge_attr=None, return_attention_weights=None):
        if isinstance(x, (tuple, list)):
            x = x[1]
        if edge_weights is not None and self.heads != 1:
            raise ValueError("supplied edge_weights need heads == 1 (code/transformer_conv.py:199-206)")
        out, alpha = RF.transformer_conv(x, edge_index, edge_weights, self.heads, self.out_channels,
                                         self.lin_query.weight, self.lin_query.bias, self.lin_key.weight,
                                         self.lin_key.bias, self.lin_value.weight, self.lin_value.bias,
                                         self.lin_skip.weight, self.lin_skip.bias)
        if isinstance(return_attention_weights, bool):
            return out, (edge_index, alpha)
        return out

    def forward_batched(self, x, edge_index, edge_weights=None):
        """x [n_nodes, n_graphs, in]: the layer applied to every graph x[:, g, :] (same edge list) in ONE call -- the
        per-sample loop of legacy Raindrop v1 (code/models_rd.py:158-166).  Returns (out [n_nodes, n_graphs, H*F],
        alpha [n_graphs, E, H])."""
        n_nodes, n_graphs, in_ch = x.shape
        out, alpha = RF.transformer_conv(x.reshape(n_nodes * n_graphs, in_ch), edge_index, edge_weights, self.heads,
                                         self.out_channels, self.lin_query.weight, self.lin_query.bias, self.lin_key.weight,
                                         self.lin_key.bias, self.lin_value.weight, self.lin_value.bias, self.lin_skip.weight,
                                         self.lin_skip.bias, geom=(n_nodes, n_graphs, n_graphs, 1))
        return out.view(n_nodes, n_graphs, -1), alpha

    def __repr__(self):
        return "{}({}, {}, heads={})".format(self.__class__.__name__, self.in_channels, self.out_channels, self.heads)


class Raindrop_v2(nn.Module):
    """code/models_rd.py:194-387.  Same positional constructor (code/Raindrop.py:245-251), same
    64 state-dict keys, `forward(src, static, times, lengths) -> (logits, distance, None)`.

    Differences that are visible to a caller: none on the live path.  Not built (raises):
    `sensor_wise_mask=True` (crashes in the reference as well, SURVEY.md section 7)."""

    def __init__(self, d_inp=36, d_model=64, nhead=4, nhid=128, nlayers=2, dropout=0.3, max_len=215, d_static=9,
                 MAX=100, perc=0.5, aggreg='mean', n_classes=2, global_structure=None, sensor_wise_mask=False,
                 static=True):
        super().__init__()
        from torch.nn import TransformerEncoder, TransformerEncoderLayer
        if sensor_wise_mask:
            raise NotImplementedError("sensor_wise_mask=True raises a shape error in the reference itself")
        if aggreg != 'mean':
            raise NotImplementedError("aggreg must be 'mean' (the only branch of code/models_rd.py:378)")
        self.model_type = 'Transformer'
        self.global_structure = global_structure
        self.sensor_wise_mask = sensor_wise_mask
        d_pe = 16
        self.d_inp, self.d_model, self.static = d_inp, d_model, static
        self.max_len, self.n_classes, self.nhead, self.nhid, self.nlayers = max_len, n_classes, nhead, nhid, nlayers
        if static:
            self.emb = nn.Linear(d_static, d_inp)
        self.d_ob = int(d_model / d_inp)
        self.encoder = nn.Linear(d_inp * self.d_ob, d_inp * self.d_ob)          # unused on the path (8a19)
        self.pos_encoder = PositionalEncodingTF(d_pe, max_len, MAX)
        # parameter container only: its forward is never called, the kernels read its tensors
        self.transformer_encoder = TransformerEncoder(TransformerEncoderLayer(d_model + d_pe, nhead, nhid, dropout),
                                                      nlayers, enable_nested_tensor=False)
        self.adj = torch.ones([d_inp, d_inp])
        self.R_u = torch.Tensor(1, d_inp * self.d_ob)   # plain tensor: never trained, not in the state dict (:241)
        C = max_len * self.d_ob
        self.ob_propagation = Observation_progation(in_channels=C, out_channels=C, heads=1, n_nodes=d_inp,
                                                    ob_dim=self.d_ob)
        self.ob_propagation_layer2 = Observation_progation(in_channels=C, out_channels=C, heads=1, n_nodes=d_inp,
                                                           ob_dim=self.d_ob)
        d_final = d_model + d_pe + (d_inp if static else 0)
        self.mlp_static = nn.Sequential(nn.Linear(d_final, d_final), nn.ReLU(), nn.Linear(d_final, n_classes))
        self.mlp = nn.Sequential(nn.Linear(d_model, d_model), nn.ReLU(), nn.Linear(d_model, n_classes))
        self.aggreg = aggreg
        self.relu = nn.ReLU()
        self.dropout = nn.Dropout(dropout)
        self.init_weights()

        self._plan = RF.Plan(d_inp, self.d_ob, nhead, nhid, nlayers, d_static, n_classes, max_len, dropout, static)
        self._plan.owner = weakref.ref(self)
        self._graph_key = None
        self._flat_grad = None
        self._flat_optim = None           # weakref to a bound raindrop_b200.optim.FlatAdam
        self._seed = int(torch.initial_seed()) & 0x7FFFFFFFFFFFFFFF

    def init_weights(self):
        initrange = 1e-10
        self.encoder.weight.data.uniform_(-initrange, initrange)
        if self.static:
            self.emb.weight.data.uniform_(-initrange, initrange)
        _glorot(self.R_u)

    def _apply(self, fn, recurse=True):
        super()._apply(fn, recurse)
        self.R_u = fn(self.R_u)       # moves with the module; the reference creates it on the GPU (:241)
        self.adj = fn(self.adj)
        self.__dict__.pop("_used_params", None)
        return self

    def load_state_dict(self, *args, **kwargs):
        out = super().load_state_dict(*args, **kwargs)
        self.__dict__.pop("_used_params", None)      # `assign=True` may have replaced Parameter objects
        return out

    # ---- host-side graph prologue, cached (code/models_rd.py:307-311) ---------------------------
    def _prepare(self, device):
        plan = self._plan
        gs = self.global_structure
        if gs is None:
            gs = self.adj
        key = (id(gs), gs._version, str(device))
        if key != self._graph_key:
            adj = gs.detach().to(device=device, dtype=torch.float32).clone()
            n = self.d_inp
            adj[torch.arange(n, device=device), torch.arange(n, device=device)] = 1
            edge_index = torch.nonzero(adj).T.contiguous()
            edge_weights = adj[edge_index[0], edge_index[1]].contiguous()
            plan.node_scale = RF.node_scale(edge_index, edge_weights, n)
            self._edge_index, self._edge_weights = edge_index, edge_weights
            self._graph_key = key
        if self.R_u.device != device or self.R_u.dtype != torch.float32:
            self.R_u = self.R_u.to(device=device, dtype=torch.float32)
        plan.R_u = self.R_u.contiguous()
        if plan.rng_state is None or plan.rng_state.device != device:
            plan.rng_state = torch.tensor([self._seed, 0], dtype=torch.int64, device=device)
        return plan

    def used_parameters(self):
        """The tensors that receive gradient, in flat-bucket order (SURVEY.md section 8a18)."""
        cached = self.__dict__.get("_used_params")
        if cached is None:
            sd = dict(self.named_parameters())
            cached = [sd[k] for k, _ in self._plan.fields]
            self.__dict__["_used_params"] = cached      # plain attribute: not a registered sub-module/parameter
        return cached

    def forward(self, src, static, times, lengths):
        """src [T, B, 2*d_inp]; static [B, d_static] or None; times [T, B]; lengths [B] (int64).
        Returns (logits [B, n_classes], distance (0-d), None)."""
        device = _device_of(src)
        plan = self._prepare(device)
        if self.static and static is None:
            raise ValueError("this model was built with static=True: `static` must be a tensor")
        src = src.to(device=device, dtype=torch.float32).contiguous()
        times = times.to(device=device, dtype=torch.float32).contiguous()
        lengths = lengths.to(device=device, dtype=torch.int64).contiguous()
        st = static.to(device=device, dtype=torch.float32).contiguous() if (self.static and static is not None) else None
        logits = None
        flat = self._flat_optim() if self._flat_optim is not None else None
        if flat is not None and flat.flat_p.device == device:
            # parameters live in one flat leaf (raindrop_b200.optim.FlatAdam): graph-captured fast path
            logits = RF.flat_forward(plan, self.training, flat, src, st, times, lengths)
        if logits is None:
            logits = RF.RaindropV2Function.apply(plan, self.training, src, st, times, lengths, *self.used_parameters())
        # alpha_all has identical columns on the live path, so mean(cdist) == 0 (code/models_rd.py:343-346)
        distance = torch.zeros((), dtype=torch.float32, device=device)
        return logits, distance, None


class Raindrop(nn.Module):
    """Legacy v1 model (code/models_rd.py:46-191), hard-coded to 36 sensors like the reference.  Same constructor, same
    state-dict keys, `forward(src, static, times, lengths) -> (logits, distance, None)`.

    What the reference computes, and where it runs here:
      src = encoder(values) * sqrt(d_model); dropout                      (:131-135)  rd_linear_fwd, rd_dropout
      per sample: TransformerConv over the T timestamps as nodes with the 36 x 36 sensor graph's edges (so only the
      first 36 timestamps exchange messages) and the supplied edge weights (:148-166)
                                                                          rd_transformer_conv_fwd/_bwd, all samples in one call
      cat positional encoding (d_pe = 36), nn.TransformerEncoder, masked mean / (lengths + 1), cat emb(static),
      mlp_static (:168-189)                                               rd_encoder_head_fwd/_bwd (the Raindrop_v2 kernels)
    `distance` = mean pairwise distance of the per-sample attention vectors (:165-166): the edge weights are shared by
    all samples, so it is 0 -- evaluated from the returned alphas, not assumed.
    Autograd reaches src, static, times and a global_structure that requires grad, as in the reference (:131-166)."""

    def __init__(self, d_inp=36, d_model=64, nhead=4, nhid=128, nlayers=2, dropout=0.3, max_len=215, d_static=9,
                 MAX=100, perc=0.5, aggreg='mean', n_classes=2, global_structure=None):
        super().__init__()
        from torch.nn import TransformerEncoder, TransformerEncoderLayer
        if aggreg != 'mean':
            raise NotImplementedError("aggreg must be 'mean' (the only branch of code/models_rd.py:182)")
        self.model_type = 'Transformer'
        self.global_structure = global_structure
        d_pe, d_enc = 36, 36
        self.pos_encoder = PositionalEncodingTF(d_pe, max_len, MAX)
        self.transformer_encoder = TransformerEncoder(TransformerEncoderLayer(d_model + 36, nhead, nhid, dropout),
                                                      nlayers, enable_nested_tensor=False)
        self.gcs = nn.ModuleList()
        self.dim = int(d_model / d_inp)
        self.transconv = TransformerConv(in_channels=36, out_channels=36 * self.dim, heads=1)
        d_final = 36 * (self.dim + 1) + d_model
        self.mlp_static = nn.Sequential(nn.Linear(d_final, d_final), nn.ReLU(), nn.Linear(d_final, n_classes))
        self.d_inp, self.d_model, self.max_len, self.n_classes = d_inp, d_model, max_len, n_classes
        self.encoder = nn.Linear(d_inp, d_enc)
        self.emb = nn.Linear(d_static, d_model)
        self.MLP_replace_transformer = nn.Linear(72, 36)
        self.mlp = nn.Sequential(nn.Linear(d_model, d_model), nn.ReLU(), nn.Linear(d_model, n_classes))
        self.aggreg = aggreg
        self.relu = nn.ReLU()
        self.dropout = nn.Dropout(dropout)
        self.encoder.weight.data.uniform_(-1e-10, 1e-10)
        self.emb.weight.data.uniform_(-1e-10, 1e-10)
        if d_inp != 36 or 36 * self.dim != d_model:
            raise ValueError("Raindrop v1 is hard-coded to 36 sensors and d_model = 36 * k (code/models_rd.py:68-88)")
        # the shared encoder/head kernels see "36 sensors x dim channels" + a 36-wide positional encoding
        self._plan = RF.Plan(36, self.dim, nhead, nhid, nlayers, d_static, n_classes, max_len, dropout, True, d_pe=36,
                             emb_dim=d_model, obprop=False)
        self._seed = int(torch.initial_seed()) & 0x7FFFFFFFFFFFFFFF
        self._drop_p = float(dropout)

    def used_parameters(self):
        sd = dict(self.named_parameters())
        return [sd[k] for k, _ in self._plan.fields]

    def forward(self, src, static, times, lengths):
        device = _device_of(src)
        plan = self._plan
        if plan.rng_state is None or plan.rng_state.device != device:
            plan.rng_state = torch.tensor([self._seed, 0], dtype=torch.int64, device=device)
        src = src.to(device=device, dtype=torch.float32)
        times = times.to(device=device, dtype=torch.float32).contiguous()
        lengths = lengths.to(device=device, dtype=torch.int64).contiguous()
        static = static.to(device=device, dtype=torch.float32).contiguous()
        T, B = src.shape[0], src.shape[1]
        if T != self.max_len or src.shape[2] != 2 * self.d_inp:
            raise ValueError("src must be [max_len=%d, B, 72], got %s" % (self.max_len, tuple(src.shape)))
        values = src[:, :, :self.d_inp].reshape(T * B, self.d_inp)                                  # :128-129
        x = RF.LinearFunction.apply(values, self.encoder.weight, self.encoder.bias) * math.sqrt(self.d_model)   # :131
        if self.training and self._drop_p > 0:                                                        # :134
            x = RF.DropoutFunction.apply(x, self._drop_p, plan.rng_state.clone(), 2)
        gs = self.global_structure
        if gs is None:
            raise ValueError("Raindrop v1 needs global_structure (code/models_rd.py:148)")
        # the edge weights stay differentiable w.r.t. global_structure; the diagonal is forced to 1 out of place, so it
        # gets zero gradient as under the reference's in-place write (:149); edge_index is data
        eye = torch.eye(36, dtype=torch.bool, device=device)
        adj = torch.where(eye, 1.0, gs.to(device=device, dtype=torch.float32))                        # :149
        edge_index = torch.nonzero(adj.detach()).T.contiguous()
        edge_weights = adj[edge_index[0], edge_index[1]].contiguous()
        out, alpha = self.transconv.forward_batched(x.view(T, B, self.d_inp), edge_index, edge_weights)   # :155-166
        alpha_all = alpha[:, :, 0]                                                                    # [B, E]
        distance = torch.mean(torch.cdist(alpha_all, alpha_all, p=2, compute_mode='donot_use_mm_for_euclid_dist'))   # :165-166
        pe = self.pos_encoder(times)                                                                   # [T, B, 36]
        z0 = torch.cat([out, pe], dim=-1)                                                              # :168
        logits = RF.EncoderHeadFunction.apply(plan, self.training, z0, static, lengths, *self.used_parameters())
        return logits, distance, None

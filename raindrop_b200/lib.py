"""ctypes binding of librd_b200.so (the C ABI declared in include/raindrop_b200.h).

The library is built in-tree by `raindrop_b200/csrc/build.sh` (see __graft_entry__.build) and is
the ONLY compute path: if it is missing or a call fails, we raise -- there is no CPU fallback.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "librd_b200.so")

RD_MAX_LAYERS = 8
ABI_VERSION = 2
BWD_ENCODER, BWD_OBPROP, BWD_ALL = 1, 2, 3
RD_D_PE = 16

# enum rd_ws_buffer
WS_X0, WS_H1, WS_ENC_IN, WS_ENC_OUT, WS_FEAT, WS_RNG = range(6)

# dropout site ids (rd_common.cuh: DropSite)
SITE_LIFT, SITE_ATTN, SITE_RESID1, SITE_FFN, SITE_RESID2 = 1, 16, 32, 48, 64

c_float_p = C.c_void_p  # device pointers travel as integers


class RdDims(C.Structure):
    _fields_ = [("B", C.c_int32), ("T", C.c_int32), ("N", C.c_int32), ("d_ob", C.c_int32),
                ("nhead", C.c_int32), ("nhid", C.c_int32), ("nlayers", C.c_int32),
                ("d_static", C.c_int32), ("n_classes", C.c_int32), ("training", C.c_int32),
                ("dropout_p", C.c_float), ("ln_eps", C.c_float),
                ("pe_timescales", C.c_float * (RD_D_PE // 2)), ("d_pe", C.c_int32), ("emb_dim", C.c_int32),
                ("obprop_mode", C.c_int32)]


_LAYER_FIELDS = ["in_proj_weight", "in_proj_bias", "out_proj_weight", "out_proj_bias",
                 "linear1_weight", "linear1_bias", "linear2_weight", "linear2_bias",
                 "norm1_weight", "norm1_bias", "norm2_weight", "norm2_bias"]


class RdLayer(C.Structure):
    _fields_ = [(f, C.c_void_p) for f in _LAYER_FIELDS]


class RdParams(C.Structure):
    _fields_ = [("R_u", C.c_void_p), ("emb_weight", C.c_void_p), ("emb_bias", C.c_void_p),
                ("ob1_value_weight", C.c_void_p), ("ob1_value_bias", C.c_void_p),
                ("ob2_value_weight", C.c_void_p), ("ob2_value_bias", C.c_void_p),
                ("mlp0_weight", C.c_void_p), ("mlp0_bias", C.c_void_p),
                ("mlp2_weight", C.c_void_p), ("mlp2_bias", C.c_void_p),
                ("layer", RdLayer * RD_MAX_LAYERS)]


class RdGrads(C.Structure):
    _fields_ = [("emb_weight", C.c_void_p), ("emb_bias", C.c_void_p),
                ("ob1_value_weight", C.c_void_p), ("ob1_value_bias", C.c_void_p),
                ("ob2_value_weight", C.c_void_p), ("ob2_value_bias", C.c_void_p),
                ("mlp0_weight", C.c_void_p), ("mlp0_bias", C.c_void_p),
                ("mlp2_weight", C.c_void_p), ("mlp2_bias", C.c_void_p),
                ("layer", RdLayer * RD_MAX_LAYERS)]


class RdInputGrads(C.Structure):
    _fields_ = [("src", C.c_void_p), ("statics", C.c_void_p), ("times", C.c_void_p)]


class RdWgradItem(C.Structure):
    _fields_ = [("d_out", C.c_void_p), ("x", C.c_void_p), ("rows", C.c_int64), ("out_features", C.c_int32),
                ("in_features", C.c_int32), ("d_weight", C.c_void_p), ("d_bias", C.c_void_p), ("partial", C.c_void_p)]


# name -> (restype, argtypes); every symbol include/raindrop_b200.h declares
SIGNATURES = {
    "rd_abi_version": (C.c_int, []),
    "rd_last_error_string": (C.c_char_p, []),
    "rd_launch_count": (C.c_uint64, []),
    "rd_node_scale": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "rd_obprop_fwd_scratch_bytes": (C.c_size_t, [C.c_int64, C.c_int32]),
    "rd_obprop_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int64,
                                C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rd_obprop_bwd_scratch_bytes": (C.c_size_t, [C.c_int64, C.c_int32]),
    "rd_obprop_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p]),
    "rd_obprop_beta_scratch_bytes": (C.c_size_t, [C.c_int32] * 4),
    "rd_obprop_beta_fwd": (C.c_int, [C.c_void_p] * 5 + [C.c_int32] * 4 + [C.c_void_p] * 11),
    "rd_obprop_beta_bwd_scratch_bytes": (C.c_size_t, [C.c_int32] * 4),
    "rd_obprop_beta_bwd": (C.c_int, [C.c_void_p] * 5 + [C.c_int32] * 4 + [C.c_void_p] * 5 + [C.c_void_p] * 2 + [C.c_void_p] * 8 +
                           [C.c_void_p, C.c_void_p]),
    "rd_workspace_bytes": (C.c_size_t, [C.POINTER(RdDims)]),
    "rd_backward_scratch_bytes": (C.c_size_t, [C.POINTER(RdDims)]),
    "rd_workspace_offset": (C.c_int64, [C.POINTER(RdDims), C.c_int32, C.POINTER(C.c_int64)]),
    "rd_raindrop_v2_fwd": (C.c_int, [C.POINTER(RdDims), C.POINTER(RdParams), C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rd_raindrop_v2_bwd": (C.c_int, [C.POINTER(RdDims), C.POINTER(RdParams), C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(RdGrads), C.c_void_p,
                                     C.c_int32, C.c_void_p]),
    "rd_input_grad_scratch_bytes": (C.c_size_t, [C.POINTER(RdDims)]),
    "rd_raindrop_v2_bwd_inputs": (C.c_int, [C.POINTER(RdDims), C.POINTER(RdParams), C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.POINTER(RdGrads), C.POINTER(RdInputGrads),
                                            C.c_void_p, C.c_void_p, C.c_void_p]),
    "rd_positional_encoding": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(C.c_float), C.c_int32, C.c_void_p,
                                         C.c_int64, C.c_int32, C.c_void_p]),
    "rd_positional_encoding_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_float), C.c_int32, C.c_int64,
                                             C.c_int32, C.c_void_p, C.c_void_p]),
    "rd_encoder_head_fwd": (C.c_int, [C.POINTER(RdDims), C.POINTER(RdParams)] + [C.c_void_p] * 9),
    "rd_encoder_head_bwd": (C.c_int, [C.POINTER(RdDims), C.POINTER(RdParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.POINTER(RdGrads), C.c_void_p, C.c_void_p, C.c_void_p]),
    "rd_encoder_head_bwd_inputs": (C.c_int, [C.POINTER(RdDims), C.POINTER(RdParams), C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.POINTER(RdGrads), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rd_dropout": (C.c_int, [C.c_void_p, C.c_int64, C.c_float, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "rd_linear_scratch_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "rd_linear_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                C.c_void_p, C.c_void_p, C.c_void_p]),
    "rd_temporal_attention_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float,
                                            C.c_void_p, C.c_uint32, C.c_int32, C.c_void_p, C.c_void_p]),
    "rd_temporal_attention_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                            C.c_float, C.c_void_p, C.c_uint32, C.c_int32, C.c_void_p, C.c_void_p]),
    "rd_linear_wgrad_partial_bytes": (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32]),
    "rd_linear_wgrad_group": (C.c_int, [C.POINTER(RdWgradItem), C.c_int32, C.c_void_p]),
    "rd_transformer_conv_scratch_bytes": (C.c_size_t, [C.c_int32] * 7),
    "rd_transformer_conv_fwd": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32] + [C.c_void_p] * 8 +
                                [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rd_transformer_conv_bwd": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32] + [C.c_void_p] * 7 +
                                [C.c_void_p] * 2 + [C.c_void_p] * 10 + [C.c_void_p, C.c_void_p]),
    "rd_gather_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_void_p,
                                  C.c_void_p]),
    "rd_assemble_batch": (C.c_int, [C.c_void_p] * 5 + [C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int32] + [C.c_void_p] * 6),
    "rd_feature_stats_scratch_bytes": (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32]),
    "rd_feature_stats": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rd_mask_normalize": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p]),
    "rd_zero_features": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "rd_cross_entropy_fwd_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p,
                                           C.c_void_p, C.c_void_p]),
    "rd_adam_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_void_p,
                               C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_void_p]),
    "rd_debug_attention_timing": (C.c_int, [C.c_void_p]),
    "rd_debug_gemm_timing": (C.c_int, [C.c_void_p]),
    "rd_debug_dropout_mask": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int64, C.c_float, C.c_void_p,
                                        C.c_void_p]),
}

_lib = None


class RaindropB200Error(RuntimeError):
    pass


def load():
    """Loads librd_b200.so (once).  Raises if it has not been built: there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RaindropB200Error(
            "%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(raindrop_b200/csrc/build.sh).  raindrop_b200 has no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    if lib.rd_abi_version() != ABI_VERSION:
        raise RaindropB200Error("ABI version mismatch: %d" % lib.rd_abi_version())
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().rd_last_error_string()
        raise RaindropB200Error("%s failed (rc=%d): %s" % (what, rc, msg.decode() if msg else "?"))


def ptr(t):
    """Device pointer of a tensor (0 for None)."""
    return 0 if t is None else t.data_ptr()


def stream_ptr(device=None):
    """cudaStream_t of torch's current stream on `device` (default: the current device)."""
    import torch
    return torch.cuda.current_stream(device).cuda_stream

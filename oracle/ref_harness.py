"""TEST INFRASTRUCTURE ONLY -- never imported by the product path (raindrop_b200/).

Loads the reference's OWN, UNMODIFIED files (`code/{models_rd,Ob_propagation,transformer_conv}.py`
of a checkout of the original Raindrop project, located by the environment variable
RAINDROP_REFERENCE) on CPU, to generate the committed golden fixtures under `tests/golden/`
(script: `oracle/make_golden.py`) that pin the oracle restatement in `oracle/raindrop_oracle.py`
and the CUDA path.  The tests read only those fixtures, never the reference itself.

Why patches are needed (SURVEY.md section 8c):
  * torch_geometric / torch_scatter / torch_sparse are not installed -> `oracle/pyg_shim`.
  * `os.add_dll_directory` (models_rd.py:8-9) does not exist on Linux -> no-op.
  * `.cuda()` is hard-coded (models_rd.py:42,143,239,241,299,307,315,321) -> identity on
    CPU; for an `nn.Parameter` it returns a non-Parameter view, reproducing the fact that
    `self.R_u = Parameter(...).cuda()` (models_rd.py:241) is NOT a registered parameter.
  * `adj[torch.eye(n).byte()] = 1` (models_rd.py:308): uint8 masks are rejected by
    torch 2.11 -> `Tensor.byte` returns bool (harness-local).
"""
import importlib
import os
import sys

import torch
import torch.nn as nn

REFERENCE_CODE = os.path.join(os.path.abspath(os.environ.get("RAINDROP_REFERENCE") or os.devnull), "code")
_SHIM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "pyg_shim")
_loaded = None


def reference_available():
    return os.path.isfile(os.path.join(REFERENCE_CODE, "models_rd.py"))


def load_reference():
    """Returns the reference's `models_rd` module, imported from where it lies."""
    global _loaded
    if _loaded is not None:
        return _loaded
    if not reference_available():
        raise RuntimeError("reference tree not found: set RAINDROP_REFERENCE to a checkout of the original project")
    if torch.cuda.is_available():
        raise RuntimeError("the reference harness is CPU-only (it patches Tensor.cuda)")

    if not hasattr(os, "add_dll_directory"):
        os.add_dll_directory = lambda p: None

    def _tensor_cuda(self, *a, **k):
        if isinstance(self, nn.Parameter):
            return self.view_as(self)  # non-leaf, non-Parameter: like a device copy
        return self

    torch.Tensor.cuda = _tensor_cuda
    nn.Module.cuda = lambda self, *a, **k: self
    torch.Tensor.byte = lambda self, *a, **k: self.bool()

    for p in (_SHIM, REFERENCE_CODE):
        if p not in sys.path:
            sys.path.insert(0, p)
    # our own drop-in is also called `models_rd`; make sure the reference's one is loaded
    for name in ("models_rd", "Ob_propagation", "transformer_conv"):
        mod = sys.modules.get(name)
        if mod is not None and not getattr(mod, "__file__", "").startswith(REFERENCE_CODE):
            del sys.modules[name]
    mod = importlib.import_module("models_rd")
    assert mod.__file__.startswith(REFERENCE_CODE), mod.__file__
    _loaded = mod
    return mod


def build_reference_model(cfg, seed=1):
    """Constructs Raindrop_v2 exactly as code/Raindrop.py:245-251 does (positional args)."""
    ref = load_reference()
    torch.manual_seed(seed)
    gs = torch.ones(cfg["d_inp"], cfg["d_inp"]) if cfg.get("global_structure") is None \
        else cfg["global_structure"].clone()
    d_model = cfg["d_inp"] * cfg["d_ob"]
    kw = {}
    if not cfg.get("static", True):
        kw["static"] = False
    model = ref.Raindrop_v2(cfg["d_inp"], d_model, cfg["nhead"], cfg["nhid"], cfg["nlayers"],
                            cfg["dropout"], cfg["max_len"], cfg["d_static"], cfg.get("MAX", 100),
                            0.5, "mean", cfg["n_classes"], gs, sensor_wise_mask=False, **kw)
    return model

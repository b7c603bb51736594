"""Import the UNMODIFIED reference from /root/reference (build container only; TEST INFRASTRUCTURE).

The reference needs `timm` and `pyiqa`, neither installed here (network_swinir.py:11,
losses/losses.py:11, models/femasr_model.py:15).  timm contributes no inference arithmetic
(DropPath is nn.Identity at drop_path=0, network_swinir.py:204), so two stub modules are enough.
Used only by tests/golden/make_golden.py: the tests compare with what it stored under tests/golden/.
"""
from __future__ import annotations

import importlib
import os
import sys
import types

REFERENCE_ROOT = "/root/reference"


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "basicsr"))


def import_reference():
    """Returns the reference's ``basicsr.archs.femasr_arch`` module (fresh import, our own
    ``basicsr`` boundary package is temporarily shadowed and restored afterwards)."""
    import torch
    from torch import nn

    if not reference_available():
        raise RuntimeError("reference tree not present")
    sys.dont_write_bytecode = True
    saved = {k: v for k, v in sys.modules.items() if k == "basicsr" or k.startswith("basicsr.")}
    for k in saved:
        del sys.modules[k]

    class DropPath(nn.Module):
        def __init__(self, p=0.0):
            super().__init__()

        def forward(self, x):
            return x

    def to_2tuple(x):
        return tuple(x) if isinstance(x, (tuple, list)) else (x, x)

    layers = types.ModuleType("timm.models.layers")
    layers.DropPath, layers.to_2tuple, layers.trunc_normal_ = DropPath, to_2tuple, torch.nn.init.trunc_normal_
    timm, models = types.ModuleType("timm"), types.ModuleType("timm.models")
    timm.models, models.layers = models, layers
    stubs = {"timm": timm, "timm.models": models, "timm.models.layers": layers,
             "pyiqa": types.ModuleType("pyiqa")}
    had = {k: sys.modules.get(k) for k in stubs}
    sys.modules.update(stubs)
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        mod = importlib.import_module("basicsr.archs.femasr_arch")
        ref_modules = {k: v for k, v in sys.modules.items() if k == "basicsr" or k.startswith("basicsr.")}
    finally:
        sys.path.remove(REFERENCE_ROOT)
        for k in [k for k in sys.modules if k == "basicsr" or k.startswith("basicsr.")]:
            del sys.modules[k]
        sys.modules.update(saved)
        for k, v in had.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    mod._ref_modules = ref_modules      # keep the reference package alive for its own lazy lookups
    return mod

"""CPU: the parameter inventory (femasr_b200/spec.py), the drop-in module (basicsr/archs/femasr_arch.py) and the C
engine's own spec agree with the REFERENCE's state_dict() - names, shapes, dtypes - for every supported configuration.
The reference's inventories are stored in tests/golden/reference_boundary.json.gz (written by tests/golden/make_golden.py
from the unmodified reference)."""
import ctypes
import gzip
import json
import os

import pytest
import torch

from femasr_b200.spec import param_spec, random_state_dict

CONFIGS = [
    (4, [[32, 1024, 256]]), (4, [[32, 1024, 512]]), (2, [[32, 1024, 256]]), (1, [[32, 1024, 512]]),
    (4, [[32, 1024, 256], [64, 512, 128]]), (2, [[32, 512, 256], [64, 512, 256], [128, 256, 128]]),
    (1, [[32, 1024, 256], [128, 256, 64]]),
]
IDS = [f"x{s}_{len(c)}cb_e{c[0][2]}" for s, c in CONFIGS]
REFERENCE_BOUNDARY = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_boundary.json.gz")


def reference_state_dict_inventory(cid):
    """{name: (shape, dtype)} of the reference's FeMaSRNet(...).state_dict() for configuration `cid`."""
    with gzip.open(REFERENCE_BOUNDARY, "rt") as f:
        entries = json.load(f)["state_dict"][cid]
    return {k: (tuple(shape), getattr(torch, dtype)) for k, shape, dtype in entries}


@pytest.mark.parametrize("scale,cbs", CONFIGS, ids=IDS)
def test_spec_matches_reference_state_dict(scale, cbs):
    want = reference_state_dict_inventory(IDS[CONFIGS.index((scale, cbs))])
    spec = {n: s for n, s, _k, _f in param_spec(scale, cbs[0][2], cbs[0][1], codebooks=cbs)}
    assert set(spec) == set(want), (sorted(set(spec) - set(want))[:5], sorted(set(want) - set(spec))[:5])
    for n, s in spec.items():
        assert tuple(s) == want[n][0], n
    # a state_dict made here has the reference's keys and shapes (what its strict load checks), and one with the
    # reference's keys, shapes and dtypes loads strictly into ours
    sd = random_state_dict(scale, cbs[0][2], seed=3, codebooks=cbs)
    assert {k: tuple(v.shape) for k, v in sd.items()} == {k: s for k, (s, _d) in want.items()}
    from basicsr.archs.femasr_arch import FeMaSRNet
    mine = FeMaSRNet(codebook_params=cbs, LQ_stage=scale != 1, scale_factor=scale)
    res = mine.load_state_dict({k: torch.zeros(s, dtype=d) for k, (s, d) in want.items()}, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    for k, v in mine.state_dict().items():
        assert v.dtype == want[k][1], k


@pytest.mark.parametrize("scale,cbs", CONFIGS, ids=IDS)
def test_engine_spec_matches_python_spec(built_lib, scale, cbs):
    """The C engine accepts exactly the float tensors of the Python inventory (right sizes), rejects unknown names and
    wrong sizes, and reports completeness only when all are set.  Host buffers, no kernel launches."""
    from femasr_b200 import lib
    L = lib.load()
    I3 = ctypes.c_int * 3
    K = len(cbs)
    pad = lambda col: I3(*([c[col] for c in cbs] + [0] * (3 - K)))
    cfg = lib.NetConfig(scale, cbs[0][1], cbs[0][2], 3, 1, 1, 0, K, pad(0), pad(1), pad(2))
    h = ctypes.c_void_p()
    assert L.femasr_net_create(ctypes.byref(cfg), ctypes.byref(h)) == 0
    try:
        floats = [(n, s) for n, s, k, _f in param_spec(scale, cbs[0][2], cbs[0][1], codebooks=cbs) if k not in ("rpi", "mask")]
        if not torch.cuda.is_available():
            # without a device set_param cannot upload; the spec is still checked through the error codes for bad input
            buf = torch.zeros(4)
            assert L.femasr_net_set_param(h, b"no.such.parameter", buf.data_ptr(), 4, 0, None) == -1
            n0, s0 = floats[0]
            assert L.femasr_net_set_param(h, n0.encode(), buf.data_ptr(), 3, 0, None) == -1      # wrong size
            assert L.femasr_net_params_complete(h) == -3
            # every name of the inventory is known to the engine: a wrong-size upload is rejected for its SIZE
            for n, s in floats:
                numel = 1
                for d in s:
                    numel *= d
                assert L.femasr_net_set_param(h, n.encode(), buf.data_ptr(), numel + 1, 0, None) == -1
                assert b"wrong size" in L.femasr_last_error(), (n, L.femasr_last_error())
    finally:
        L.femasr_net_destroy(h)

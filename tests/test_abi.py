"""CPU: the C-ABI library builds, loads and exports every symbol include/femasr_b200.h declares;
without a GPU the product path fails loudly instead of falling back."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "femasr_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(femasr_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(built_lib):
    from femasr_b200 import lib
    names = header_symbols()
    assert len(names) >= 30
    dll = ctypes.CDLL(built_lib)
    for n in names:
        assert hasattr(dll, n), f"{n} declared in the header but not exported"
    assert sorted(lib.SIGNATURES) == names, "femasr_b200/lib.py SIGNATURES out of sync with the header"
    assert lib.load().femasr_abi_version() == lib.ABI_VERSION == 5


def test_argument_validation_without_gpu(built_lib):
    from femasr_b200 import lib
    L = lib.load()
    a = lib.IgemmArgs()
    assert L.femasr_igemm_simt(ctypes.byref(a), None) == -1
    assert b"null" in L.femasr_last_error()
    h = ctypes.c_void_p()
    cfg = lib.NetConfig(3, 1024, 256, 3, 1, 1, 0)
    assert L.femasr_net_create(ctypes.byref(cfg), ctypes.byref(h)) == -1
    cfg = lib.NetConfig(1, 1024, 256, 3, 1, 1, 1)                 # HQ autoencoder stage
    assert L.femasr_net_create(ctypes.byref(cfg), ctypes.byref(h)) == 0
    need = ctypes.c_size_t()
    assert L.femasr_net_workspace_bytes(h, 2, 64, 96, ctypes.byref(need)) == 0 and need.value > 0
    assert L.femasr_net_workspace_bytes(h, 2, 60, 96, ctypes.byref(need)) == -1
    L.femasr_net_destroy(h)
    cfg = lib.NetConfig(4, 1024, 256, 3, 1, 1, 0)
    assert L.femasr_net_create(ctypes.byref(cfg), ctypes.byref(h)) == 0
    need = ctypes.c_size_t()
    # 40x40: Swin stage 20x20 is not a multiple of the 8x8 window -> the reference raises in window_partition
    assert L.femasr_net_workspace_bytes(h, 1, 40, 40, ctypes.byref(need)) == -1
    assert L.femasr_net_workspace_bytes(h, 32, 128, 128, ctypes.byref(need)) == 0
    assert 1 << 30 < need.value < 40 << 30
    assert abs(L.femasr_net_flops(h, 1, 128, 128) / 1e9 - 754.53) < 0.01
    assert L.femasr_net_params_complete(h) == -3
    L.femasr_net_destroy(h)
    # multi-scale codebooks: geometry, workspace and the FLOP model follow the extra quantisers
    I3 = ctypes.c_int * 3
    cfg = lib.NetConfig(4, 0, 0, 3, 1, 1, 0, 2, I3(32, 64, 0), I3(1024, 512, 0), I3(256, 128, 0))
    assert L.femasr_net_create(ctypes.byref(cfg), ctypes.byref(h)) == 0
    assert L.femasr_net_workspace_bytes(h, 1, 32, 32, ctypes.byref(need)) == 0 and need.value > 0
    extra = 2.0 * 512 * 128 + 2.0 * 512 * 128 + 2.0 * 9 * (128 + 256) * 256       # before_quant, z.E^T, after_quant at 128x128
    assert abs(L.femasr_net_flops(h, 1, 128, 128) - (754.53e9 + extra * 128 * 128)) < 2e7
    L.femasr_net_destroy(h)
    cfg = lib.NetConfig(4, 0, 0, 3, 1, 1, 0, 2, I3(32, 32, 0), I3(1024, 512, 0), I3(256, 128, 0))
    assert L.femasr_net_create(ctypes.byref(cfg), ctypes.byref(h)) == -1            # scales must increase


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback(built_lib):
    from basicsr.archs.femasr_arch import FeMaSRNet
    from femasr_b200.lib import FemasrError
    net = FeMaSRNet(codebook_params=[[32, 1024, 256]], LQ_stage=True, scale_factor=4).eval()
    with pytest.raises(FemasrError):
        net.test(torch.rand(1, 3, 32, 32))
    with pytest.raises(FemasrError):
        net(torch.rand(1, 3, 32, 32))


def test_unsupported_configs_raise():
    from basicsr.archs.femasr_arch import FeMaSRNet
    with pytest.raises(NotImplementedError):
        FeMaSRNet(codebook_params=[[32, 1024, 256]], LQ_stage=True, norm_type="bn")
    with pytest.raises(NotImplementedError):
        FeMaSRNet(codebook_params=[[16, 1024, 256]], LQ_stage=True)               # first codebook must sit at 32
    with pytest.raises(NotImplementedError):
        FeMaSRNet(codebook_params=[[32, 1024, 256], [256, 512, 64]], LQ_stage=True)    # no decoder level at 256
    with pytest.raises(NotImplementedError):
        FeMaSRNet(codebook_params=[[32, 1000, 256]], LQ_stage=True)                # n_e / e_dim: multiples of 64
    ms = FeMaSRNet(codebook_params=[[32, 1024, 256], [64, 512, 128]], LQ_stage=True)   # multi-scale codebooks
    sd = ms.state_dict()
    assert tuple(sd["before_quant_group.1.weight"].shape) == (128, 512, 1, 1)      # femasr_arch.py:292,297
    assert tuple(sd["after_quant_group.1.conv.weight"].shape) == (256, 256 + 128, 3, 3)     # :293-294,298
    assert tuple(sd["quantize_group.1.embedding.weight"].shape) == (512, 128)
    hq = FeMaSRNet(codebook_params=[[32, 1024, 256]], LQ_stage=False, scale_factor=4)    # HQ stage: scale forced to 1
    assert hq.scale_factor == 1 and not any("swin" in k for k in hq.state_dict())


def test_module_copy_and_checkpoint_roundtrip(tmp_path):
    import copy
    from basicsr.archs.femasr_arch import FeMaSRNet
    net = FeMaSRNet(codebook_params=[[32, 1024, 256]], LQ_stage=True, scale_factor=2).eval()
    net._engine = object()          # stands in for a live native handle
    clone = copy.deepcopy(net)
    assert clone._engine is None and clone._engine_sig is None
    path = tmp_path / "w.pth"
    torch.save({"params": net.state_dict()}, path)            # the reference's checkpoint format (base_model.py:212-239)
    other = FeMaSRNet(codebook_params=[[32, 1024, 256]], LQ_stage=True, scale_factor=2)
    missing = other.load_state_dict(torch.load(path)["params"], strict=False)
    assert not missing.missing_keys and not missing.unexpected_keys
    for k, v in net.state_dict().items():
        assert torch.equal(v, other.state_dict()[k])


def test_graft_entry_build_runs():
    """The driver's build check: __graft_entry__.build() must compile the library and import the package (CPU only)."""
    import importlib
    ge = importlib.import_module("__graft_entry__")
    ge.build()

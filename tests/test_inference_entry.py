"""Config 1 plumbing (image folder -> PNGs): the reference's own entry script against this repo's surface on
CPU (must get as far as the device check), and the demo entry on the GPU against the oracle."""
import gzip
import hashlib
import json
import os
import runpy
import sys

import cv2
import numpy as np
import pytest
import torch

from basicsr.utils import img2tensor, tensor2img
from femasr_b200.spec import random_state_dict
from oracle import femasr_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# the reference's entry script, committed verbatim as a test input (tests/fixtures/README.md)
ENTRY_SCRIPT = os.path.join(ROOT, "tests", "fixtures", "inference_femasr.py")


def _write_inputs(folder, sizes, seed=3):
    rng = np.random.default_rng(seed)
    os.makedirs(folder, exist_ok=True)
    paths = []
    for i, (h, w) in enumerate(sizes):
        p = os.path.join(folder, f"img{i}.png")
        cv2.imwrite(p, rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
        paths.append(p)
    return paths


def test_image_helpers_roundtrip():
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, (9, 7, 3), dtype=np.uint8)
    t = img2tensor(img) / 255.0
    assert t.shape == (3, 9, 7) and t.dtype == torch.float32
    assert np.array_equal(t[0].numpy() * 255, img[:, :, 2])          # BGR -> RGB
    back = tensor2img(t.unsqueeze(0))
    assert back.dtype == np.uint8 and np.array_equal(back, img)
    assert tensor2img(torch.full((1, 3, 2, 2), 1.7)).max() == 255     # clamp before scaling


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour without a GPU")
def test_reference_entry_script_runs_unchanged_up_to_the_device(tmp_path, built_lib):
    """inference_femasr.py of the reference, unmodified, imports our basicsr, builds and loads the network and
    reads the image; without a GPU it must stop exactly at the first compute call (no CPU fallback)."""
    from femasr_b200.lib import FemasrError
    ins = _write_inputs(str(tmp_path / "in"), [(32, 32)])
    w = tmp_path / "w.pth"
    torch.save({"params": random_state_dict(4, 512, seed=1)}, w)
    argv = sys.argv
    sys.argv = ["inference_femasr.py", "-s", "4", "-i", ins[0], "-o", str(tmp_path / "out"), "-w", str(w)]
    try:
        with pytest.raises(FemasrError, match="CUDA sm_100"):
            runpy.run_path(ENTRY_SCRIPT, run_name="__main__")
    finally:
        sys.argv = argv


def test_fixture_is_the_reference_script():
    """tests/fixtures/inference_femasr.py (what tests/test_reference_entry_gpu.py executes) must be the reference's
    entry script byte for byte: its SHA-256 is the one tests/golden/make_golden.py recorded from the reference."""
    with gzip.open(os.path.join(ROOT, "tests", "golden", "reference_boundary.json.gz"), "rt") as f:
        want = json.load(f)["inference_femasr.py"]["sha256"]
    with open(ENTRY_SCRIPT, "rb") as f:
        assert hashlib.sha256(f.read()).hexdigest() == want


@pytest.mark.gpu
def test_demo_entry_matches_oracle_pngs(tmp_path, cuda):
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import run_inference
    sd = random_state_dict(4, 512, seed=2, init="perturbed")
    w = tmp_path / "w.pth"
    torch.save({"params": sd}, w)
    ins = _write_inputs(str(tmp_path / "in"), [(32, 48), (48, 32), (80, 64)])
    out_dir = tmp_path / "out"
    # max_size 70: the 80x64 image takes the test_tile path (default tile 240 -> one tile, still exercises it)
    assert run_inference.main(["-s", "4", "-i", str(tmp_path / "in"), "-o", str(out_dir), "-w", str(w), "--max_size", "70"]) == 0
    for p in ins:
        img = cv2.imread(p, cv2.IMREAD_UNCHANGED)
        x = (img2tensor(img) / 255.0).unsqueeze(0)
        with torch.no_grad():
            want = O.test(sd, x, 4) if x.shape[2] * x.shape[3] < 70 * 70 else O.test_tile(sd, x, 4)
        want_img = tensor2img(want)
        got = cv2.imread(str(out_dir / os.path.basename(p)), cv2.IMREAD_UNCHANGED)
        assert got.shape == want_img.shape == (img.shape[0] * 4, img.shape[1] * 4, 3)
        diff = np.abs(got.astype(int) - want_img.astype(int))
        assert diff.max() <= 1 and (diff > 0).mean() < 0.01, "PNG outputs must match to +-1 LSB"
    # bucketed uint8 fast path writes the same files
    out2 = tmp_path / "out2"
    assert run_inference.main(["-s", "4", "-i", str(tmp_path / "in"), "-o", str(out2), "-w", str(w), "--max_size", "70",
                               "--batch", "4"]) == 0
    for p in ins:
        a = cv2.imread(str(out_dir / os.path.basename(p)), cv2.IMREAD_UNCHANGED)
        b = cv2.imread(str(out2 / os.path.basename(p)), cv2.IMREAD_UNCHANGED)
        d = np.abs(a.astype(int) - b.astype(int))
        # not bit-identical: torch's CUDA `tensor / 255.` multiplies by fl(1/255) while the fused boundary kernel divides
        # (like torch on the CPU and the oracle), a last-bit difference of some inputs; +-1 LSB on a few bytes per thousand
        assert d.max() <= 1 and (d > 0).mean() < 5e-3


@pytest.mark.gpu
def test_uint8_boundary_matches_reference_image_pipeline(cuda):
    """sr_uint8 == tensor2img(test(img2tensor(img)/255)) of the reference's loop, bit for bit in uint8 except where
    the fp32 value sits within rounding noise of a .5 boundary."""
    from basicsr.archs.femasr_arch import FeMaSRNet
    sd = random_state_dict(4, 256, seed=4, init="perturbed")
    net = FeMaSRNet(codebook_params=[[32, 1024, 256]], LQ_stage=True, scale_factor=4)
    net.load_state_dict(sd, strict=True)
    net = net.to(cuda).eval()
    rng = np.random.default_rng(5)
    imgs = rng.integers(0, 256, (3, 40, 24, 3), dtype=np.uint8)
    got = net.sr_uint8(torch.from_numpy(imgs).to(cuda)).cpu().numpy()
    assert got.shape == (3, 160, 96, 3) and got.dtype == np.uint8
    for k in range(3):
        x = (img2tensor(imgs[k]) / 255.0).unsqueeze(0)
        want_f = net.test(x.to(cuda))
        want = tensor2img(want_f)
        diff = np.abs(got[k].astype(int) - want.astype(int))
        assert diff.max() <= 1 and (diff > 0).mean() < 5e-3      # see test_demo_entry_matches_oracle_pngs

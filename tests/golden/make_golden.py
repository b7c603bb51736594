"""Generate tests/golden/*.npz by running the UNMODIFIED reference (imported from /root/reference
through oracle/ref_shim.py) on seeded weights and inputs.  Run in the build container only:

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py

Weights are not stored: they are re-created anywhere by femasr_b200.spec.random_state_dict
(seeded per tensor name); a digest of the weights is stored so a drift in the generator is caught.
Inputs are stored (small), together with the reference's outputs at the public boundary and a
strided sample of its internal stage outputs (forward hooks on the reference modules).

reference_boundary.json.gz records the reference's state_dict() inventory (name, shape, dtype) for every
configuration of tests/test_boundary.py and the SHA-256 of its entry script, inference_femasr.py.
"""
from __future__ import annotations

import gzip
import hashlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from femasr_b200.spec import encode_depth, random_state_dict  # noqa: E402
from oracle.ref_shim import REFERENCE_ROOT, import_reference  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))

# name, scale, e_dim, init, seed, entry, input shape, extra
CASES = [
    ("x4_e256_fwd", 4, 256, "perturbed", 11, "forward", (2, 3, 32, 32), {}),
    ("x4_e512_fwd_default", 4, 512, "default", 12, "forward", (1, 3, 48, 64), {}),
    ("x2_e256_fwd", 2, 256, "perturbed", 13, "forward", (1, 3, 64, 96), {}),
    ("x4_e256_test", 4, 256, "perturbed", 14, "test", (1, 3, 40, 24), {}),
    ("x2_e512_test", 2, 512, "default", 15, "test", (1, 3, 40, 72), {}),
    ("x4_e256_tile", 4, 256, "perturbed", 16, "test_tile", (1, 3, 72, 56), {"tile_size": 32, "tile_pad": 8}),
    ("x4_e256_decode_indices", 4, 256, "perturbed", 17, "decode_indices", (2, 1, 4, 6), {}),
    # scale 1 = the HQ autoencoder (LQ_stage=False)
    ("hq_e512_fwd", 1, 512, "perturbed", 18, "forward", (1, 3, 64, 96), {}),
    ("hq_e256_test", 1, 256, "default", 19, "test", (1, 3, 40, 72), {}),
    # multi-scale codebooks (femasr_arch.py:280-299, 329-359): extra = codebook_params rows
    ("x4_ms2_fwd", 4, 256, "perturbed", 20, "forward", (1, 3, 32, 32), {"codebooks": [[32, 1024, 256], [64, 512, 128]]}),
    ("x2_ms3_fwd", 2, 256, "perturbed", 21, "forward", (1, 3, 64, 64),
     {"codebooks": [[32, 512, 256], [64, 512, 256], [128, 256, 128]]}),
    ("hq_ms2_fwd", 1, 256, "default", 22, "forward", (1, 3, 64, 64), {"codebooks": [[32, 1024, 256], [128, 256, 64]]}),
    # gt_indices loss branch (femasr_arch.py:70-78, 84-90): forward(input, gt_indices=[...])
    ("x4_e256_gt_fwd", 4, 256, "perturbed", 23, "forward", (2, 3, 32, 32), {"gt": True}),
    ("x4_ms2_gt_fwd", 4, 256, "perturbed", 24, "forward", (1, 3, 32, 32),
     {"codebooks": [[32, 1024, 256], [64, 512, 128]], "gt": True}),
]


# constructor flags (femasr_arch.py:224,226,349-350,361-362): pinned for the ORACLE only (tests/golden/cpu_only/, read by
# tests/test_oracle.py); the CUDA path is compared with the oracle for these flags in tests/test_net_gpu.py
CPU_ONLY_CASES = [
    ("x4_e256_noresidual_fwd", 4, 256, "perturbed", 25, "forward", (1, 3, 32, 32), {"ctor": {"use_residual": False}}),
    ("x4_e256_noquant_fwd", 4, 256, "perturbed", 26, "forward", (1, 3, 32, 32), {"ctor": {"use_quantize": False}}),
    ("x4_ms2_noquant_fwd", 4, 256, "perturbed", 27, "forward", (1, 3, 32, 32),
     {"codebooks": [[32, 1024, 256], [64, 512, 128]], "ctor": {"use_quantize": False}}),
]


def sd_digest(sd) -> str:
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(sd[k].contiguous().numpy().tobytes())
    return h.hexdigest()


def sample(t: torch.Tensor) -> np.ndarray:
    """Strided sample of an NCHW stage tensor (keeps fixtures small)."""
    return t[:, ::17, ::3, ::3].contiguous().numpy()


def write_reference_boundary(ref):
    from tests.test_boundary import CONFIGS, IDS
    inventory = {}
    for (scale, cbs), cid in zip(CONFIGS, IDS):
        net = ref.FeMaSRNet(codebook_params=cbs, LQ_stage=scale != 1, scale_factor=scale)
        inventory[cid] = [[k, list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in net.state_dict().items()]
    with open(os.path.join(REFERENCE_ROOT, "inference_femasr.py"), "rb") as f:
        script_sha256 = hashlib.sha256(f.read()).hexdigest()
    rec = {"state_dict": inventory, "inference_femasr.py": {"sha256": script_sha256}}
    path = os.path.join(OUT, "reference_boundary.json.gz")
    with open(path, "wb") as f:
        f.write(gzip.compress(json.dumps(rec, sort_keys=True).encode(), mtime=0))
    print(f"reference_boundary: {len(inventory)} state_dict inventories -> {os.path.getsize(path) / 1e3:.0f} kB")


def main():
    ref = import_reference()
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    only = set(sys.argv[1:])
    if not only or "reference_boundary" in only:
        write_reference_boundary(ref)
    for name, scale, e_dim, init, seed, entry, shape, extra in CASES + CPU_ONLY_CASES:
        if only and name not in only:
            continue
        extra = dict(extra)
        ctor = extra.pop("ctor", {})
        cbs = extra.pop("codebooks", [[32, 1024, e_dim]])
        use_gt = extra.pop("gt", False)
        sd = random_state_dict(scale, e_dim, seed=seed, init=init, codebooks=cbs)
        net = ref.FeMaSRNet(codebook_params=cbs, LQ_stage=scale != 1, scale_factor=scale, **ctor).eval()
        net.load_state_dict(sd, strict=True)
        g = torch.Generator().manual_seed(1000 + seed)
        rec = dict(scale=scale, e_dim=e_dim, init=init, seed=seed, entry=entry, digest=sd_digest(sd),
                   codebooks=np.array(cbs, dtype=np.int64))
        rec.update({f"arg_{k}": v for k, v in extra.items()})
        rec.update({f"ctor_{k}": v for k, v in ctor.items()})
        taps = {}
        d = encode_depth(scale)
        hooks = []

        def hook(key):
            def fn(_m, _i, o):
                taps[key] = o.detach().clone()
            return fn
        enc = net.multiscale_encoder
        hooks.append(enc.in_conv.register_forward_hook(hook("in_conv")))
        hooks.append(enc.blocks[d - 1].register_forward_hook(hook("down")))
        if scale != 1:
            hooks.append(enc.blocks[d].register_forward_hook(hook("swin")))
            hooks.append(enc.blocks[d + 1].register_forward_hook(hook("up1")))
            hooks.append(enc.blocks[d + 2].register_forward_hook(hook("up2")))
        hooks.append(net.before_quant_group[0].register_forward_hook(hook("z")))
        for k in range(1, len(cbs)):
            hooks.append(net.before_quant_group[k].register_forward_hook(hook(f"z{k}")))
        hooks.append(net.after_quant_group[0].register_forward_hook(hook("after_quant")))
        for i in range(3):
            hooks.append(net.decoder_group[i].register_forward_hook(hook(f"dec{i}")))
        with torch.no_grad():
            if entry == "decode_indices":
                x = torch.randint(0, 1024, shape, generator=g)
                out = net.decode_indices(x)
            else:
                x = torch.rand(shape, generator=g)
                if entry == "forward":
                    gt = None
                    if use_gt:          # random "HQ codes" of the right shapes
                        hb = shape[2] * scale // 8
                        gt = [torch.randint(0, n, (shape[0], 1, hb * s // 32, shape[3] * scale // 8 * s // 32), generator=g)
                              for s, n, _ in cbs]
                        rec.update({f"gt_indices{k}": v.numpy() for k, v in enumerate(gt)})
                    out, loss, sem, idx = net(x, gt) if use_gt else net(x)
                    rec.update(loss=loss.numpy(), sem=sem.numpy(), indices=idx[0].numpy())
                    rec.update({f"indices{k}": v.numpy() for k, v in enumerate(idx) if k > 0})
                elif entry == "test":
                    out = net.test(x)
                else:
                    out = net.test_tile(x, **extra)
        for h in hooks:
            h.remove()
        rec.update(input=x.numpy(), out=out.numpy())
        if entry == "forward":
            rec.update({f"tap_{k}": sample(v) for k, v in taps.items()})
        sub = os.path.join(OUT, "cpu_only") if ctor else OUT
        os.makedirs(sub, exist_ok=True)
        path = os.path.join(sub, name + ".npz")
        np.savez_compressed(path, **rec)
        print(f"{name}: out {tuple(out.shape)} |out|max {out.abs().max():.3f}  -> {os.path.getsize(path) / 1e3:.0f} kB")


if __name__ == "__main__":
    main()

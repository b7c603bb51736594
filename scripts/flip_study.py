#!/usr/bin/env python
"""GPU-box study behind tests/test_fullsize_gpu.py: codebook-index differences against the CPU oracle at the FULL benchmark
geometry (x4, 128x128, batch 32 = 131072 VQ rows, default tie-heavy init) for the tensor-core path and the fp32 path,
each classified by the ORACLE's own fp32 distances: a difference is "tie-equivalent" when the oracle's distance of our
code is within `k` grid steps (ulp of A = sum z^2) of the oracle's best - i.e. the two codes are separated by less than
the rounding noise of ANY fp32 evaluation order (the oracle itself moves this many rows when its thread count changes,
profiles/oracle_selfcheck_r2.json).

    python scripts/flip_study.py > gpurun_out/flip_study.json       (about 3 minutes, mostly the CPU oracle)
"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

VARIANTS = {
    "default (tcgen05, K-slice 256)": {},
    "fp32 FFMA path (gemm_path=0)": {"FEMASR_GEMM_PATH": "0"},
}


def child(out_path):
    from basicsr.archs.femasr_arch import FeMaSRNet
    from femasr_b200.spec import random_state_dict
    dev = torch.device("cuda", 0)
    sd = random_state_dict(4, 256, seed=0, init="default")
    x = torch.rand(32, 3, 128, 128, generator=torch.Generator().manual_seed(1))
    net = FeMaSRNet(codebook_params=[[32, 1024, 256]], LQ_stage=True, scale_factor=4)
    net.load_state_dict(sd, strict=True)
    net = net.to(dev).eval()
    _out, _loss, idx, taps = net._native(dev).forward(x.to(dev), taps=["z"])
    np.savez(out_path, idx=idx.cpu().numpy(), z=taps["z"].cpu().numpy())


def main():
    if len(sys.argv) > 2 and sys.argv[1] == "--child":
        return child(sys.argv[2])
    from femasr_b200.spec import random_state_dict
    from oracle import femasr_oracle as O
    sd = random_state_dict(4, 256, seed=0, init="default")
    x = torch.rand(32, 3, 128, 128, generator=torch.Generator().manual_seed(1))
    torch.set_num_threads(min(16, torch.get_num_threads()))
    zs, idxs = [], []
    with torch.no_grad():
        for i in range(0, 32, 8):
            taps = {}
            idxs.append(O.encode_and_decode(sd, x[i:i + 8], 4, taps)[3][0])
            zs.append(taps["z"])
    widx = torch.cat(idxs).reshape(-1)
    wz = torch.cat(zs).permute(0, 2, 3, 1).reshape(-1, 256).contiguous()
    cb = sd["quantize_group.0.embedding.weight"]
    res = {"rows": int(widx.numel())}
    for name, env in VARIANTS.items():
        path = f"/tmp/flip_{abs(hash(name)) % 10**8}.npz"
        e = dict(os.environ); e.update(env)
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", path], env=e, capture_output=True, text=True)
        if r.returncode != 0:
            res[name] = {"error": r.stderr[-400:]}
            continue
        d = np.load(path)
        idx = torch.from_numpy(d["idx"]).reshape(-1)
        z = torch.from_numpy(d["z"]).reshape(-1, 256)
        rows = torch.nonzero(idx != widx).reshape(-1)
        gaps = []
        for r_ in rows.tolist():
            dd = O.vq_dist(wz[r_:r_ + 1], cb)[0]                 # the oracle's own fp32 distances of this row
            a = float((wz[r_] ** 2).sum())
            ulp = float(np.spacing(np.float32(a)))
            gaps.append(round(float(dd[idx[r_]] - dd[widx[r_]]) / ulp, 2))
        zrel = float((z - wz).abs().max() / wz.abs().max())
        res[name] = {"flips": int(rows.numel()), "oracle_gap_in_grid_steps": gaps, "z_max_rel_err": zrel}
        print(name, res[name], file=sys.stderr, flush=True)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()

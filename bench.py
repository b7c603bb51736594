#!/usr/bin/env python
"""bench.py - images/sec of the FeMaSR x4 SR hot path (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config 2|3|5|2test] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one encode_and_decode pass (`FeMaSRNet.forward`) over one batch of synthetic LR images:
config 2 of BASELINE.json (x4, 128x128 LR, batch 32 per GPU, codebook 1024x256, random-init weights).
With N GPUs every rank runs its own batch of 32 (weak scaling, config 4 at N=8) followed by one NCCL
all-gather of the output shards, issued on a side stream so that it overlaps the NEXT step's forward (the rank's
output is first copied to a double-buffered staging tensor; the timed region ends only after the last all-gather).
--config selects another BASELINE.json configuration with the same line shape (3: x2 256x256 batch 16; 5: x4
test_tile(256,32) on one 1024x1024 image; 2test: config 2 through FeMaSRNet.test).  Prints ONE JSON line (rank 0).

  value     images/s, whole job, inputs already resident in HBM (forward [+ all-gather])
  e2e       same metric through the public surface with HOST buffers: pinned H2D of the LR batch,
            FeMaSRNet.forward, [all-gather], D2H of the rank's SR shard, all inside the timed region
  roofline  the dominant kernel (implicit-GEMM conv/linear) timed per launch with CUDA events on the
            launching stream (engine profile mode, extra steps after the timed region)
  cpu_baseline  the CPU oracle port (the reference's ATen-CPU arithmetic) on this host's cores, bounded sample
--impl reference runs only that CPU arm as the step and prints the same line shape.

--dump-outputs DIR writes what the timed path returned in its last timed step as DIR/<name>.npy (float32): `sr` (with N
GPUs the all-gathered batch) and, for the forward entry, rank 0's `codebook_loss` and `indices`.  Inputs and weights are
seeded, so two builds run with the same arguments can be compared output for output.  An array of more than
DUMP_MAX_VALUES values is stored as the 1-D sample of its values at a fixed seeded set of sorted flat positions (the same
set for every run of that shape), which keeps a dump under 64 MB.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "images/sec x4 SR 128->512 batch32"
GFLOP_PER_IMAGE = 754.53      # algorithmic, SURVEY.md 8d / BASELINE.md section 2 (x4 128x128 forward, e256)
# BASELINE.json configs; "2" is the one the metric is quoted on, the others print the same line shape for profiles/
CONFIGS = {
    "2": {"scale": 4, "lr": 128, "batch": 32, "entry": "forward", "name": "config 2"},
    "2test": {"scale": 4, "lr": 128, "batch": 32, "entry": "test", "name": "config 2 through test() (flip-pad to 144)"},
    "3": {"scale": 2, "lr": 256, "batch": 16, "entry": "forward", "name": "config 3"},
    "5": {"scale": 4, "lr": 1024, "batch": 1, "entry": "tile", "name": "config 5: test_tile(256, 32)"},
}
TILE, TILE_PAD = 256, 32
DUMP_MAX_VALUES = 1 << 23       # 32 MB of float32 per dumped array


def dump_array(path, t):
    """Saves an output to `path` as float32 (float64 stays float64), sampled as described in the module docstring."""
    import numpy as np
    import torch
    flat = t.detach().reshape(-1)
    if flat.numel() > DUMP_MAX_VALUES:
        pos = np.unique(np.random.default_rng(0).integers(0, flat.numel(), DUMP_MAX_VALUES))
        t = flat[torch.from_numpy(pos).to(flat.device)]
    a = t.detach().cpu().numpy()
    np.save(path, a if a.dtype == np.float64 else a.astype(np.float32))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops_burst": d.get("bf16_tflops"), "tflops_sustained": d.get("bf16_tflops_sustained"),
                "hbm_gbs": d.get("hbm_gbs"), "source": "measured (MEASURED_PEAKS.json)"}
    return {"tflops_burst": 1590.0, "tflops_sustained": 1400.0, "hbm_gbs": 6650.0,
            "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [v.strip() for v in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def cpu_arm(args, steps: int, warmup: int, budget_s: float = 25.0):
    """Times the CPU oracle port (ATen-CPU fp32) on a bounded sample of the workload: `sample_b` images of the
    configuration per step (entry `forward` / `test`), or ONE interior tile of the tiled configuration scaled by the
    padded-pixel count of all tiles (CPU time is proportional to pixels; BASELINE.md section 3).  The thread count is
    calibrated (all cores is often slower than fewer on a many-core host) and the best one is used and reported as
    `cores`.  Returns (img/s, ms/step, sample_b, info)."""
    import torch
    from femasr_b200.spec import random_state_dict
    from oracle import femasr_oracle as O
    try:
        ncpu = len(os.sched_getaffinity(0))
    except AttributeError:
        ncpu = os.cpu_count() or 1
    sd = random_state_dict(args.scale, args.e_dim, seed=0, init="default")
    g = torch.Generator().manual_seed(1)
    t_begin = time.perf_counter()
    tiled = args.entry == "tile"
    side = min(args.lr, TILE + 2 * TILE_PAD) if tiled else args.lr

    def run(x):
        if args.entry == "forward":
            return O.encode_and_decode(sd, x, args.scale)
        return O.test(sd, x, args.scale)

    with torch.no_grad():
        torch.set_num_threads(min(ncpu, 16))
        O.encode_and_decode(sd, torch.rand(1, 3, 32, 32, generator=g), args.scale)     # warm thread pools / primitives
        xc = torch.rand(1, 3, side, side, generator=g)
        best_t, best_n = None, min(ncpu, 8)
        # ascending: a container may see 128 CPUs but be allowed far fewer; stop as soon as more threads hurt
        for n in sorted({min(ncpu, 8), min(ncpu, 16), min(ncpu, 32), min(ncpu, 64), ncpu}):
            torch.set_num_threads(n)
            t0 = time.perf_counter()
            run(xc)
            dt = time.perf_counter() - t0
            if best_t is None or dt < best_t:
                best_t, best_n = dt, n
            elif dt > 1.15 * best_t:
                break
            if time.perf_counter() - t_begin > budget_s * 0.5:
                break
        torch.set_num_threads(best_n)
        left = max(2.0, budget_s - (time.perf_counter() - t_begin))
        per_step_budget = left / max(1, steps + warmup)
        sample_b = 1 if tiled else int(max(1, min(args.batch, per_step_budget / max(best_t, 1e-3))))
        x = torch.rand(sample_b, 3, side, side, generator=g)
        for _ in range(warmup):
            run(x)
        times = []
        for _ in range(steps):
            t0 = time.perf_counter()
            run(x)
            times.append(time.perf_counter() - t0)
    total = sum(times)
    if tiled:
        wsz = 8 // args.scale * 8
        pad = lambda n: (n // wsz + 1) * wsz
        px_all = sum(pad(t["in_win"][1] - t["in_win"][0]) * pad(t["in_win"][3] - t["in_win"][2])
                     for t in O.tile_plan(args.lr, args.lr, TILE, TILE_PAD))
        units = steps * (pad(side) * pad(side)) / px_all          # fraction of one whole tiled image per timed run
        ips = units / total
        what = (f"{steps} steps x ONE {side}x{side} interior tile through test() (padded {pad(side)}^2 of the {px_all} padded "
                f"pixels of the {len(O.tile_plan(args.lr, args.lr, TILE, TILE_PAD))} tiles of a {args.lr}x{args.lr} image; scaled by pixels)")
    else:
        ips = sample_b * steps / total
        what = f"{steps} steps x {sample_b} of the {args.batch} images of one batch ({args.lr}x{args.lr} LR, entry {args.entry})"
    info = {"value": round(ips, 4), "unit": "images/s", "cores": best_n, "host_cpus": ncpu, "kind": "port",
            "sample": f"{what}, x{args.scale}, e{args.e_dim}, oracle/femasr_oracle.py (the reference's ATen-CPU arithmetic) fp32, "
                      f"{best_n} threads (best of a calibration over thread counts on {ncpu} CPUs)"}
    return ips, total / steps * 1e3, sample_b, info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="2", choices=sorted(CONFIGS), help="BASELINE.json configuration (default 2 = the headline)")
    ap.add_argument("--batch", type=int, default=None, help="LR images per GPU per step (default: the configuration's)")
    ap.add_argument("--lr", type=int, default=None)
    ap.add_argument("--scale", type=int, default=None)
    ap.add_argument("--e-dim", type=int, default=256)
    ap.add_argument("--gemm-path", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs to DIR/<name>.npy (--impl b200)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200 (the CPU arm sizes its sample by timing, so its inputs vary)")
    cfgd = CONFIGS[args.config]
    args.batch = args.batch or cfgd["batch"]
    args.lr = args.lr or cfgd["lr"]
    args.scale = args.scale or cfgd["scale"]
    args.entry = cfgd["entry"]
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    # stdout carries exactly ONE JSON line (rank 0).  Everything else this process or its libraries write to fd 1 - NCCL's
    # version banner (printed at NCCL_DEBUG=VERSION and WARN), logger output - is sent to stderr: fd 1 is re-pointed at
    # stderr for the whole run and the JSON line goes to the saved descriptor at the end.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

    def emit(line: dict):
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    entry_name = {"forward": "FeMaSRNet.forward (encode_and_decode)", "test": "FeMaSRNet.test",
                  "tile": f"FeMaSRNet.test_tile({TILE}, {TILE_PAD})"}[args.entry]
    workload = (f"{CONFIGS[args.config]['name']}: x{args.scale} SR, synthetic {args.lr}x{args.lr} LR, batch {args.batch}/GPU, "
                f"codebook 1024x{args.e_dim}, {entry_name}, random-init weights")
    config = {"workload": workload, "global_batch": args.batch * max(world, 1), "per_gpu_batch": args.batch,
              "lr_size": args.lr, "scale": args.scale, "codebook": [1024, args.e_dim],
              "parallelism": (f"dp{world} (batch shards; one NCCL all-gather of the output shards per step on a side stream, "
                              "overlapping the next step's forward; drained inside the timed region)") if world > 1 else "single GPU",
              "l2": "no explicit flush: per-step working set (2.1 GB per decoder tensor at batch 32) >> 126 MB L2",
              "launch": "CUDA graph replay of the engine's launch list" if os.environ.get("FEMASR_CUDA_GRAPH", "1") != "0" else "eager launches"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        ips, ms, sample_b, info = cpu_arm(args, args.steps, args.warmup, budget_s=60.0)
        line = {"impl": "reference", "metric": METRIC if args.config == "2" else f"images/sec ({CONFIGS[args.config]['name']})", "value": info["value"], "unit": "images/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": info, "gpu_launches": 0,
                "e2e": {"value": info["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return 0

    # ------------------------------------------------------------------ B200 arm
    import torch
    import torch.distributed as dist
    from basicsr.archs import build_network
    from femasr_b200 import default_gemm_path
    from femasr_b200.spec import random_state_dict

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA sm_100 device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    gemm_path = args.gemm_path if args.gemm_path is not None else default_gemm_path()

    net = build_network(dict(type="FeMaSRNet", codebook_params=[[32, 1024, args.e_dim]], LQ_stage=True,
                             scale_factor=args.scale, gemm_path=gemm_path))
    net.load_state_dict(random_state_dict(args.scale, args.e_dim, seed=0, init="default"), strict=True)
    net = net.to(dev).eval()
    B, S = args.batch, args.lr
    g = torch.Generator().manual_seed(1 + rank)
    x_host = torch.rand(B, 3, S, S, generator=g).pin_memory()
    x_dev = x_host.to(dev)
    y_host = torch.empty(B, 3, S * args.scale, S * args.scale).pin_memory()
    eng = net._native(dev)

    def run_resident():
        """One pass of the configuration's entry over the device-resident batch -> {name: tensor} as its caller receives
        them (from a graph replay they live in the graph's static buffers until the next replay)."""
        if args.entry == "forward":
            # the engine's fixed launch list, replayed as a CUDA graph (same kernels, no per-launch host work)
            y, loss, idx = eng.forward_graph(x_dev) if eng.use_graph else eng.forward(x_dev, want_indices=True, want_loss=True)
            return {"sr": y, "codebook_loss": loss, "indices": idx}
        if args.entry == "test":
            return {"sr": eng.test(x_dev)}
        return {"sr": eng.test_tile(x_dev, TILE, TILE_PAD)}

    def run_public(xd):
        """The same through the reference-facing surface (what a user of FeMaSRNet calls)."""
        if args.entry == "forward":
            return net(xd)[0]
        if args.entry == "test":
            return net.test(xd)
        return net.test_tile(xd, TILE, TILE_PAD)

    # Output collective (N > 1): the rank's SR shard is copied to one of two staging tensors and all-gathered from there
    # on a side stream, so the collective of step i runs under the forward of step i+1 (the reference has no inference
    # collective; SURVEY 8e).  `drain` makes the timed region wait for the last one.
    class Gather:
        def __init__(self):
            shape = (B, 3, S * args.scale, S * args.scale)
            self.stage = [torch.empty(shape, device=dev) for _ in range(2)]
            self.done = [None, None]
            self.i = 0
            # Scheme: copy-engine peer writes (femasr_b200.parallel.PeerGather: no SM kernel next to the persistent
            # tensor-core kernels) when the GPUs can map each other, else the NCCL all-gather; FEMASR_GATHER=nccl|p2p forces one.
            want = os.environ.get("FEMASR_GATHER", "auto")
            self.peer = None
            if want in ("auto", "p2p"):
                try:
                    from femasr_b200.parallel import PeerGather
                    self.peer = PeerGather(shape, torch.float32, dev, rank, world, nbuf=2)
                except Exception as ex:       # any rank failing raises on every rank (collective self-check): uniform fallback
                    if want == "p2p":
                        raise
                    print(f"[bench] peer-copy gather unavailable ({type(ex).__name__}: {ex}); using NCCL", file=sys.stderr)
                    self.peer = None
            if self.peer is None:
                self.full = [torch.empty((world * B,) + shape[1:], device=dev) for _ in range(2)]
                self.stream = torch.cuda.Stream()
            else:
                self.full = self.peer.full
                self.stream = self.peer.stream
            self.scheme = "copy-engine peer writes over NVLink (CUDA IPC; no SM kernel)" if self.peer else "NCCL all-gather"

        def __call__(self, out):
            k = self.i & 1
            self.i += 1
            cur = torch.cuda.current_stream()
            if self.done[k] is not None:
                cur.wait_event(self.done[k])          # staging buffer k is free once its previous gather finished
            self.stage[k].copy_(out, non_blocking=True)
            ready = torch.cuda.Event()
            ready.record(cur)
            if self.peer is not None:
                self.done[k] = self.peer.push(k, self.stage[k], after=ready)
                return
            with torch.cuda.stream(self.stream):
                self.stream.wait_event(ready)
                dist.all_gather_into_tensor(self.full[k], self.stage[k])
                ev = torch.cuda.Event()
                ev.record(self.stream)
            self.done[k] = ev

        def drain(self):
            torch.cuda.current_stream().wait_stream(self.stream)

    gather = Gather() if world > 1 else None
    if gather:
        config["parallelism"] = (f"dp{world} (batch shards; one all-gather of the output shards per step - {gather.scheme} - on a side "
                                 "stream, overlapping the next step's forward; drained inside the timed region)")

    def step_resident():
        outs = run_resident()
        if gather:
            gather(outs["sr"])
        return outs

    def step_e2e():
        xd = x_host.to(dev, non_blocking=True)
        out = run_public(xd)
        if gather:
            gather(out)
        y_host.copy_(out, non_blocking=True)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """-> (ms for `steps` calls of fn, what the last call returned)."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            last = fn()
        if gather:
            gather.drain()                      # the last step's all-gather belongs to the timed region
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return ms.item(), last

    for _ in range(args.warmup):
        step_resident()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_total, last = timed(step_resident, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # before anything else runs: the e2e pass below replays the same graph into the same static buffers
        if gather:
            last = dict(last, sr=gather.full[(gather.i - 1) & 1])      # every rank's shard of the last step
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in last.items():
            dump_array(os.path.join(args.dump_outputs, f"{name}.npy"), t)
        print(f"[bench] last timed step's outputs written to {args.dump_outputs}: {sorted(last)}", file=sys.stderr)
    # one eager pass with the engine's profile mode on: counts the kernels one step launches (and their FLOPs)
    eng.set_profile(True)
    if args.entry == "forward":
        eng.forward(x_dev)
    else:
        run_resident()
    prof1 = eng.profile()
    eng.set_profile(False)
    launches = sum(v["launches"] for v in prof1.values()) * args.steps
    flops_step = sum(v["flops"] for v in prof1.values())
    for _ in range(2):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)

    # per-kernel CUDA-event timing (engine profile mode), 2 extra steps
    eng.set_profile(True)
    for _ in range(2):
        if args.entry == "forward":
            eng.forward(x_dev)
        else:
            run_resident()
    prof = eng.profile()
    eng.set_profile(False)

    if gather is not None and gather.peer is not None:
        torch.cuda.synchronize()
        gather.peer.close()               # unmap the peers' buffers while every exporting process is still alive
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peaks = load_peaks()
    ms_step = ms_total / args.steps
    imgs = B * world
    value = imgs / (ms_step / 1e3)
    e2e_value = imgs / (ms_e2e / args.steps / 1e3)
    if args.entry == "forward":
        flops_step = eng.flops(B, S, S)           # closed form == the sum over the launches' algorithmic FLOPs
    dom = max(prof.items(), key=lambda kv: kv[1]["ms"])
    dname, d = dom
    achieved = d["flops"] / (d["ms"] / 1e3) / 1e12 if d["ms"] > 0 else 0.0
    peak = peaks["tflops_sustained"] or peaks["tflops_burst"]
    tot_ms = sum(v["ms"] for v in prof.values())
    traffic, traffic_src = None, None
    tps = [os.path.join(ROOT, "profiles", f"tc_igemm_traffic_r{r}.json") for r in (2, 1)]
    tp = next((t for t in tps if os.path.exists(t)), None)
    if dname == "tc_igemm" and tp and args.config == "2":
        tj = json.load(open(tp))
        traffic = int(tj["dram_bytes_per_launch"])
        traffic_src = (f"profiles/{os.path.basename(tp)}: ncu dram__bytes_read.sum+dram__bytes_write.sum averaged over the "
                       f"{tj['launches']} tc_igemm launches of one batch-32 step (L2->SM traffic is "
                       f"{tj['l2_bytes_total'] / (tj['dram_read_bytes_total'] + tj['dram_write_bytes_total']):.1f}x that: the kernel is L2-bandwidth bound)")
    roofline = {"bound": "tensor", "kernel": dname, "achieved": round(achieved, 2), "peak": peak, "unit": "TFLOP/s",
                "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peaks["source"] + ", cuBLAS bf16 sustained (kernel timed inside a long step)",
                "launches_per_step": d["launches"] // 2, "avg_launch_ms": round(d["ms"] / max(1, d["launches"]), 4),
                "share_of_step": round(d["ms"] / tot_ms, 4) if tot_ms else None,
                "flops_counted": "algorithmic 2*MAC of the convs/linears this kernel executed",
                "arithmetic": "fp32 FFMA (SIMT)" if gemm_path == 0 else (
                    "tcgen05, fp32 accumulate in TMEM; in front of the VQ 3-MMA split-fp16 kind::f16 (hi*hi+hi*lo+lo*hi); behind it "
                    + ("a_hi*w_hi on kind::f16 + ONE kind::f8f6f4 e4m3 product for both cross terms (2.0 MMA units per algorithmic MMA)"
                       if os.environ.get("FEMASR_F8_CROSS", "1") != "0" else "the same 3 products")),
                "path_tflops": round(flops_step / (ms_step / 1e3) / 1e12, 2),
                "path_frac": round(flops_step / (ms_step / 1e3) / 1e12 / peak, 4),
                "kernels": {k: {"launches": v["launches"] // 2, "ms_per_step": round(v["ms"] / 2, 3)} for k, v in prof.items()}}
    metric = METRIC if args.config == "2" else f"images/sec ({CONFIGS[args.config]['name']})"
    line = {"metric": metric, "value": round(value, 2), "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_step, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "gflop_per_image": round(flops_step / B / 1e9, 2), "clocks": clocks, "gpu_launches": launches,
            "e2e": {"value": round(e2e_value, 2), "unit": "images/s", "h2d_bytes_per_step": x_host.numel() * 4,
                    "d2h_bytes_per_step": y_host.numel() * 4,
                    "note": f"{entry_name} on a pinned-host batch: H2D + the call (+ pipelined all-gather) + D2H of the rank's SR shard"},
            "roofline": roofline}
    if not args.no_cpu_baseline and world == 1:
        _, _, _, info = cpu_arm(args, steps=2, warmup=0, budget_s=20.0)
        line["cpu_baseline"] = info
    else:
        line["cpu_baseline"] = None
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())

#!/usr/bin/env python
"""SAC / TQC update time at precision 0 (fp32 FFMA tiles), 1 (tcgen05 from the break-even batch) and 2 (tcgen05 from
128 rows), one gcrl_sac_update_batch per update with the actor, alpha and Polyak steps (flags 1 | 2 | 4).

Method: per shape, three agents with the same seeded weights and the same seeded batch; 5 warm-up updates each (graph
capture included), then `--reps` rounds in which the precisions alternate, each timing `--updates` back-to-back
updates with CUDA events; the median round per precision is reported.  The working set (weights, activations, a
batch of at most 16384 rows) fits in L2; it is what an update reads every step.  A separate torch.profiler pass
lists each update's kernels and launch count (`--profile`).  Prints the GPU's name and power limit and one JSON line;
`--out FILE` also writes it there.

Usage: python profiles/sac_precision.py [--out FILE] [--profile FILE] [--updates N] [--reps R]"""
import argparse
import json
import os
import subprocess
import sys
from collections import Counter

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "goal-conditioned-rl-framework_b200"))
import numpy as np  # noqa: E402

# (algo, B, H): BASELINE configs[3] (TQC, Slide shape, hidden 512) and hidden 256 from 256 to 16384 rows
SHAPES = [(algo, B, H) for algo in ("tqc", "sac")
          for B, H in ((512, 512), (256, 256), (1024, 256), (2048, 256), (4096, 256), (16384, 256))]
D, A, L = 28, 4, 3            # FetchSlide / FetchPush: 25 observation + 3 goal dimensions, 4 actions; 3 hidden layers


def make(algo, B, H, precision):
    import torch
    from gcrl_b200 import SACAgent, TQCAgent
    from tests.test_sac_gpu import sac_config
    torch.manual_seed(0)
    cfg = sac_config(hidden_dim=H, layer_count=L, batch_size=B, grad_clip=5.0, tau=0.05, alpha_min_steps=0)
    return (SACAgent if algo == "sac" else TQCAgent)(D, A, cfg, None, 1, 2, precision=precision)


def batch(B):
    import torch
    rng = np.random.default_rng(B)
    s = rng.standard_normal((B, D)).astype(np.float32)
    arrs = (s, rng.uniform(-1, 1, (B, A)).astype(np.float32), -(rng.random((B, 1)) > 0.3).astype(np.float32),
            (s + 0.1 * rng.standard_normal((B, D))).astype(np.float32), (rng.random((B, 1)) < 0.1).astype(np.float32),
            rng.standard_normal((B, A)).astype(np.float32), rng.standard_normal((B, A)).astype(np.float32))
    return tuple(torch.from_numpy(x).cuda() for x in arrs)


def updater(ag, b):
    import torch
    from gcrl_b200._lib import check, lib, vp
    st = vp(torch.cuda.current_stream().cuda_stream)
    ptrs = [vp(t.data_ptr()) for t in b]
    B = b[0].shape[0]
    return lambda: check(lib.gcrl_sac_update_batch(ag._h, B, *ptrs, 1e-4, 1e-4, 1 | 2 | 4, None, st))


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--profile")
    ap.add_argument("--updates", type=int, default=20)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    name, power = gpu_info()
    print(f"GPU: {name}, power limit {power}", flush=True)
    result = {"gpu": name, "power_limit": power, "updates_per_round": args.updates, "rounds": args.reps,
              "flags": "actor + alpha + Polyak", "D": D, "A": A, "L": L, "shapes": []}
    profiles = []
    for algo, B, H in SHAPES:
        b = batch(B)
        run = {p: updater(make(algo, B, H, p), b) for p in (0, 1, 2)}
        for p in run:
            for _ in range(5):
                run[p]()
        torch.cuda.synchronize()
        times = {p: [] for p in run}
        for _ in range(args.reps):
            for p in run:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.updates):
                    run[p]()
                e1.record()
                e1.synchronize()
                times[p].append(e0.elapsed_time(e1) / args.updates)
        row = {"algo": algo, "B": B, "H": H}
        for p in run:
            row[f"p{p}_ms"] = round(float(np.median(times[p])), 4)
            row[f"p{p}_spread_ms"] = [round(float(min(times[p])), 4), round(float(max(times[p])), 4)]
        result["shapes"].append(row)
        print(json.dumps(row), flush=True)
        if args.profile:
            from torch.profiler import ProfilerActivity, profile
            for p in (0, 2):
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    run[p]()
                    torch.cuda.synchronize()
                kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
                by = Counter()
                us = Counter()
                for e in kern:
                    short = e.name.replace("(anonymous namespace)::", "").replace("void ", "")
                    short = short.split("<")[0].split("(")[0].split("::")[-1]
                    by[short] += 1
                    us[short] += e.device_time
                profiles.append({"algo": algo, "B": B, "H": H, "precision": p, "launches": len(kern),
                                 "kernel_us": round(sum(us.values()), 1),
                                 "kernels": {k: [by[k], round(us[k], 1)] for k in sorted(us, key=lambda k: -us[k])}})
        del run
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if args.profile:
        with open(args.profile, "w") as f:
            json.dump({"gpu": name, "power_limit": power, "profiles": profiles}, f, indent=1)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""The flushed B = 256 DDPG step of bench.py, with the time of each of its kernels.

Method: the bench's agent at the bench's shape (Push: obs 18, goal 3, action 3, H = 256 x 3, HER buffer of 1M
stored transitions from bench.py's seeded generator, device index stream, batch 256), warmed up like bench.py
(graph capture for both flag sets).  Then
  1. `--steps` steps, each after the same 256 MiB L2 flush as bench.py and bracketed by CUDA events: the median,
     10th / 90th percentile, minimum and mean step time;
  2. a separate torch.profiler run (CUDA activities) over `--profile-steps` flushed steps.  Every step's kernels
     lie between two flush kernels.  Per position of the six-launch step (steps with the Polyak of the actor
     target have seven and are reported apart) it gives the median kernel duration and the median time the kernel
     adds to the step: its end minus the previous kernel's end (its end minus its start for the first one).  With
     programmatic dependent launch a kernel may start before its predecessor ends, so its duration includes the
     wait; the added time does not.
Prints the GPU's name and power limit and one JSON line; `--out FILE` also writes it there.  The library is the
package's own unless GCRL_B200_LIB names another build, which is how two builds are compared: run the script once
per build, alternating.

Usage: python profiles/update_tail.py [--out FILE] [--steps N] [--profile-steps N] [--label TEXT]"""
import argparse
import json
import os
import subprocess
import sys
import time
import types
from collections import defaultdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "goal-conditioned-rl-framework_b200"))
import numpy as np  # noqa: E402

import bench  # noqa: E402  (synth, agent_config: the bench's data and agent, not its timing loop)


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:   # noqa: BLE001
        pl = "unknown"
    return name, pl


def short(name):
    return name.replace("void ", "").split("(")[0].replace("gcrl::", "")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--label", default="")
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--profile-steps", type=int, default=200)
    ap.add_argument("--batch", type=int, default=256)
    args = ap.parse_args()

    import torch
    from gcrl_b200 import DDPG, _lib
    assert torch.cuda.is_available(), "update_tail.py measures on a CUDA device"
    name, power = gpu_info()
    bargs = types.SimpleNamespace(hidden=256, layers=3, batch=args.batch, k_future=4)
    T, k, O, G, A, B = 50, bargs.k_future, 18, 3, 3, args.batch
    D = O + G
    E = 1_000_000 // T
    max_len = E * ((T - 1) * (k + 1) + 1)
    data = bench.synth(np.random.default_rng(1000), E, T, O, G, A, k)
    torch.manual_seed(1898)
    agent = DDPG(D, A, bench.agent_config(bargs, max_len), None, 1, 40, index_source="device", device=0,
                 max_batch=B, seed=1898)
    for e in range(E):
        agent.buffer.push_episode(data["s"][e], data["a"][e], data["ns"][e], data["r"][e], data["d"][e],
                                  data["ag"][e], data["fut"][e])
    torch.cuda.synchronize()
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)

    step = 1

    def run(n, timed):
        nonlocal step
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        for i, (e0, e1) in enumerate(evs):
            flush.fill_(i & 0xFF)
            if timed:
                e0.record(stream)
            agent._run_update(step, sync=False)
            step += 1
            if timed:
                e1.record(stream)
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in evs] if timed else None

    for _ in range(100):                       # bench.py: spinup 80 + warmup 20, graphs of both flag sets captured
        agent._run_update(step, sync=False)
        step += 1
    run(3, True)
    t = np.array(run(args.steps, True))
    timing = {"median_ms": round(float(np.median(t)), 5), "p10_ms": round(float(np.quantile(t, 0.1)), 5),
              "p90_ms": round(float(np.quantile(t, 0.9)), 5), "min_ms": round(float(t.min()), 5),
              "mean_ms": round(float(t.mean()), 5), "steps": int(t.size)}
    print(f"{name} ({power}): flushed step median {timing['median_ms']:.5f} ms", file=sys.stderr)

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run(args.profile_steps, False)
    kern = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                  key=lambda e: e.time_range.start)
    steps, cur = [], None
    for e in kern:
        if "gcrl::" not in e.name:             # the flush: a step boundary
            if cur:
                steps.append(cur)
            cur = []
            continue
        if cur is not None:
            cur.append((short(e.name), e.time_range.start, e.time_range.end))
    if cur:
        steps.append(cur)
    by_sig = defaultdict(list)
    for s in steps:
        by_sig[tuple(n for n, _, _ in s)].append(s)
    kernels = []
    for sig, group in sorted(by_sig.items(), key=lambda kv: -len(kv[1])):
        rows = []
        for i, kname in enumerate(sig):
            dur = [s[i][2] - s[i][1] for s in group]
            add = [s[i][2] - (s[i - 1][2] if i else s[i][1]) for s in group]
            rows.append({"kernel": kname, "duration_us": round(float(np.median(dur)), 2),
                         "adds_us": round(float(np.median(add)), 2)})
        span = [s[-1][2] - s[0][1] for s in group]
        kernels.append({"launches": len(sig), "steps": len(group), "span_us": round(float(np.median(span)), 2),
                        "kernels": rows})
    result = {"what": "flushed DDPG step, B = %d, H = 256 x 3, Push shape, 1M stored transitions" % B,
              "label": args.label, "gpu": name, "power_limit": power, "library": _lib.library_path(),
              "pdl_mask": os.environ.get("GCRL_PDL_MASK", "default"), "step": timing, "profile": kernels,
              "time": time.strftime("%Y-%m-%d %H:%M:%S")}
    line = json.dumps(result)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

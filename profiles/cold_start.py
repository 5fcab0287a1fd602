#!/usr/bin/env python
"""How much of the flushed B = 256 DDPG step is cold data and how much is cold code.

Method: the bench's agent at the bench's shape, built and warmed up as in profiles/update_tail.py.  The same update
then runs in three regimes, `--steps` steps each, every step bracketed by CUDA events (the events enclose the update
only):
  flush   : the 256 MiB L2 flush of bench.py before every step;
  rewarm  : the same flush, then reductions over every parameter array of the four networks (flat buffer and
            transposed copy) and the HER store's episode and bucket index tables, which pull them back into L2.
            The update then starts with warm data and cold instruction caches;
  b2b     : no flush, steps back to back.
A separate torch.profiler pass (CUDA activities, `--profile-steps` steps per regime) gives the median duration of
each kernel of the six-launch step.  flush - rewarm is the part of a time that re-reading the data costs, and
rewarm - b2b the part left to cold code (and to the data the re-warm does not touch: the sampled rows and goals).
Prints the GPU's name and power limit and one JSON line; `--out FILE` also writes it there.  The library is the
package's own unless GCRL_B200_LIB names another build: run the script once per build, alternating.

Usage: python profiles/cold_start.py [--out FILE] [--steps N] [--profile-steps N] [--label TEXT]"""
import argparse
import ctypes as C
import json
import os
import sys
import time
import types
from collections import defaultdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "goal-conditioned-rl-framework_b200"))
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import numpy as np  # noqa: E402

import bench  # noqa: E402  (synth, agent_config: the bench's data and agent, not its timing loop)
from update_tail import gpu_info, short  # noqa: E402

REGIMES = ("flush", "rewarm", "b2b")


def device_arrays(agent):
    """float32 views of every array the re-warm reads."""
    from gcrl_b200 import _lib
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC, NET_T_ACTOR, NET_T_CRITIC
    from gcrl_b200.parallel import device_tensor
    dev = agent.device_index
    views = []
    for net in (NET_ACTOR, NET_CRITIC, NET_T_ACTOR, NET_T_CRITIC):
        p, n, pt, nt = _lib.vp(), C.c_int64(), _lib.vp(), C.c_int64()
        _lib.check(_lib.lib.gcrl_agent_param_buffers(agent._h, net, C.byref(p), C.byref(n), C.byref(pt),
                                                     C.byref(nt)))
        views.append(device_tensor(p.value, n.value, dev))
        if pt.value and nt.value:
            views.append(device_tensor(pt.value, nt.value, dev))
    e, eb, b, bb = _lib.vp(), C.c_int64(), _lib.vp(), C.c_int64()
    _lib.check(_lib.lib.gcrl_her_index_tables(agent.buffer.handle, C.byref(e), C.byref(eb), C.byref(b), C.byref(bb)))
    views.append(device_tensor(e.value, eb.value // 4, dev))
    views.append(device_tensor(b.value, bb.value // 4, dev))
    return views


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--label", default="")
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--profile-steps", type=int, default=200)
    ap.add_argument("--batch", type=int, default=256)
    args = ap.parse_args()

    import torch
    from gcrl_b200 import DDPG, _lib
    assert torch.cuda.is_available(), "cold_start.py measures on a CUDA device"
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
    views = device_arrays(agent)
    sink = torch.empty(len(views), dtype=torch.float32, device=dev)
    rewarm_mib = sum(v.numel() for v in views) * 4 / 2**20

    step = 1

    def run(regime, n, timed):
        nonlocal step
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        for i, (e0, e1) in enumerate(evs):
            if regime != "b2b":
                flush.fill_(i & 0xFF)
            if regime == "rewarm":
                for j, v in enumerate(views):
                    torch.sum(v, dim=0, keepdim=True, out=sink[j:j + 1])
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
    for regime in REGIMES:
        run(regime, 3, True)

    timing = {}
    for regime in REGIMES:
        t = np.array(run(regime, args.steps, True))
        timing[regime] = {"median_ms": round(float(np.median(t)), 5), "p10_ms": round(float(np.quantile(t, 0.1)), 5),
                          "p90_ms": round(float(np.quantile(t, 0.9)), 5), "steps": int(t.size)}
        print(f"{name} ({power}): {regime} step median {timing[regime]['median_ms']:.5f} ms", file=sys.stderr)

    from torch.profiler import ProfilerActivity, profile
    kernels = {}
    for regime in REGIMES:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run(regime, args.profile_steps, False)
        kern = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                      key=lambda e: e.time_range.start)
        # a step is the run of library kernels between two foreign (flush / re-warm) kernels; back to back there
        # are none, so the step is cut at its first kernel, the critic phase
        steps, cur = [], None
        for e in kern:
            nm = short(e.name)
            if "gcrl::" not in e.name or (regime == "b2b" and "fused_critic_kernel" in nm):
                if cur:
                    steps.append(cur)
                cur = []
                if "gcrl::" not in e.name:
                    continue
            if cur is not None:
                cur.append((nm, e.time_range.start, e.time_range.end))
        if cur:
            steps.append(cur)
        by_sig = defaultdict(list)
        for s in steps:
            by_sig[tuple(n for n, _, _ in s)].append(s)
        sig, group = max(by_sig.items(), key=lambda kv: len(kv[1]))
        kernels[regime] = {"launches": len(sig), "steps": len(group),
                           "kernels": [{"kernel": kn, "duration_us": round(float(np.median(
                               [s[i][2] - s[i][1] for s in group])), 2)} for i, kn in enumerate(sig)]}

    split = {}
    sigs = {tuple(r["kernel"] for r in kernels[g]["kernels"]) for g in REGIMES}
    if len(sigs) == 1:
        for i, kn in enumerate(next(iter(sigs))):
            a, b, c = (kernels[g]["kernels"][i]["duration_us"] for g in REGIMES)
            split[f"{i}:{kn}"] = {"data_us": round(a - b, 2), "code_us": round(b - c, 2)}
    a, b, c = (timing[g]["median_ms"] * 1e3 for g in REGIMES)
    split["step"] = {"data_us": round(a - b, 2), "code_us": round(b - c, 2)}
    result = {"what": "cold-start split of the flushed DDPG step, B = %d, H = 256 x 3, Push shape, 1M stored "
                      "transitions" % B,
              "label": args.label, "gpu": name, "power_limit": power, "library": _lib.library_path(),
              "rewarm_mib": round(rewarm_mib, 2), "step": timing, "profile": kernels, "split": split,
              "time": time.strftime("%Y-%m-%d %H:%M:%S")}
    line = json.dumps(result)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

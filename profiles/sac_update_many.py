#!/usr/bin/env python
"""End-to-end wall time per SAC / TQC update: the ``update()`` loop against ``update_many(40)`` (one CUDA graph launch
per call, csrc/sac.cu: gcrl_sac_update_many).

Method as profiles/update_many.py: per shape one agent whose HER buffer holds 1M stored transitions (20 000 seeded
episodes of 50 steps, no eviction), for the host and the device index stream in turn.  Both variants are warmed up
first (graph capture included), then `--rounds` rounds in which the loop and ``update_many`` alternate (which one
goes first alternates too); a round times `--updates` updates of a variant -- `--updates / 40` calls of 40 steps --
from the first call to a device synchronise after the last, on the host clock.  The median round per variant is
reported.  Step lists start at 40 k + 1, so every call has the same flag pattern (actor every second step, SAC
Polyak at 40, alpha_min_steps not reached).  Prints the GPU's name and power limit and one JSON line; `--out FILE`
also writes it there.

Shapes (Push / Slide: obs 18 + goal 3, 3 actions, 3 hidden layers): SAC and TQC at B = 256, H = 256, precision 0;
TQC at BASELINE configs[3] (B = 512, H = 512, precision 1); TQC at B = 4096, H = 256, precision 1.

Usage: python profiles/sac_update_many.py [--out FILE] [--rounds R] [--updates N]"""
import argparse
import json
import os
import random
import sys
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "goal-conditioned-rl-framework_b200"))
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import numpy as np  # noqa: E402

from update_many import EPISODES, DISTINCT, A, D, K, L, T, episodes, gpu_info  # noqa: E402,F401

CONFIGS = [("sac", 256, 256, 0), ("tqc", 256, 256, 0), ("tqc", 512, 512, 1), ("tqc", 4096, 256, 1)]
N = 40


def make(algo, B, H, precision, eps):
    import torch
    from gcrl_b200 import SACAgent, TQCAgent
    max_len = EPISODES * ((T - 1) * (K + 1) + 1)
    cfg = types.SimpleNamespace(
        hidden_dim=H, layer_count=L, actor_lr=1e-3, actor_lr_min=1e-3, ac_scheduler_steps=1, critic_lr=1e-3,
        critic_lr_min=1e-3, cr_scheduler_steps=1, buffer_type="HER", max_len=max_len, alpha=1.0, batch_size=B,
        gamma=0.98, ac_update_freq=2, noise_std=0.2, noise_clamp=0.5, policy_noise=0.2, grad_clip=10.0, beta=1.0,
        beta_end=1, k_future=K, max_eps_len=T, tau=0.05, alpha_lr=3e-4, alpha_min=0.05, alpha_min_steps=10**6)
    torch.manual_seed(1898)
    ag = (SACAgent if algo == "sac" else TQCAgent)(D, A, cfg, None, 1, 40, index_source="device", max_batch=B,
                                                    precision=precision)
    for e in range(EPISODES):
        ag.buffer.push_episode(*eps[e % DISTINCT])
    torch.cuda.synchronize()
    assert len(ag.buffer) == max_len
    return ag


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--updates", type=int, default=80)
    args = ap.parse_args()
    name, power = gpu_info()
    print(f"GPU: {name}, power limit {power}", flush=True)
    result = {"gpu": name, "power_limit": power, "rounds": args.rounds, "updates_per_round": args.updates, "n": N,
              "buffer_transitions": EPISODES * T, "shape": {"D": D, "A": A, "L": L}, "rows": []}
    eps = episodes()
    random.seed(1898)
    for algo, B, H, precision in CONFIGS:
        ag = make(algo, B, H, precision, eps)
        for source in ("host", "device"):
            ag.index_source = ag.buffer.index_source = source
            calls = max(1, args.updates // N)
            lists = [list(range(40 * c + 1, 40 * c + 1 + N)) for c in range(calls)]

            def loop():
                for steps in lists:
                    for s in steps:
                        ag.update(s)

            def many():
                for steps in lists:
                    ag.update_many(steps)

            variants = {"loop": loop, "update_many": many}
            for fn in variants.values():           # warm-up: every graph of this shape captured
                fn()
            torch.cuda.synchronize()
            times = {k: [] for k in variants}
            for r in range(args.rounds):
                order = list(variants) if r % 2 == 0 else list(variants)[::-1]
                for k in order:
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    variants[k]()
                    torch.cuda.synchronize()
                    times[k].append((time.perf_counter() - t0) * 1e3 / (calls * N))
            row = {"algo": algo, "B": B, "H": H, "precision": precision, "index_source": source, "n": N,
                   "loop_ms": float(np.median(times["loop"])), "update_many_ms": float(np.median(times["update_many"])),
                   "loop_rounds_ms": times["loop"], "update_many_rounds_ms": times["update_many"]}
            row["speedup"] = row["loop_ms"] / row["update_many_ms"]
            print(json.dumps({k: v for k, v in row.items() if not k.endswith("rounds_ms")}), flush=True)
            result["rows"].append(row)
        del ag
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

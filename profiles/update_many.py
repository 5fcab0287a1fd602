#!/usr/bin/env python
"""End-to-end wall time per update: the ``update()`` loop against ``update_many`` (one CUDA graph launch per call).

Method: per (algorithm, batch) one agent whose HER buffer holds 1M stored transitions (20 000 seeded episodes of
50 steps, no eviction), for the host and the device index stream in turn.  For n in {1, 8, 40} every shape is
warmed up first (graph capture included), then `--rounds` rounds in which the two variants alternate (which one
goes first alternates too); a round times `--updates` updates of a variant -- `--updates / n` calls of n steps --
from the first call to a device synchronise after the last, on the host clock.  The median round per variant is
reported.  Step lists start at 40 k + 1, so every call of one n has the same flag pattern (DDPG Polyak at 40,
TD3 actor every second step).  Prints the GPU's name and power limit and one JSON line; `--out FILE` also writes
it there.

Usage: python profiles/update_many.py [--out FILE] [--rounds R] [--updates N]"""
import argparse
import json
import os
import random
import subprocess
import sys
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "goal-conditioned-rl-framework_b200"))
import numpy as np  # noqa: E402

O, G, A, H, L, T, K = 18, 3, 3, 256, 3, 50, 4      # the Push shape of bench.py's defaults
D = O + G
EPISODES, DISTINCT = 20000, 200                    # 1M transitions, cycling over 200 seeded episodes
CONFIGS = [("ddpg", 256), ("ddpg", 4096), ("ddpg", 65536), ("td3", 256)]
NS = (1, 8, 40)


def episodes():
    rng = np.random.default_rng(0)
    out = []
    for _ in range(DISTINCT):
        obs = rng.standard_normal((T + 1, D)).astype(np.float32)
        ag = np.cumsum(rng.normal(0, 0.05, (T + 1, G)), 0).astype(np.float32)
        fut = np.zeros((T, K), np.uint8)
        for t in range(T - 1):
            fut[t] = rng.integers(t + 1, T, K)
        out.append((obs[:-1], rng.uniform(-1, 1, (T, A)).astype(np.float32), obs[1:],
                    -(rng.random(T) > 0.2).astype(np.float32), np.zeros(T, np.float32), ag[1:], fut))
    return out


def make(algo, B, eps):
    import torch
    from gcrl_b200 import DDPG, TD3Agent
    max_len = EPISODES * ((T - 1) * (K + 1) + 1)
    cfg = types.SimpleNamespace(
        hidden_dim=H, layer_count=L, actor_lr=1e-3, actor_lr_min=1e-3, ac_scheduler_steps=1, critic_lr=1e-3,
        critic_lr_min=1e-3, cr_scheduler_steps=1, buffer_type="HER", max_len=max_len, alpha=1.0, batch_size=B,
        gamma=0.98, ac_update_freq=1 if algo == "ddpg" else 2, noise_std=0.2, noise_clamp=0.5, policy_noise=0.2,
        grad_clip=10.0, beta=1.0, beta_end=1, k_future=K, max_eps_len=T, tau=0.05)
    torch.manual_seed(1898)
    ag = (DDPG if algo == "ddpg" else TD3Agent)(D, A, cfg, None, 1, 40, index_source="device", max_batch=B)
    for e in range(EPISODES):
        ag.buffer.push_episode(*eps[e % DISTINCT])
    torch.cuda.synchronize()
    assert len(ag.buffer) == max_len
    return ag


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:   # noqa: BLE001
        pl = "unknown"
    return name, pl


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--updates", type=int, default=40)
    args = ap.parse_args()
    name, power = gpu_info()
    print(f"GPU: {name}, power limit {power}", flush=True)
    result = {"gpu": name, "power_limit": power, "rounds": args.rounds, "updates_per_round": args.updates,
              "buffer_transitions": EPISODES * T, "shape": {"D": D, "A": A, "H": H, "L": L}, "rows": []}
    eps = episodes()
    random.seed(1898)
    for algo, B in CONFIGS:
        ag = make(algo, B, eps)
        for source in ("host", "device"):
            ag.index_source = ag.buffer.index_source = source
            for n in NS:
                calls = max(1, args.updates // n)
                lists = [list(range(40 * c + 1, 40 * c + 1 + n)) for c in range(calls)]

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
                        times[k].append((time.perf_counter() - t0) * 1e3 / (calls * n))
                row = {"algo": algo, "B": B, "index_source": source, "n": n,
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

#!/usr/bin/env python
"""End-to-end wall time per update from a uniform (REPLAY) or prioritised (PER) buffer: the ``update()`` loop against
``update_many(40)`` (csrc/agent.cu: gcrl_agent_update_many_replay, csrc/sac.cu: gcrl_sac_update_many_replay).

Method as profiles/update_many.py: per shape one agent whose ring holds 1M stored transitions (seeded rows, full, no
eviction during the run).  Both variants are warmed up first (graph capture included: a PER key is captured on its
second call), then `--rounds` rounds in which the loop and ``update_many`` alternate (which one goes first alternates
too); a round times `--updates` updates of a variant -- `--updates / 40` calls of 40 steps -- from the first call to a
device synchronise after the last, on the host clock.  The median round per variant is reported.  Step lists start at
40 k + 1, so every call has the same flag pattern.  Prints the GPU's name and power limit and one JSON line; `--out
FILE` also writes it there.

Shapes (Push / Slide: obs 18 + goal 3, 3 actions, 3 hidden layers of 256): DDPG and TQC at B = 256 (TQC precision 0)
and B = 4096 (precision 1: tcgen05), each with REPLAY and PER (alpha 0.6, beta annealing from 0.4).

Usage: python profiles/replay_update_many.py [--out FILE] [--rounds R] [--updates N]"""
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

from update_many import A, D, L, gpu_info  # noqa: E402

CONFIGS = [("ddpg", 256, 1), ("ddpg", 4096, 1), ("tqc", 256, 0), ("tqc", 4096, 1)]
KINDS = ("REPLAY", "PER")
STORED = 1 << 20
H, N = 256, 40


def make(algo, kind, B, precision):
    import torch
    from gcrl_b200 import DDPG, TQCAgent
    cfg = types.SimpleNamespace(
        hidden_dim=H, layer_count=L, actor_lr=1e-3, actor_lr_min=1e-3, ac_scheduler_steps=1, critic_lr=1e-3,
        critic_lr_min=1e-3, cr_scheduler_steps=1, buffer_type=kind, max_len=STORED, alpha=0.6, batch_size=B,
        gamma=0.98, ac_update_freq=2, noise_std=0.2, noise_clamp=0.5, policy_noise=0.2, grad_clip=10.0, beta=0.4,
        beta_end=10**5, k_future=4, max_eps_len=50, tau=0.05, alpha_lr=3e-4, alpha_min=0.05, alpha_min_steps=10**6)
    torch.manual_seed(1898)
    ag = (DDPG if algo == "ddpg" else TQCAgent)(D, A, cfg, None, 1, 40, max_batch=B, precision=precision)
    rng = np.random.default_rng(1898)
    for lo in range(0, STORED, 1 << 17):
        n = min(1 << 17, STORED - lo)
        ag.buffer.push_rows(rng.standard_normal((n, D), np.float32), rng.uniform(-1, 1, (n, A)).astype(np.float32),
                            -(rng.random(n) > 0.3).astype(np.float32), rng.standard_normal((n, D), np.float32),
                            (rng.random(n) < 0.02).astype(np.float32))
    torch.cuda.synchronize()
    assert len(ag.buffer) == STORED
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
              "buffer_transitions": STORED, "shape": {"D": D, "A": A, "H": H, "L": L}, "rows": []}
    random.seed(1898)
    np.random.seed(1898)
    for algo, B, precision in CONFIGS:
        for kind in KINDS:
            ag = make(algo, kind, B, precision)
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
            for _ in range(2):                     # warm-up: every graph of this shape captured
                for fn in variants.values():
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
            row = {"algo": algo, "buffer": kind, "B": B, "precision": precision, "n": N,
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

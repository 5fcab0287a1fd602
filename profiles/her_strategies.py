#!/usr/bin/env python
"""HER sampling cost of the goal-selection modes: eager `future` (offsets drawn at commit, three dependent round trips:
bucket record -> packed row || offset word -> goal) against online `future` / `final` / `episode` (coin and goal step
hashed at sample time, so the goal gather is issued beside the row gather).

Method, one command, all variants alternating inside every round:
  * standalone sampler (gcrl_her_sample, device positions) at B = 256, 4096, 65 536 and 1M (10^6, the whole online
    store) over stores of 1M stored
    transitions (20 000 seeded episodes of 50 steps; eager k = 4 -> 4.92M deque entries, online k = 4 -> 1M).  A
    timed pass is: overwrite the L2 (a 512 MB fill), then CUDA events around ONE sample launch, enqueued behind
    the fill so that the GPU runs them back to back.  Median over `--rounds` passes.
  * DDPG `update_many(40)` per update at B = 256 and 65 536 (device index stream, Push shape H = 256), eager
    `future` against online `future`: L2 overwritten, then the host clock from the call to a device synchronise.
    Median over `--rounds` passes, after a warm-up call (graph capture).
Prints the GPU's name and power limit and one JSON line; `--out FILE` also writes it there.

Usage: python profiles/her_strategies.py [--out FILE] [--rounds R]"""
import argparse
import json
import os
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
SAMPLER_B = (256, 4096, 65536, 1000000)
UPDATE_B = (256, 65536)
MODES = {"eager_future": ("future", False), "online_future": ("future", True), "online_final": ("final", True),
         "online_episode": ("episode", True)}


def episodes():
    rng = np.random.default_rng(0)
    out = []
    for _ in range(DISTINCT):
        obs = rng.standard_normal((T + 1, D)).astype(np.float32)
        ag = np.cumsum(rng.normal(0, 0.05, (T + 1, G)), 0).astype(np.float32)
        out.append((obs[:-1], rng.uniform(-1, 1, (T, A)).astype(np.float32), obs[1:],
                    -(rng.random(T) > 0.2).astype(np.float32), np.zeros(T, np.float32), ag[1:]))
    return out


def max_len(online):
    return EPISODES * (T if online else (T - 1) * (K + 1) + 1)


def fill(buf, eps):
    import torch
    for e in range(EPISODES):
        buf.push_episode(*eps[e % DISTINCT])
    torch.cuda.synchronize()


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:   # noqa: BLE001
        pl = "unknown"
    return name, pl


def time_sampler(eps, rounds, flush):
    import torch
    from gcrl_b200 import HERBuffer
    from gcrl_b200._lib import check, lib, vp
    bufs = {}
    for mode, (strategy, online) in MODES.items():
        b = HERBuffer(max_len(online), T, 1, k_future=K, index_source="device", goal_selection_strategy=strategy,
                      online_sampling=online)
        fill(b, eps)
        assert len(b) == max_len(online)
        bufs[mode] = b
    st = torch.cuda.current_stream()
    rows = []
    for B in SAMPLER_B:
        out = [torch.empty((B, w), dtype=torch.float32, device="cuda") for w in (D, A, 1, D, 1)]
        ptrs = [vp(x.data_ptr()) for x in out]
        times = {m: [] for m in bufs}
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for m, b in bufs.items():                                 # warm-up
            check(lib.gcrl_her_sample(b.handle, B, None, *ptrs, None, vp(st.cuda_stream)))
        for r in range(rounds):
            order = list(bufs) if r % 2 == 0 else list(bufs)[::-1]
            for m in order:
                flush.fill_(float(r))
                ev0.record(st)
                check(lib.gcrl_her_sample(bufs[m].handle, B, None, *ptrs, None, vp(st.cuda_stream)))
                ev1.record(st)
                ev1.synchronize()
                times[m].append(ev0.elapsed_time(ev1) * 1e3)
        row = {"what": "sampler", "B": B}
        for m in bufs:
            row[f"{m}_us"] = float(np.median(times[m]))
        row["online_future_over_eager"] = row["online_future_us"] / row["eager_future_us"]
        print(json.dumps(row), flush=True)
        rows.append(row)
        del out
    del bufs
    torch.cuda.empty_cache()
    return rows


def time_updates(eps, rounds, flush):
    import torch
    from gcrl_b200 import DDPG
    rows = []
    for B in UPDATE_B:
        agents = {}
        for mode in ("eager_future", "online_future"):
            strategy, online = MODES[mode]
            cfg = types.SimpleNamespace(
                hidden_dim=H, layer_count=L, actor_lr=1e-3, actor_lr_min=1e-3, ac_scheduler_steps=1, critic_lr=1e-3,
                critic_lr_min=1e-3, cr_scheduler_steps=1, buffer_type="HER", max_len=max_len(online), alpha=1.0,
                batch_size=B, gamma=0.98, ac_update_freq=1, noise_std=0.2, noise_clamp=0.5, policy_noise=0.2,
                grad_clip=10.0, beta=1.0, beta_end=1, k_future=K, max_eps_len=T, tau=0.05)
            torch.manual_seed(1898)
            ag = DDPG(D, A, cfg, None, 1, 40, index_source="device", max_batch=B, goal_selection_strategy=strategy,
                      online_sampling=online)
            fill(ag.buffer, eps)
            agents[mode] = ag
        steps = list(range(41, 81))
        for ag in agents.values():
            ag.update_many(steps)                                   # warm-up: graph capture
        torch.cuda.synchronize()
        times = {m: [] for m in agents}
        for r in range(rounds):
            order = list(agents) if r % 2 == 0 else list(agents)[::-1]
            for m in order:
                flush.fill_(float(r))
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                agents[m].update_many(steps)
                torch.cuda.synchronize()
                times[m].append((time.perf_counter() - t0) * 1e3 / len(steps))
        row = {"what": "ddpg_update_many_40_per_update", "B": B}
        for m in agents:
            row[f"{m}_ms"] = float(np.median(times[m]))
        row["online_future_over_eager"] = row["online_future_ms"] / row["eager_future_ms"]
        print(json.dumps(row), flush=True)
        rows.append(row)
        del agents
        torch.cuda.empty_cache()
    return rows


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--rounds", type=int, default=31)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("profiles/her_strategies.py measures on the GPU; no CUDA device found")
    name, power = gpu_info()
    print(f"GPU: {name}, power limit {power}", flush=True)
    flush = torch.empty(128 << 20, dtype=torch.float32, device="cuda")    # 512 MB: four times the L2
    eps = episodes()
    result = {"gpu": name, "power_limit": power, "rounds": args.rounds, "stored_transitions": EPISODES * T,
              "k_future": K, "shape": {"D": D, "A": A, "G": G, "H": H, "L": L}, "index_source": "device",
              "rows": time_sampler(eps, args.rounds, flush) + time_updates(eps, max(5, args.rounds // 3), flush)}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

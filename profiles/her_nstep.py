#!/usr/bin/env python
"""Cost of n-step rows in the HER sampler (her_sample_kernel<..., NSTEP = true>) against one-step rows.

Method as profiles/her_strategies.py (whose store, flush and timing helpers this script reuses), one command, all
variants alternating inside every round:
  * standalone sampler (gcrl_her_sample, device positions) at B = 256, 4096, 65 536 and 10^6 over stores of 1M stored
    transitions (20 000 seeded episodes of 50 steps, Push shape), eager `future` (k = 4) and online `future`, at
    n = 1, 3 and 5.  A timed pass overwrites the L2 (a 512 MB fill), then CUDA events around ONE sample launch.
    Median over `--rounds` passes.  Bytes per row are modelled: the one-step row's 373 B (the profile of
    profiles/her_strategies.py) plus, for n > 1, the s' segment of row t+k-1 (D floats) and one 32 B sector per
    extra window step (a reward word, or a compact achieved goal) -- an upper bound, k = min(n, T - t) <= n.
  * per update of `update_many(40)` (device index stream, eager `future`, H = 256): DDPG B = 256 (n = 1 samples
    inside the row-slab critic kernel, n = 3 launches the standalone sampler), DDPG B = 4096, TQC B = 256.  L2
    overwritten, then the host clock from the call to a device synchronise; median over max(5, rounds / 3) passes.
Prints the GPU's name and power limit and one JSON line; `--out FILE` also writes it there.

Usage: python profiles/her_nstep.py [--out FILE] [--rounds R]"""
import argparse
import json
import os
import sys
import time
import types

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import her_strategies as HS  # noqa: E402
import numpy as np  # noqa: E402

NS = (1, 3, 5)
MODES = {"eager_future": False, "online_future": True}
ROW_BYTES = 373


def row_bytes(n):
    return ROW_BYTES + (0 if n == 1 else HS.D * 4 + (n - 1) * 32)


def time_sampler(eps, rounds, flush):
    import torch
    from gcrl_b200 import HERBuffer
    from gcrl_b200._lib import check, lib, vp
    bufs = {}
    for mode, online in MODES.items():
        for n in NS:
            b = HERBuffer(HS.max_len(online), HS.T, 1, k_future=HS.K, index_source="device", online_sampling=online,
                          n_step=n, gamma=0.98)
            HS.fill(b, eps)
            bufs[(mode, n)] = b
    st = torch.cuda.current_stream()
    rows = []
    for B in HS.SAMPLER_B:
        out = [torch.empty((B, w), dtype=torch.float32, device="cuda") for w in (HS.D, HS.A, 1, HS.D, 1)]
        ptrs = [vp(x.data_ptr()) for x in out]
        times = {key: [] for key in bufs}
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for b in bufs.values():
            check(lib.gcrl_her_sample(b.handle, B, None, *ptrs, None, vp(st.cuda_stream)))
        for r in range(rounds):
            order = list(bufs) if r % 2 == 0 else list(bufs)[::-1]
            for key in order:
                flush.fill_(float(r))
                ev0.record(st)
                check(lib.gcrl_her_sample(bufs[key].handle, B, None, *ptrs, None, vp(st.cuda_stream)))
                ev1.record(st)
                ev1.synchronize()
                times[key].append(ev0.elapsed_time(ev1) * 1e3)
        for mode in MODES:
            row = {"what": "sampler", "mode": mode, "B": B}
            for n in NS:
                us = float(np.median(times[(mode, n)]))
                row[f"n{n}_us"] = us
                row[f"n{n}_bytes_per_row"] = row_bytes(n)
                row[f"n{n}_GBps"] = B * row_bytes(n) / (us * 1e-6) / 1e9
            print(json.dumps(row), flush=True)
            rows.append(row)
        del out
    del bufs
    torch.cuda.empty_cache()
    return rows


def time_updates(eps, rounds, flush):
    import torch
    from gcrl_b200 import DDPG, TQCAgent
    rows = []
    for algo, B in (("ddpg", 256), ("ddpg", 4096), ("tqc", 256)):
        agents = {}
        for n in (1, 3):
            cfg = types.SimpleNamespace(
                hidden_dim=HS.H, layer_count=HS.L, actor_lr=1e-3, actor_lr_min=1e-3, ac_scheduler_steps=1,
                critic_lr=1e-3, critic_lr_min=1e-3, cr_scheduler_steps=1, buffer_type="HER", max_len=HS.max_len(False),
                alpha=1.0, batch_size=B, gamma=0.98, ac_update_freq=1, noise_std=0.2, noise_clamp=0.5,
                policy_noise=0.2, grad_clip=10.0, beta=1.0, beta_end=1, k_future=HS.K, max_eps_len=HS.T, tau=0.05)
            torch.manual_seed(1898)
            cls = DDPG if algo == "ddpg" else TQCAgent
            ag = cls(HS.D, HS.A, cfg, None, 1, 40, index_source="device", max_batch=B, n_step=n)
            HS.fill(ag.buffer, eps)
            agents[n] = ag
        steps = list(range(41, 81))
        for ag in agents.values():
            ag.update_many(steps)                                   # warm-up: graph capture
        torch.cuda.synchronize()
        times = {n: [] for n in agents}
        for r in range(rounds):
            order = list(agents) if r % 2 == 0 else list(agents)[::-1]
            for n in order:
                flush.fill_(float(r))
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                agents[n].update_many(steps)
                torch.cuda.synchronize()
                times[n].append((time.perf_counter() - t0) * 1e3 / len(steps))
        row = {"what": f"{algo}_update_many_40_per_update", "B": B}
        for n in agents:
            row[f"n{n}_ms"] = float(np.median(times[n]))
        row["n3_minus_n1_us"] = (row["n3_ms"] - row["n1_ms"]) * 1e3
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
        raise SystemExit("profiles/her_nstep.py measures on the GPU; no CUDA device found")
    name, power = HS.gpu_info()
    print(f"GPU: {name}, power limit {power}", flush=True)
    flush = torch.empty(128 << 20, dtype=torch.float32, device="cuda")    # 512 MB: four times the L2
    eps = HS.episodes()
    result = {"gpu": name, "power_limit": power, "rounds": args.rounds, "stored_transitions": HS.EPISODES * HS.T,
              "k_future": HS.K, "gamma": 0.98, "shape": {"D": HS.D, "A": HS.A, "G": HS.G, "H": HS.H, "L": HS.L},
              "index_source": "device",
              "rows": time_sampler(eps, args.rounds, flush) + time_updates(eps, max(5, args.rounds // 3), flush)}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Cost of quantile critics: per-update wall time of scalar TQC (5 scalar critics, MSE) against quantile TQC
(``TQCAgent(n_quantiles=25, top_quantiles_to_drop_per_net=2)``), and the time of the quantile mode's own kernels.

Timing (profiler off): per shape one scalar and one quantile agent, each with a HER buffer of `--episodes` seeded
episodes (device index stream).  Four variants -- scalar / quantile through ``update()`` and through
``update_many(40)`` -- are warmed up (graph capture included), then `--rounds` rounds in which they alternate (the
order reverses every round); a round times `--updates` updates of a variant from the first call to a device
synchronise after the last, on the host clock.  The median round per variant is reported.  Step lists start at
40 k + 1, so every call has the same flag pattern (actor every second step, alpha_min_steps not reached).

Kernels (a separate run, torch.profiler with CUDA activities): `--prof-updates` update() calls of each agent; per
kernel name the total device time per update.  quantile_target_kernel and quantile_huber_kernel run once per
update; the huber kernel's pair rate is B n M K pairs (u = y_j - Z_ik) over its time.  The head GEMMs of the
quantile mode run on the same fp32 tile kernels as the hidden layers (batched_gemm_kernel, multi_wgrad_kernel), so
their time is reported as the difference of those kernels' per-update time between the quantile and the scalar
agent (the hidden layers are the same launches in both), next to the scalar head kernels they replace.

Shapes (obs 18 + goal 3, 3 actions, 3 hidden layers): B = 256, H = 256, precision 0; B = 512, H = 512, precision 1
(BASELINE configs[3]); B = 4096, H = 256, precision 1.  Prints the GPU's name and power limit and one JSON line;
`--out FILE` also writes it there.

Usage: python profiles/tqc_quantiles.py [--out FILE] [--rounds R] [--updates N]"""
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

from update_many import DISTINCT, A, D, K, L, T, episodes, gpu_info  # noqa: E402

SHAPES = [(256, 256, 0), (512, 512, 1), (4096, 256, 1)]
M, DROP, NCRIT = 25, 2, 5
N = 40
GEMM_KERNELS = ("batched_gemm_kernel", "multi_wgrad_kernel", "gemm_kernel")
SCALAR_HEAD_KERNELS = ("head_fwd_batched_kernel", "head_bwd_batched_kernel", "head_bwd_kernel", "head_fwd_kernel")


def make(B, H, precision, quantile, eps, n_episodes):
    import torch
    from gcrl_b200 import TQCAgent
    max_len = n_episodes * ((T - 1) * (K + 1) + 1)
    cfg = types.SimpleNamespace(
        hidden_dim=H, layer_count=L, actor_lr=1e-3, actor_lr_min=1e-3, ac_scheduler_steps=1, critic_lr=1e-3,
        critic_lr_min=1e-3, cr_scheduler_steps=1, buffer_type="HER", max_len=max_len, alpha=1.0, batch_size=B,
        gamma=0.98, ac_update_freq=2, noise_std=0.2, noise_clamp=0.5, policy_noise=0.2, grad_clip=10.0, beta=1.0,
        beta_end=1, k_future=K, max_eps_len=T, tau=0.05, alpha_lr=3e-4, alpha_min=0.05, alpha_min_steps=10**6)
    torch.manual_seed(1898)
    kw = dict(n_quantiles=M, top_quantiles_to_drop_per_net=DROP) if quantile else {}
    ag = TQCAgent(D, A, cfg, None, 1, 40, index_source="device", max_batch=B, precision=precision, **kw)
    for e in range(n_episodes):
        ag.buffer.push_episode(*eps[e % DISTINCT])
    torch.cuda.synchronize()
    return ag


def kernel_times(ag, updates, first_step):
    """{kernel name: (device us per update, launches per update)} over `updates` update() calls."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    for s in range(first_step, first_step + 4):
        ag.update(s)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for s in range(first_step + 4, first_step + 4 + updates):
            ag.update(s)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t and e.count:
            out[e.key] = (t / updates, e.count / updates)
    return out


def summed(times, names):
    return sum(v[0] for k, v in times.items() if any(n in k for n in names))


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--updates", type=int, default=80)
    ap.add_argument("--prof-updates", type=int, default=40)
    ap.add_argument("--episodes", type=int, default=2000)
    args = ap.parse_args()
    name, power = gpu_info()
    print(f"GPU: {name}, power limit {power}", flush=True)
    result = {"gpu": name, "power_limit": power, "rounds": args.rounds, "updates_per_round": args.updates, "n": N,
              "n_quantiles": M, "top_quantiles_to_drop_per_net": DROP, "n_critics": NCRIT,
              "buffer_transitions": args.episodes * T, "shape": {"D": D, "A": A, "L": L}, "rows": []}
    eps = episodes()
    random.seed(1898)
    for B, H, precision in SHAPES:
        agents = {"scalar": make(B, H, precision, False, eps, args.episodes),
                  "quantile": make(B, H, precision, True, eps, args.episodes)}
        calls = max(1, args.updates // N)
        lists = [list(range(40 * c + 1, 40 * c + 1 + N)) for c in range(calls)]

        def loop(ag):
            for steps in lists:
                for s in steps:
                    ag.update(s)

        def many(ag):
            for steps in lists:
                ag.update_many(steps)

        variants = {f"{k}_{how}": (lambda ag=ag, fn=fn: fn(ag)) for k, ag in agents.items()
                    for how, fn in (("update", loop), ("update_many", many))}
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
        row = {"B": B, "H": H, "precision": precision}
        for k, v in times.items():
            row[f"{k}_ms"] = float(np.median(v))
            row[f"{k}_rounds_ms"] = v
        for how in ("update", "update_many"):
            row[f"quantile_over_scalar_{how}"] = row[f"quantile_{how}_ms"] / row[f"scalar_{how}_ms"]
        # kernels, profiler on (a separate run)
        kt = {k: kernel_times(ag, args.prof_updates, 10_001) for k, ag in agents.items()}
        K_keep = NCRIT * (M - DROP)
        pairs = B * NCRIT * M * K_keep
        q = kt["quantile"]
        huber_us = summed(q, ("quantile_huber_kernel",))
        row["kernels"] = {
            "quantile_target_us": summed(q, ("quantile_target_kernel",)),
            "quantile_huber_us": huber_us,
            "quantile_huber_pairs": pairs,
            "quantile_huber_pairs_per_s": pairs / (huber_us * 1e-6) if huber_us else None,
            "quantile_metrics_us": summed(q, ("quantile_metrics_kernel",)),
            "quantile_row_mean_us": summed(q, ("quantile_row_mean_kernel",)),
            "fp32_gemm_us_quantile": summed(q, GEMM_KERNELS),
            "fp32_gemm_us_scalar": summed(kt["scalar"], GEMM_KERNELS),
            "head_gemms_us": summed(q, GEMM_KERNELS) - summed(kt["scalar"], GEMM_KERNELS),
            "scalar_head_kernels_us": summed(kt["scalar"], SCALAR_HEAD_KERNELS),
            "scalar_target_and_loss_us": summed(kt["scalar"], ("sac_target_kernel", "critic_metrics_kernel",
                                                               "actor_trunc_kernel")),
            "all_us_quantile": sum(v[0] for v in q.values()),
            "all_us_scalar": sum(v[0] for v in kt["scalar"].values()),
        }
        row["kernel_table_quantile"] = {k: v for k, v in q.items()}
        row["kernel_table_scalar"] = {k: v for k, v in kt["scalar"].items()}
        print(json.dumps({k: v for k, v in row.items() if not k.endswith("rounds_ms") and not k.startswith("kernel_table")}),
              flush=True)
        result["rows"].append(row)
        del agents, variants
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- HER sample + DDPG update hot path on B200, next to the CPU port of the reference.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch: draw B positions of the HER buffer,
gather + future-relabel + sparse reward, then one DDPG update (target forward, Bellman target,
critic backward, clip, Adam, Polyak every 40th step, actor backward, clip, Adam) -- what
``DDPG.update(step)`` does in the reference (src/agent.py:1378-1404).

Workload at N=1 (BASELINE.json configs[1]): PandaPush shape (obs 18, goal 3, action 3), T=50,
k_future=4, 1M stored transitions per GPU (20 000 episodes = 4.92M deque entries), batch 256,
hidden 256 x 3 layers, synthetic data (SURVEY 8d recipe).  N>1: every rank owns its own
1M-transition episode shard and samples its local batch of 256 (weak scaling); critic and actor
gradients are averaged with NCCL between backward and optimiser phases.

One JSON line on stdout (rank 0); progress on stderr.  ``--dump-outputs DIR`` also writes what the last timed
step computed (its metrics and the weights of all four networks) as ``DIR/<name>.npy``: the inputs are seeded, so
two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import random
import sys
import threading
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "goal-conditioned-rl-framework_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "her_relabelled_transitions_per_s"   # sampled+relabelled transitions consumed by DDPG updates
UNIT = "transitions/s"
DUMP_BYTES = 60 << 20      # payload cap of --dump-outputs: with the .npy headers the files stay under 64 MB


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def positive_int(text):
    n = int(text)
    if n < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {n}")
    return n


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=1000, help="timed steps")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--hidden", type=int, default=256)
    ap.add_argument("--layers", type=int, default=3)
    ap.add_argument("--obs", type=int, default=18)
    ap.add_argument("--goal", type=int, default=3)
    ap.add_argument("--act", type=int, default=3)
    ap.add_argument("--k-future", type=int, default=4)
    ap.add_argument("--transitions", type=int, default=1_000_000, help="stored raw transitions per GPU")
    ap.add_argument("--no-sweep", action="store_true", help="skip the batch sweep / kernel rooflines")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dp", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1: average gradients over NVLink peer memory inside the captured graph (p2p) or with "
                         "NCCL all-reduce between the update phases (nccl)")
    ap.add_argument("--no-big-buffer", action="store_true", help="skip the 10M-transition sampler point")
    ap.add_argument("--huge-buffer", action="store_true",
                    help="also time the sampler on 100x the transitions (100M stored transitions, 23 GB; +1 min)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--spinup", type=int, default=80, help="extra untimed steps before the W warm-up steps")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (the 8 update metrics, the weights "
                         "and biases of actor, critic and both targets) as DIR/<name>.npy in float32; rank 0 only")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """Writes every named array as ``out_dir/<name>.npy`` in float32.  When they hold more than ``budget`` bytes in
    all, each array is cut to the same fraction of its elements (flattened), at positions drawn from a fixed seed,
    so that runs with the same arguments write the same positions."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, np.float32) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    for name, v in arrays.items():
        if total > budget:
            keep = max(1, v.size * budget // total)
            v = v.reshape(-1)[np.sort(np.random.default_rng(0).choice(v.size, keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), v)


# ------------------------------------------------------------------------------------------
# synthetic data (SURVEY 8d): obs ~ N(0,1); achieved goal = random walk, 30 % rest steps;
# desired goal ~ U(-0.15, 0.15)^3 constant per episode; actions ~ U(-1, 1); done = 0
# ------------------------------------------------------------------------------------------
def sparse_reward(ag, dg):
    d = ag - dg
    sq = d * d
    acc = sq[..., 0]
    for i in range(1, sq.shape[-1]):
        acc = acc + sq[..., i]
    return -(np.sqrt(acc) > np.float32(0.05)).astype(np.float32)


def synth(rng, E, T, O, G, A, k):
    obs = rng.standard_normal((E, T + 1, O), dtype=np.float32)
    steps = rng.normal(0, 0.02, (E, T, G)).astype(np.float32) * (rng.random((E, T, 1)) > 0.3)
    ag0 = rng.uniform(-0.15, 0.15, (E, 1, G)).astype(np.float32)
    ag = np.concatenate([ag0, ag0 + np.cumsum(steps, 1, dtype=np.float32)], 1)
    dg = np.repeat(rng.uniform(-0.15, 0.15, (E, 1, G)).astype(np.float32), T, 1)
    s = np.concatenate([obs[:, :-1], dg], -1)
    ns = np.concatenate([obs[:, 1:], dg], -1)
    a = rng.uniform(-1, 1, (E, T, A)).astype(np.float32)
    r = sparse_reward(ag[:, 1:], dg)
    d = np.zeros((E, T), np.float32)
    fut = np.zeros((E, T, max(k, 1)), np.uint8)
    for t in range(T - 1):
        fut[:, t] = rng.integers(t + 1, T, (E, max(k, 1)))
    return dict(s=s, a=a, ns=ns, r=r, d=d, ag=np.ascontiguousarray(ag[:, 1:]), fut=fut[:, :, :k] if k else fut)


def agent_config(args, max_len):
    return types.SimpleNamespace(
        hidden_dim=args.hidden, layer_count=args.layers, actor_lr=1e-3, actor_lr_min=1e-3,
        ac_scheduler_steps=1, critic_lr=1e-3, critic_lr_min=1e-3, cr_scheduler_steps=1, buffer_type="HER",
        max_len=max_len, alpha=1.0, batch_size=args.batch, gamma=0.98, ac_update_freq=1, noise_std=0.2,
        noise_clamp=0.5, policy_noise=0.0, grad_clip=10.0, beta=1.0, beta_end=1, k_future=args.k_future,
        max_eps_len=50, tau=0.05)


# ------------------------------------------------------------------------------------------
# CPU arm: the NumPy port of the reference (oracle/), eager deque buffer + DDPG update
# ------------------------------------------------------------------------------------------
def cpu_arm(args, steps, warmup, seconds=None):
    """Times sample(B) + update on the host.  The eager deque design is run at the reference's
    own cap, max_len = 1M entries (src/config/DDPG/config_ddpg_push.yaml:28); beyond that it needs
    >5 GB of Python objects."""
    from collections import deque
    from oracle import ddpg as OD
    from oracle import her as OH
    try:
        from threadpoolctl import threadpool_info
        cores = max([p.get("num_threads", 1) for p in threadpool_info()] + [1])
    except Exception:
        cores = os.cpu_count() or 1
    rng = np.random.default_rng(0)
    T, k, O, G, A = 50, args.k_future, args.obs, args.goal, args.act
    D = O + G
    max_len = 1_000_000
    E = max_len // ((T - 1) * (k + 1) + 1) + 1
    t0 = time.time()
    data = synth(rng, E, T, O, G, A, k)
    buf = OH.HERBufferOracle(max_len, 50, 1, k_future=k)
    for e in range(E):   # vectorised materialisation of apply_her's entries, then the same deque
        S, Aa, R, NS, Dn = OH.materialise_episode(data["s"][e], data["a"][e], data["ns"][e], data["r"][e],
                                                  data["d"][e], data["ag"][e], data["fut"][e], k)
        buf.buffer.extend(zip(S, Aa, NS, R[:, 0], Dn[:, 0] > 0, S[:, -G:], S[:, -G:]))
    log(f"[cpu] deque of {len(buf)} entries built in {time.time() - t0:.1f}s; BLAS threads {cores}")
    actor0, critic0 = OD.init_mlp(rng, D, args.hidden, A, args.layers), OD.init_mlp(rng, D + A, args.hidden, 1, args.layers)
    agent = OD.DDPGOracle(actor0, critic0, gamma=0.98, tau=0.05, grad_clip=10.0, actor_lr=1e-3, critic_lr=1e-3)
    random.seed(1898)
    B = args.batch

    def one(step):
        s, a, r, ns, d = buf.sample(B)
        agent.update_on_batch(step, s, a, r, ns, d)

    for i in range(warmup):
        one(i + 1)
    n, t0 = 0, time.perf_counter()
    while n < steps:
        one(warmup + n + 1)
        n += 1
        if seconds is not None and time.perf_counter() - t0 > seconds:
            break
    dt = time.perf_counter() - t0
    return dict(value=n * B / dt, unit=UNIT, cores=cores, kind="port",
                sample=f"{n} steps of sample({B}) + DDPG update (H={args.hidden}, L={args.layers}) on a "
                       f"{len(buf)}-entry eager deque (the reference's own max_len), NumPy/BLAS port of the "
                       f"reference (oracle/her.py, oracle/ddpg.py), {dt:.1f}s",
                updates_per_s=n / dt, ms_per_step=dt / n * 1e3, steps=n)


def reference_arm(args, steps, warmup, seconds=None):
    """The UNMODIFIED reference (oracle/_ref/src/{buffer,agent,model,utils}.py, vendored by oracle/make_ref.py in
    the build container): its own HERBuffer -- filled through its own push() / apply_her() up to its own cap of
    max_len = 1M entries -- and its own DDPG.update(step) = HERBuffer.sample(B) + critic_update + actor_update
    (src/agent.py:1378-1404), on the host's cores with torch's default thread count.  Returns None when
    oracle/_ref is absent (a checkout that never ran build() next to the reference)."""
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isfile(os.path.join(ref_dir, "src", "agent.py")):
        return None
    sys.path.insert(0, ref_dir)
    import torch
    import src.agent as ref_agent      # noqa: E402  (the vendored reference)
    import src.utils as ref_utils      # noqa: E402
    torch.manual_seed(1898)
    random.seed(1898)
    T, k, O, G, A, B = 50, args.k_future, args.obs, args.goal, args.act, args.batch
    D = O + G
    max_len = 1_000_000
    cfg = ref_utils.BaseAgentConfig(
        hidden_dim=args.hidden, layer_count=args.layers, actor_lr=1e-3, actor_lr_min=1e-3, ac_scheduler_steps=1,
        critic_lr=1e-3, critic_lr_min=1e-3, cr_scheduler_steps=1, buffer_type="HER", max_len=max_len, alpha=1.0,
        batch_size=B, gamma=0.98, ac_update_freq=1, noise_std=0.2, noise_clamp=0.5, policy_noise=0.0, grad_clip=10.0,
        beta=1.0, beta_end=1, k_future=k, max_eps_len=50, tau=0.05)
    ag = ref_agent.DDPG(obs_dim=D, ac_dim=A, config=cfg, weights=None, nenvs=1, gradient_step=40)
    # panda-gym's sparse reward (un-vendored dependency; the published rule, as in tests/golden/make_golden.py)
    ag.buffer.compute_reward = lambda a, b, info: -np.array(np.linalg.norm(a - b, axis=-1) > 0.05, dtype=np.float32)
    rng = np.random.default_rng(0)
    per_ep = (T - 1) * (k + 1) + 1
    E = max_len // per_ep + 1
    data = synth(rng, E, T, O, G, A, k)
    t0 = time.time()
    for e in range(E):                      # the reference's own ingest path, transition by transition
        s_t, ns_t = torch.from_numpy(data["s"][e]), torch.from_numpy(data["ns"][e])
        for t in range(T):
            ag.buffer.push(0, s_t[t], data["a"][e][t], ns_t[t], np.float64(data["r"][e][t]), bool(t == T - 1 and False),
                           data["s"][e][t][-G:], data["ag"][e][t])
    fill_s = time.time() - t0
    # torch's intra-op thread count: its default (all cores) is often SLOWER than a few threads on these small
    # GEMMs, so the baseline gets the best of {default, 8, 4, 1} -- measured here, two updates each
    best, cores = None, torch.get_num_threads()
    for nt in sorted({torch.get_num_threads(), 8, 4, 1}, reverse=True):
        if nt > (os.cpu_count() or 1):
            continue
        torch.set_num_threads(nt)
        ag.update(1)
        t0 = time.perf_counter()
        ag.update(2)
        ag.update(3)
        dt = (time.perf_counter() - t0) / 2
        if best is None or dt < best:
            best, cores = dt, nt
    torch.set_num_threads(cores)
    log(f"[reference] HERBuffer of {len(ag.buffer)} entries filled through push()/apply_her() in {fill_s:.1f}s "
        f"({len(ag.buffer) / fill_s:.0f} entries/s); torch threads {cores} (fastest of the candidates)")
    for i in range(warmup):
        ag.update(i + 1)
    n, t0 = 0, time.perf_counter()
    while n < steps:
        ag.update(warmup + n + 1)
        n += 1
        if seconds is not None and time.perf_counter() - t0 > seconds:
            break
    dt = time.perf_counter() - t0
    return dict(value=n * B / dt, unit=UNIT, cores=cores, kind="reference",
                sample=f"{n} calls of the unmodified reference DDPG.update(step) (src/agent.py:1378-1404: "
                       f"HERBuffer.sample({B}) over a {len(ag.buffer)}-entry deque + critic and actor updates, H={args.hidden}, "
                       f"L={args.layers}), {dt:.1f}s; the buffer was filled by the reference's own push()/apply_her() at "
                       f"{len(ag.buffer) / fill_s:.0f} entries/s",
                updates_per_s=n / dt, ms_per_step=dt / n * 1e3, steps=n, ingest_entries_per_s=len(ag.buffer) / fill_s)


def reference_main(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    res = reference_arm(args, args.steps, min(args.warmup, 3), seconds=90.0)
    port = None
    if res is None:                      # no vendored reference in this checkout: the NumPy port stands in
        res = cpu_arm(args, args.steps, args.warmup, seconds=120.0)
    elif not args.no_cpu:
        port = cpu_arm(args, 10 ** 9, 2, seconds=10.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": res["steps"], "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.gpus), "updates_per_s": res["updates_per_s"],
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if port is not None:
        line["cpu_port"] = {k: port[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    return {"workload": f"DDPG sample+update, PandaPush shape (obs {args.obs}, goal {args.goal}, act {args.act}), "
                        f"T=50, k_future={args.k_future}, {args.transitions} stored transitions per GPU, "
                        f"batch {args.batch} per GPU, hidden {args.hidden} x {args.layers}",
            "batch_per_gpu": args.batch, "global_batch": args.batch * world, "hidden": args.hidden,
            "layers": args.layers, "buffer_transitions_per_gpu": args.transitions,
            "parallelism": (f"dp{world} (episode-sharded buffer, gradients averaged over NVLink peer memory inside the "
                            f"captured graph)" if args.dp == "p2p" else
                            f"dp{world} (episode-sharded buffer, NCCL gradient all-reduce)") if world > 1 else "single GPU",
            "index_stream": "on-device (value) / host Mersenne-Twister random.sample (e2e)",
            "engines": "batch <= 1024: row-slab fused fp32 kernels; >= 2048: tcgen05 3xTF32 hidden layers (sweep)",
            "l2": "flushed between timed steps (256 MiB write); buffer (224 MB) larger than L2"}


# ------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
    NOTE = {"sw_power_cap": 0x4}

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.times, self.reasons, self.stop_flag = [], [], set(), False
        self.max_mhz, self.ok = None, False
        self.armed, self.window = False, [None, None]   # throttle reasons / clocks are reported for the armed window
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:   # noqa: BLE001
            log(f"[clocks] NVML unavailable: {e}")

    def sample(self):
        nv = self.nv
        self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        self.times.append(time.perf_counter())
        try:
            mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:   # noqa: BLE001
            mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        if self.armed:
            for name, bit in {**self.BAD, **self.NOTE}.items():
                if mask & bit:
                    self.reasons.add(name)

    def run(self):
        while self.ok and not self.stop_flag:
            try:
                self.sample()
            except Exception:   # noqa: BLE001
                break
            time.sleep(self.period)

    def arm(self):
        """Start of the window the clocks line describes (the thread itself was started long before, so that its
        start-up cannot disturb the timed steps)."""
        self.armed, self.window[0] = True, time.perf_counter()

    def disarm(self):
        self.armed, self.window[1] = False, time.perf_counter()

    def result(self):
        self.stop_flag = True
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml_unavailable"]}
        if not self.samples:
            self.sample()
        t0, t1 = self.window
        inwin = [m for m, t in zip(self.samples, self.times) if t0 is not None and t0 <= t <= (t1 or t)]
        use = inwin if len(inwin) >= 3 else self.samples
        return {"sm_mhz": float(np.median(use)), "sm_max_mhz": float(self.max_mhz),
                "reasons": sorted(self.reasons), "samples": len(use),
                "window": "timed steps + 0.3 s of the same load" if use is inwin else "whole run (window too short)"}



# ------------------------------------------------------------------------------------------
# data-parallel evidence (N > 1): replicas identical, and N ranks == 1 rank on the concatenated batch
# ------------------------------------------------------------------------------------------
def dp_parity(args, local, rank, world, dp_mode, updates=4):
    """Outside every timed region: `updates` DDPG updates on fixed per-rank batches through the data-parallel
    path that is being benchmarked; every rank hashes all four networks (replicas must be bit-identical); rank 0
    repeats the run with ONE agent (fp32 FFMA engine) on the concatenated batches and reports the largest
    deviation, relative to the largest weight of the tensor, and whether every tensor is inside the tolerance the
    parity tests use for post-update weights (SURVEY 8e parity rule)."""
    import hashlib

    import torch
    import torch.distributed as dist
    from gcrl_b200 import DDPG
    O, G, A, B = args.obs, args.goal, args.act, args.batch
    D = O + G

    def batch_of(r, i):
        g = np.random.default_rng(5000 + 97 * i + r)
        s = g.standard_normal((B, D)).astype(np.float32)
        ns = (s + 0.1 * g.standard_normal((B, D))).astype(np.float32)
        a = g.uniform(-1, 1, (B, A)).astype(np.float32)
        rew = -(g.random((B, 1)) > 0.3).astype(np.float32)
        d = (g.random((B, 1)) < 0.1).astype(np.float32)
        return s, a, rew, ns, d

    def nets(ag):
        return [w for net in (ag.actor, ag.critic, ag.target_actor, ag.target_critic) for pair in net.layers() for w in pair]

    def fresh(max_batch, precision=1):
        torch.manual_seed(777)
        return DDPG(D, A, agent_config(args, 1000), None, 1, 40, device=local, max_batch=max_batch, precision=precision)

    steps = list(range(38, 38 + updates))            # crosses the step-40 Polyak update
    ag = fresh(B)
    if dp_mode == "p2p":
        ag.enable_peer_data_parallel()
    else:
        ag.enable_data_parallel()
    for i, st in enumerate(steps):
        info = ag.update(st, batch=tuple(torch.from_numpy(x).cuda(local) for x in batch_of(rank, i)))
    mine = nets(ag)
    digest = hashlib.sha1(b"".join(np.ascontiguousarray(w).tobytes() for w in mine)).hexdigest()
    digests = [None] * world
    dist.all_gather_object(digests, digest)
    metrics = [None] * world
    dist.all_gather_object(metrics, [float(x) for x in info])
    out = {"replicas_identical": len(set(digests)) == 1, "updates": updates, "batch_per_rank": B, "path": dp_mode,
           "metrics_identical": all(m == metrics[0] for m in metrics)}
    if rank == 0:
        one = fresh(world * B, precision=0)
        for i, st in enumerate(steps):
            cat = [np.concatenate([batch_of(r, i)[j] for r in range(world)]) for j in range(5)]
            one.update(st, batch=tuple(torch.from_numpy(x).cuda(local) for x in cat))
        ref = nets(one)
        rel = max(float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-30)) for a, b in zip(mine, ref))
        out["max_rel_vs_concat"] = rel
        # the parity tests' own rule (tests/helpers.py::weights_close): per tensor |w - ref| <= 1e-5 max|ref| + 5e-3 lr n
        # for all but 2e-4 of the elements, those inside Adam's hard bound 2 lr n -- restated here so that the bench
        # does not import the test tree; the old flat 1e-4 on max_rel is kept in the line for comparison
        lr, worst_used, within = 1e-3, 0.0, True
        for a, b in zip(mine, ref):
            err = np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64))
            tol = 1e-5 * float(np.max(np.abs(b))) + 5e-3 * lr * updates
            worst_used = max(worst_used, float(np.max(err)) / tol)
            within = within and float(np.max(err)) <= 2.0 * lr * updates + 1e-5 * float(np.max(np.abs(b))) \
                and int(np.count_nonzero(err > tol)) <= 2e-4 * err.size
        out["tolerance"] = "weights_close: 1e-5 max|w| + 5e-3 lr n per tensor (<= 2e-4 of the elements up to Adam's bound 2 lr n)"
        out["worst_fraction_of_tolerance"] = worst_used
        out["max_rel_below_1e-4"] = bool(rel < 1e-4)
        out["ok"] = bool(out["replicas_identical"] and within)
        del one
    del ag
    torch.cuda.synchronize()
    return out


# ------------------------------------------------------------------------------------------
# the other BASELINE configs, short runs (also at N > 1, so that the scaling record carries them)
# ------------------------------------------------------------------------------------------
def extra_configs(args, local, rank, world, dp_mode, flush, stream, peaks):
    import types as _t

    import torch
    import torch.distributed as dist
    from gcrl_b200 import DDPG, HERBuffer, TQCAgent
    from gcrl_b200._lib import check, lib, vp
    dev = torch.device("cuda", local)
    sp = vp(stream.cuda_stream)
    out = {}
    T = 50

    def maxr(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def fill(buf, data, E):
        for e in range(E):
            buf.push_episode(data["s"][e], data["a"][e], data["ns"][e], data["r"][e], data["d"][e], data["ag"][e], data["fut"][e])

    def timed(fn, n, align=None):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        for i, (e0, e1) in enumerate(evs):
            flush.fill_(i & 0xFF)
            if align is not None:
                align()
            e0.record(stream)
            fn(i)
            e1.record(stream)
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs) / n

    # ---- configs[2]: DDPG, PickAndPlace shape (obs 19 + goal 3, act 4, H 256 x 3, k_future 8), GLOBAL batch 65536
    try:
        O, G, A, k, H, L = 19, 3, 4, 8, 256, 3
        gb = 65536
        Bl = gb // world
        E = 2000
        rng = np.random.default_rng(3000 + rank)
        data = synth(rng, E, T, O, G, A, k)
        a2 = _t.SimpleNamespace(**vars(args))
        a2.obs, a2.goal, a2.act, a2.k_future, a2.hidden, a2.layers, a2.batch = O, G, A, k, H, L, Bl
        torch.manual_seed(1898)
        ag = DDPG(O + G, A, agent_config(a2, E * ((T - 1) * (k + 1) + 1)), None, 1, 40, index_source="device",
                  device=local, max_batch=Bl, seed=4000 + rank)
        fill(ag.buffer, data, E)
        align = None
        if world > 1:
            if dp_mode == "p2p":
                ag.enable_peer_data_parallel()
                align = ag.peer_barrier
            else:
                ag.enable_data_parallel()
        st = [1]

        def one(_i):
            ag._run_update(st[0], sync=False)
            st[0] += 1
        for _ in range(12):
            one(0)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms_k = maxr(timed(one, 10, align))
        amac = (O + G) * H + (L - 1) * H * H + H * A
        cmac = (O + G + A) * H + (L - 1) * H * H + H
        flops = 2.0 * (4 * amac + 6 * cmac) * gb
        info = ag.read_metrics()
        out["ddpg_pickplace_global_B65536"] = {
            "workload": f"DDPG sample+update, PickAndPlace shape (obs {O}, goal {G}, act {A}), k_future {k}, hidden {H} x {L}, "
                        f"global batch {gb} = {Bl} per GPU x {world}, {E * T} stored transitions per GPU",
            "ms_per_step": ms_k, "transitions_per_s": gb / (ms_k * 1e-3), "updates_per_s": 1e3 / ms_k,
            "update_tflops": flops / (ms_k * 1e-3) / 1e12, "scaling": "strong", "path": dp_mode if world > 1 else "single GPU",
            "engine": "tcgen05 3xTF32" if Bl >= 2048 else "row-slab fp32", "finite": bool(all(np.isfinite(float(x)) for x in info))}
        del ag, data
        torch.cuda.empty_cache()
    except Exception as e:   # noqa: BLE001
        out["ddpg_pickplace_global_B65536"] = {"error": repr(e)}

    # ---- configs[3]: TQC, Slide shape (= Push: obs 18 + goal 3, act 3), 5 critics / drop 2, batch 512 per GPU
    try:
        O, G, A, k, H, L, Bl = 18, 3, 3, 4, 512, 3, 512
        E = 2000
        rng = np.random.default_rng(6000 + rank)
        data = synth(rng, E, T, O, G, A, k)
        a3 = _t.SimpleNamespace(**vars(args))
        a3.obs, a3.goal, a3.act, a3.k_future, a3.hidden, a3.layers, a3.batch = O, G, A, k, H, L, Bl
        cfg = agent_config(a3, E * ((T - 1) * (k + 1) + 1))
        cfg.alpha_lr, cfg.alpha_min, cfg.alpha_min_steps, cfg.grad_clip, cfg.gamma = 3e-4, 3e-4, 1, 5.0, 0.95
        torch.manual_seed(1898)
        def time_tqc(sync_bn):
            torch.manual_seed(1898)
            tq = TQCAgent(O + G, A, cfg, None, 1, 40, index_source="device", device=local)
            fill(tq.buffer, data, E)
            if world > 1:
                tq.enable_data_parallel(sync_bn=sync_bn)
            for i in range(6):
                tq.update(i + 1)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            n = 30
            t0 = time.perf_counter()
            for i in range(n):
                info = tq.update(7 + i)
            torch.cuda.synchronize()
            ms = maxr((time.perf_counter() - t0) * 1e3 / n)
            fin = bool(all(np.isfinite(float(np.mean(x))) for x in info))
            del tq
            return ms, fin
        ms_k, fin = time_tqc(True)
        out["tqc_slide_B512_per_gpu"] = {
            "workload": f"TQCAgent.update (5 scalar critics, drop top 2, learned alpha), Slide shape (obs {O}, goal {G}, act {A}), "
                        f"hidden {H} x {L} (config_tqc_push.yaml), batch {Bl} per GPU, metric read-back every update",
            "ms_per_update": ms_k, "updates_per_s": 1e3 / ms_k, "transitions_per_s": world * Bl / (ms_k * 1e-3),
            "scaling": "weak",
            "path": ("NCCL between graph segments: BatchNorm statistics over the global batch (sync-BN, "
                     f"{3 * L} all-gathers) + 2 gradient averages per update = one rank on the concatenated batch"
                     if world > 1 else "single GPU"),
            "finite": fin}
        if world > 1:
            ms_l, fin_l = time_tqc(False)
            out["tqc_slide_B512_per_gpu"]["local_batchnorm_statistics"] = {
                "ms_per_update": ms_l, "transitions_per_s": world * Bl / (ms_l * 1e-3), "finite": fin_l,
                "path": "enable_data_parallel(sync_bn=False): 4 phases, 3 NCCL all-reduces per update, running "
                        "statistics averaged; close to, not equal to, the single-rank result"}
        del data
        torch.cuda.empty_cache()
    except Exception as e:   # noqa: BLE001
        out["tqc_slide_B512_per_gpu"] = {"error": repr(e)}

    # ---- configs[4]: the sampler on a 10M-transition shard per GPU (no collective: shards are independent);
    # at N = 1 the `rooflines` section already carries these points (her_sample_kernel_B*_buffer10M)
    try:
        if world == 1:
            raise StopIteration
        O, G, A, k = args.obs, args.goal, args.act, args.k_future
        D = O + G
        E = 20000
        rng = np.random.default_rng(8000 + rank)
        data = synth(rng, E, T, O, G, A, k)
        per_ep = (T - 1) * (k + 1) + 1
        big = HERBuffer(10 * E * per_ep, 50, 1, k_future=k, index_source="device", seed=7 + rank, device=local)
        for _rep in range(10):
            fill(big, data, E)
        torch.cuda.synchronize()
        alg_bytes = 4 * (2 * O + A + 2 * G) + 5 + 4 * (2 * D + A + 2)
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        rec = {}
        for batch in (256, 65536):
            outs = [torch.empty((batch, w), dtype=torch.float32, device=dev) for w in (D, A, 1, D, 1)]
            ptrs = [vp(o.data_ptr()) for o in outs]

            def one(_i):
                check(lib.gcrl_her_sample(big.handle, batch, None, *ptrs, None, sp))
            for _ in range(5):
                one(0)
            if world > 1:
                dist.barrier()
            ms_k = maxr(timed(one, 30))
            ach = batch * alg_bytes / (ms_k * 1e-3) / 1e9
            rec[f"B{batch}"] = {"ms_per_launch": ms_k, "transitions_per_s": world * batch / (ms_k * 1e-3),
                                "hbm_gbs_per_gpu": ach, "hbm_frac_per_gpu": ach / hbm_peak}
        out["sampler_10M_per_gpu"] = {
            "workload": f"HER sample + relabel + reward on {len(big)} deque entries (10M stored transitions) per GPU, "
                        f"Push shape, every GPU samples its own shard", "scaling": "weak", **rec}
        del big, data
        torch.cuda.empty_cache()
    except StopIteration:
        pass
    except Exception as e:   # noqa: BLE001
        out["sampler_10M_per_gpu"] = {"error": repr(e)}
    return out


def normaliser_rooflines(local, flush, stream, hbm_peak, dim=19):
    """RunningNormalizer.update / normalize (src/utils.py:75-98) on device-resident float32 batches [n, dim]:
    update reads the batch once (4 n dim bytes), normalize reads it and writes float32 (8 n dim bytes)."""
    import ctypes as C

    import torch
    from gcrl_b200 import RunningNormalizer
    from gcrl_b200._lib import check, lib, vp
    dev = torch.device("cuda", local)
    sp = vp(stream.cuda_stream)
    out = {}
    nz = RunningNormalizer(dim, device=local)
    for n in (64, 100_000, 1_000_000):
        x = torch.randn(n, dim, device=dev)
        y = torch.empty(n, dim, device=dev)
        for name, fn, nbytes in (
                ("norm_update", lambda: check(lib.gcrl_norm_update_dev(nz._h, vp(x.data_ptr()), n, 0, sp)), 4 * n * dim),
                ("norm_apply", lambda: check(lib.gcrl_norm_apply_dev_f32(nz._h, vp(x.data_ptr()), n, 0, vp(y.data_ptr()), dim, 0, sp)),
                 8 * n * dim)):
            for _ in range(3):
                fn()
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(20)]
            for i, (a0, a1) in enumerate(evs):
                flush.fill_(i & 0xFF)
                a0.record(stream)
                fn()
                a1.record(stream)
            torch.cuda.synchronize()
            ms_k = sum(a.elapsed_time(b) for a, b in evs) / len(evs)
            ach = nbytes / (ms_k * 1e-3) / 1e9
            out[f"{name}_n{n}_dim{dim}"] = {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                                            "frac": ach / hbm_peak, "traffic": None, "ms_per_launch": ms_k,
                                            "algorithmic_bytes_per_launch": nbytes, "rows_per_s": n / (ms_k * 1e-3)}
    return out


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
def gpu_main(args):
    import ctypes as C

    import torch
    import torch.distributed as dist

    import gcrl_b200
    from gcrl_b200 import DDPG, _lib
    from gcrl_b200._lib import check, lib, vp

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:   # noqa: BLE001
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"

    T, k, O, G, A, B = 50, args.k_future, args.obs, args.goal, args.act, args.batch
    D = O + G
    E = args.transitions // T
    per_ep = (T - 1) * (k + 1) + 1
    max_len = E * per_ep
    rng = np.random.default_rng(1000 + rank)            # every rank owns a different episode shard
    t0 = time.time()
    data = synth(rng, E, T, O, G, A, k)
    launches0 = int(lib.gcrl_kernel_launches())

    def make_agent(index_source, max_batch):
        torch.manual_seed(1898)                          # identical initial weights on every rank
        ag = DDPG(D, A, agent_config(args, max_len), None, 1, 40, index_source=index_source, device=local,
                  max_batch=max_batch, seed=1898 + rank)
        for e in range(E):
            ag.buffer.push_episode(data["s"][e], data["a"][e], data["ns"][e], data["r"][e], data["d"][e],
                                   data["ag"][e], data["fut"][e])
        return ag

    sweep_batches = [] if (args.no_sweep or world > 1) else [1024, 4096, 16384, 65536]
    agent = make_agent("device", max(B, max(sweep_batches + [B])))
    torch.cuda.synchronize()
    log(f"[rank {rank}] {E} episodes / {len(agent.buffer)} entries committed in {time.time() - t0:.1f}s")
    if world > 1:
        if args.dp == "p2p":
            try:
                agent.enable_peer_data_parallel()
            except Exception as e:   # noqa: BLE001  (every rank raises together, see enable_peer_data_parallel)
                log(f"[rank {rank}] peer-memory averaging unavailable ({e}); falling back to NCCL all-reduce")
                agent2 = make_agent("device", max(B, max(sweep_batches + [B])))   # fresh handle without the mapping
                agent = agent2
                args.dp = "nccl"
                agent.enable_data_parallel()
        else:
            agent.enable_data_parallel()
    parity = None
    if world > 1:
        try:
            parity = dp_parity(args, local, rank, world, args.dp)
            log(f"[rank {rank}] dp_parity: {parity}")
        except Exception as e:   # noqa: BLE001
            parity = {"error": repr(e)}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)
    sp = vp(stream.cuda_stream)
    clocks = ClockSampler(local)     # started here, long before the timed window (arm() marks the window)
    clocks.start()

    def device_step(step, batch=B, ag=None):
        """Async step on the device index stream, no host read-back (what `value` times)."""
        ag = ag or agent
        ag.batch_size = batch
        ag._run_update(step, sync=False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_steps(n, first_step, batch=B, do_flush=True, ag=None):
        """n steps, each bracketed by CUDA events on the launching stream; returns the per-step ms.  With the
        peer-memory path the ranks are re-aligned by one flag barrier AFTER the L2 flush and BEFORE the start
        event: the (untimed) 256 MiB flush finishes at slightly different times on every rank, and without the
        alignment that skew would be charged to the step through its first gradient barrier."""
        ag = ag or agent
        align = world > 1 and getattr(ag, "_peer_dp", None) is not None
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        for i, (e0, e1) in enumerate(evs):
            if do_flush:
                flush.fill_(i & 0xFF)
            if align:
                ag.peer_barrier()
            e0.record(stream)
            device_step(first_step + i, batch, ag)
            e1.record(stream)
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in evs]    # ms

    def over_ranks(per_step):
        """max over ranks of the summed time (the contract's number) + where the time went per rank and step."""
        t = torch.tensor(per_step, dtype=torch.float64, device=dev)
        if world > 1:
            allt = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(allt, t)
            allt = torch.stack(allt).cpu().numpy()
        else:
            allt = t.cpu().numpy()[None]
        sums = allt.sum(1)
        r, i = np.unravel_index(int(np.argmax(allt)), allt.shape)
        mx = allt.max(0)
        keep = 200                                     # long runs: the first steps + the distribution, not 3 x K numbers
        detail = {"rank0": [round(float(x), 4) for x in allt[0][:keep]],
                  "max_over_ranks": [round(float(x), 4) for x in mx[:keep]],
                  "sum_ms_per_rank": [round(float(x), 4) for x in sums],
                  "slowest": {"rank": int(r), "step": int(i), "ms": round(float(allt[r, i]), 4)},
                  "median_ms": round(float(np.median(allt)), 4),
                  "max_over_ranks_p50_p99_max": [round(float(np.median(mx)), 4), round(float(np.quantile(mx, 0.99)), 4),
                                                 round(float(mx.max()), 4)],
                  "steps_listed": int(min(keep, allt.shape[1]))}
        return float(sums.max()), detail

    # ---- warm-up (graph capture for both flag sets, clocks ramp), then the timed region ----
    step = 1
    for _ in range(max(args.warmup, 3) + args.spinup):
        device_step(step)
        step += 1
    for _ in timed_steps(3, step):        # the timed loop's own code path (events, flush, alignment), untimed
        pass
    step += 3
    barrier()
    clocks.arm()
    l0 = int(lib.gcrl_kernel_launches())
    per_step = timed_steps(args.steps, step)
    step += args.steps
    launches = int(lib.gcrl_kernel_launches()) - l0
    barrier()
    outputs = None
    if args.dump_outputs and rank == 0:
        # copied to the host before any later step changes the weights; written to disk after the measurements
        outputs = {"metrics": np.array(agent.read_metrics(), np.float32)}
        for tag in ("actor", "critic", "target_actor", "target_critic"):
            for i, (w, b) in enumerate(getattr(agent, tag).layers()):
                outputs[f"{tag}.{i}.weight"], outputs[f"{tag}.{i}.bias"] = w, b
    # keep the sampler alive over a short loaded stretch so that short runs still record clocks
    t_end = time.time() + 0.3
    while time.time() < t_end:
        device_step(step)
        step += 1
    torch.cuda.synchronize()
    clocks.disarm()
    clk = clocks.result()
    ms, per_step_detail = over_ranks(per_step)
    value = world * B * args.steps / (ms * 1e-3)
    agent.read_metrics()           # (outside the timed region) surfaces a data-parallel watchdog error right here
    log(f"[rank {rank}] timed steps done: {ms / args.steps:.4f} ms per step")

    # back-to-back (no flush, graph replays pipelined): the production regime, reported beside `value`
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for i in range(args.steps):
        device_step(step + i)
    e1.record(stream)
    torch.cuda.synchronize()
    step += args.steps
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_b2b = float(t.item())
    agent.read_metrics()
    log(f"[rank {rank}] back-to-back steps done: {ms_b2b / args.steps:.4f} ms per step")

    # ---- e2e: the public API call a user makes -- agent.update(step) with the reference's host
    # Mersenne-Twister index stream (H2D of the positions from pinned memory), the 8-float metric
    # read-back every step (D2H), and the ingest of 16 fresh episodes every 40 updates
    # (max_episode / gradient_step of config_ddpg_push.yaml) ----
    agent.index_source = "host"
    agent.buffer.index_source = "host"
    agent.batch_size = B
    random.seed(1898 + rank)
    row_bytes = 4 * (2 * D + A + 2 + G) + k
    ep_bytes = 64 + T * (row_bytes + 16)
    h2d = B * 8 + 32 + 16 * ep_bytes / 40.0
    d2h = 32

    def e2e_step(i):
        if i % 40 == 0:
            for e in range(16):
                j = (i // 40 * 16 + e) % E
                agent.buffer.push_episode(data["s"][j], data["a"][j], data["ns"][j], data["r"][j], data["d"][j],
                                          data["ag"][j], None)     # future offsets drawn by random.randint
        return agent.update(step + i)

    for i in range(max(args.warmup, 3)):
        e2e_step(i)
    n_e2e = max(40, min(args.steps, 400))
    barrier()
    e0.record(stream)
    w0 = time.perf_counter()
    for i in range(n_e2e):
        info = e2e_step(i)
    e1.record(stream)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - w0) * 1e3
    step += n_e2e
    t = torch.tensor([max(e0.elapsed_time(e1), wall)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_e2e = float(t.item())
    e2e_value = world * B * n_e2e / (ms_e2e * 1e-3)
    assert all(np.isfinite(float(x)) for x in info), info

    # the same public call with index_source="device" (positions and future offsets drawn on the GPU instead of
    # mirroring the interpreter's Mersenne-Twister stream): what the host-side stream emulation costs
    agent.index_source = "device"
    agent.buffer.index_source = "device"
    for i in range(3):
        e2e_step(i)
    barrier()
    w0 = time.perf_counter()
    for i in range(n_e2e):
        info = e2e_step(i)
    torch.cuda.synchronize()
    ms_e2e_dev = (time.perf_counter() - w0) * 1e3
    step += n_e2e
    agent.index_source = "host"
    agent.buffer.index_source = "host"

    # ---- kernel rooflines (rank 0, N=1): the HER sampler alone, CUDA events on its stream ----
    agent.index_source = "device"
    agent.buffer.index_source = "device"
    alg_bytes = 4 * (2 * O + A + 2 * G) + 5 + 4 * (2 * D + A + 2)      # SURVEY 8d: 373 B for Push
    rooflines = {}

    def time_sampler(batch, iters):
        outs = [torch.empty((batch, w), dtype=torch.float32, device=dev) for w in (D, A, 1, D, 1)]
        ptrs = [vp(o.data_ptr()) for o in outs]
        for _ in range(5):
            check(lib.gcrl_her_sample(agent.buffer.handle, batch, None, *ptrs, None, sp))
        tot = 0.0
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
        for i, (a0, a1) in enumerate(evs):
            flush.fill_(i & 0xFF)
            a0.record(stream)
            check(lib.gcrl_her_sample(agent.buffer.handle, batch, None, *ptrs, None, sp))
            a1.record(stream)
        torch.cuda.synchronize()
        tot = sum(a.elapsed_time(b) for a, b in evs) / iters
        return tot

    if rank == 0:
        # 1 048 576 is beyond BASELINE's sweep: it shows the sampler's bandwidth once launch + dependent-gather
        # latency (~16 us) is amortised
        for batch in [B] + sweep_batches + ([1 << 20] if sweep_batches else []):
            ms_k = time_sampler(batch, 50 if batch <= 65536 else 20)
            ach = batch * alg_bytes / (ms_k * 1e-3) / 1e9
            # DRAM bytes per launch from `ncu --set full` at the bench shape (profiles/r02_sampler_*_ncu_full_raw.csv:
            # dram__bytes_read.sum + dram__bytes_write.sum; 208-byte rows, 16-byte goal rows and 32-byte bucket
            # records against 64-byte DRAM bursts, the writes of the small batches are absorbed by L2)
            ncu_traffic = {65536: 27.69e6 + 0.06e6, 1 << 20: 304.31e6 + 145.9e6}   # profiles/r02_sampler_*_ncu_full_raw.csv
            rooflines[f"her_sample_kernel_B{batch}"] = {
                "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                "traffic": ncu_traffic.get(batch) if (O, G, A, k) == (18, 3, 3, 4) else None,
                "ms_per_launch": ms_k, "algorithmic_bytes_per_transition": alg_bytes,
                "transitions_per_s": batch / (ms_k * 1e-3)}
    # BASELINE configs[4]: the sampler on a 10x larger buffer (10M stored transitions = 49.2M deque entries,
    # 2.2 GB of packed rows, far beyond the 126 MB L2): the same 20 000 synthetic episodes committed 10 times
    for mult in ([10] if not args.no_big_buffer else []) + ([100] if args.huge_buffer else []):
        if not (rank == 0 and sweep_batches):
            break
        try:
            from gcrl_b200 import HERBuffer
            big = HERBuffer(mult * max_len, 50, 1, k_future=k, index_source="device", seed=7, device=local)
            t0 = time.time()
            for rep in range(mult):
                for e in range(E):
                    big.push_episode(data["s"][e], data["a"][e], data["ns"][e], data["r"][e], data["d"][e],
                                     data["ag"][e], data["fut"][e])
            torch.cuda.synchronize()
            log(f"[big buffer] {len(big)} entries committed in {time.time() - t0:.1f}s")
            for batch in (256, 65536) + ((1 << 20,) if mult >= 100 else ()):
                outs = [torch.empty((batch, w), dtype=torch.float32, device=dev) for w in (D, A, 1, D, 1)]
                ptrs = [vp(o.data_ptr()) for o in outs]
                for _ in range(5):
                    check(lib.gcrl_her_sample(big.handle, batch, None, *ptrs, None, sp))
                evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(50)]
                for i, (a0, a1) in enumerate(evs):
                    flush.fill_(i & 0xFF)
                    a0.record(stream)
                    check(lib.gcrl_her_sample(big.handle, batch, None, *ptrs, None, sp))
                    a1.record(stream)
                torch.cuda.synchronize()
                ms_k = sum(a.elapsed_time(b) for a, b in evs) / len(evs)
                ach = batch * alg_bytes / (ms_k * 1e-3) / 1e9
                rooflines[f"her_sample_kernel_B{batch}_buffer{mult * args.transitions // 1000000}M"] = {
                    "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                    "traffic": None, "ms_per_launch": ms_k, "algorithmic_bytes_per_transition": alg_bytes,
                    "transitions_per_s": batch / (ms_k * 1e-3), "buffer_transitions": mult * args.transitions}
            del big, outs
            torch.cuda.empty_cache()
        except Exception as e:   # noqa: BLE001
            log(f"[big buffer] skipped: {e}")

    # the dominant kernel of the step at the headline batch: the critic-phase row-slab kernel
    # (fp32 FFMA by design below 2048 rows; tensor cores take the hidden layers above that)
    Hh, Ll = args.hidden, args.layers
    amac = D * Hh + (Ll - 1) * Hh * Hh + Hh * A
    cmac = (D + A) * Hh + (Ll - 1) * Hh * Hh + Hh
    bf16_peak = float(peaks.get("bf16_tflops", 2250.0))
    if rank == 0:
        try:
            msk = C.c_float()
            check(lib.gcrl_agent_time_critic_kernel(agent._h, B, 200, C.byref(msk), sp))
            # algorithmic flops per launch: target actor + target critic + critic forward, critic input
            # gradients through the (L - 1) hidden layers
            fl = 2.0 * B * (amac + 2 * cmac + (Ll - 1) * Hh * Hh + Hh)
            ach = fl / (msk.value * 1e-3) / 1e12
            # DRAM bytes per launch from the `ncu --set full` capture of this kernel at the bench shape
            # (profiles/r02_update_B256_ncu_full_raw.csv, fused_critic_kernel<2,0,0>: dram__bytes_read.sum 6.71 MB +
            # write 0.01 MB: the three networks (1.65 MB) through a cold L2 under ncu, plus the in-kernel row gather)
            traffic = 6.72e6 if (B, Hh, Ll, D, A) == (256, 256, 3, 21, 3) else None
            sm_hz = float(clk.get("sm_mhz") or peaks.get("sm_max_mhz", 1965.0)) * 1e6
            fp32_peak = 148 * 128 * 2 * sm_hz / 1e12
            # what actually bounds the row-slab kernels (profiles/README.md, round 2): every CTA streams ALL the
            # weights of the phase through its SM's unified L1 / shared-memory array, which moves 128 B per clock and
            # sees every byte twice (fill + read): a 256 x 256 fp32 layer cannot take less than 2.1 us per SM,
            # whatever the load path (per-thread LDG, cp.async.bulk ring, software pipelining all measure 2.1-2.2 us)
            wbytes = 4.0 * (amac + 2 * cmac + (Ll - 1) * Hh * Hh)
            port_ms = 2.0 * wbytes / (128.0 * sm_hz) * 1e3
            rooflines[f"fused_critic_kernel_B{B}"] = {
                "bound": "tensor", "achieved": ach, "peak": bf16_peak, "unit": "TFLOP/s", "frac": ach / bf16_peak,
                "traffic": traffic, "ms_per_launch": msk.value, "algorithmic_flops_per_launch": fl,
                "pipe": "fp32 FFMA (no MMA is issued below 2048 rows; `bound`/`peak` follow the contract's bf16 "
                        "tensor denominator, the fractions below are the honest ones)",
                "frac_fp32_pipe": ach / fp32_peak, "fp32_peak_tflops": fp32_peak,
                "sram_port_bound_ms": port_ms, "frac_sram_port": port_ms / msk.value,
                "note": "row-slab kernel: each of the 128 CTAs carries 2 batch rows through every layer of the phase; "
                        "bound by the per-SM L1/shared-memory port (every weight byte crosses it twice), not by "
                        "FMA issue or HBM -- the tensor-core path serves batches >= 2048"}
        except Exception as e:   # noqa: BLE001
            log(f"[roofline] critic kernel timing skipped: {e}")
        if sweep_batches:
            Mt = 65536
            xt = torch.randn(Mt, Hh, device=dev)
            wt = torch.randn(Hh, Hh, device=dev) / Hh ** 0.5
            bt = torch.zeros(Hh, device=dev)
            yt = torch.empty(Mt, Hh, device=dev)

            whi, wlo = torch.empty_like(wt), torch.empty_like(wt)
            check(lib.gcrl_split_tf32(local, vp(wt.data_ptr()), vp(whi.data_ptr()), vp(wlo.data_ptr()), wt.numel(), sp))

            def dense(engine):
                if engine == 2:      # what the agents call: the weight operand pre-split once per optimiser step
                    check(lib.gcrl_dense_layer_presplit(local, 0, Mt, Hh, Hh, vp(xt.data_ptr()), Hh, vp(whi.data_ptr()),
                                                        vp(wlo.data_ptr()), Hh, vp(bt.data_ptr()), None, 0,
                                                        vp(yt.data_ptr()), Hh, sp))
                else:
                    check(lib.gcrl_dense_layer(local, engine, 0, Mt, Hh, Hh, vp(xt.data_ptr()), Hh, vp(wt.data_ptr()), Hh,
                                               vp(bt.data_ptr()), None, 0, vp(yt.data_ptr()), Hh, sp))
            for engine, name in ((2, "tc_dense_kernel"), (1, "tc_dense_kernel_split_in_kernel"), (0, "gemm_kernel_fp32")):
                try:
                    for _ in range(3):
                        dense(engine)
                    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(20)]
                    for i, (a0, a1) in enumerate(evs):
                        flush.fill_(i & 0xFF)
                        a0.record(stream)
                        dense(engine)
                        a1.record(stream)
                    torch.cuda.synchronize()
                    ms_k = sum(a.elapsed_time(b) for a, b in evs) / len(evs)
                    fl = 2.0 * Mt * Hh * Hh
                    ach = fl / (ms_k * 1e-3) / 1e12
                    rooflines[f"{name}_M{Mt}_H{Hh}"] = {
                        "bound": "tensor", "achieved": ach, "peak": bf16_peak, "unit": "TFLOP/s", "frac": ach / bf16_peak,
                        "traffic": (83.8e6 if (engine >= 1 and Hh == 256) else None),   # ncu: 67.4 MB read + 16.4 MB written (r01e; the pair kernel: 67.7 + 16.0, gpurun tc_pair_ncu)
                        "ms_per_launch": ms_k, "algorithmic_flops_per_launch": fl,
                        "tensor_pipe_tflops": (3.0 * ach if engine >= 1 else None),
                        "tensor_pipe_frac_of_tf32_rate": (3.0 * ach / (0.5 * bf16_peak) if engine >= 1 else None),
                        "note": ("tcgen05 kind::tf32, 3 MMAs per product (hi/lo split) for fp32 accuracy: tensor-pipe "
                                 "work is 3x the algorithmic flops; the TF32 rate is half the measured bf16 peak; " +
                                 ("weights pre-split once per optimiser step (the agents' path): at this size the CTA-pair "
                                  "kernel (cta_group::2, 256 x 256 tiles, half the weight tile per SM)" if engine == 2 else
                                  "both operands split in shared memory (round-1 scheme, for comparison)") if engine >= 1 else
                                 "fp32 FFMA tiles (the precision-0 path), for comparison")}
                except Exception as e:   # noqa: BLE001
                    log(f"[roofline] dense layer engine {engine} skipped: {e}")
            del xt, wt, bt, yt, whi, wlo

    sweep = {}
    for batch in sweep_batches:
        for _ in range(45):
            device_step(step, batch)
            step += 1
        n = max(20, min(200, args.steps))
        ms_s = sum(timed_steps(n, step, batch))
        step += n
        flops = 2.0 * (4 * (D * args.hidden + (args.layers - 1) * args.hidden ** 2 + args.hidden * A)
                       + 6 * ((D + A) * args.hidden + (args.layers - 1) * args.hidden ** 2 + args.hidden)) * batch
        sweep[f"B{batch}"] = {"ms_per_step": ms_s / n, "transitions_per_s": batch * n / (ms_s * 1e-3),
                              "updates_per_s": n / (ms_s * 1e-3), "update_tflops": flops / (ms_s / n * 1e-3) / 1e12}

    extra = {}
    if not args.no_sweep:
        extra = extra_configs(args, local, rank, world, args.dp, flush, stream, peaks)
    if rank == 0 and not args.no_sweep:
        try:
            rooflines.update(normaliser_rooflines(local, flush, stream, hbm_peak))
        except Exception as e:   # noqa: BLE001
            log(f"[roofline] normaliser timing skipped: {e}")
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            cpu = reference_arm(args, 10 ** 9, 2, seconds=args.cpu_seconds)
        except Exception as e:   # noqa: BLE001
            log(f"[cpu] the vendored reference failed ({e!r}); timing the NumPy port instead")
            cpu = None
        if cpu is None:
            cpu = cpu_arm(args, 10 ** 9, 2, seconds=args.cpu_seconds)
    variants = {}
    if rank == 0 and world == 1 and not args.no_sweep:
        variants = time_variants(args, data, E, max_len, dev, local)
    if rank == 0:
        key = f"fused_critic_kernel_B{B}" if f"fused_critic_kernel_B{B}" in rooflines else f"her_sample_kernel_B{B}"
        roof = dict(rooflines.get(key, {}))
        roof["kernel"] = key.rsplit("_B", 1)[0]
        roof["share_of_step"] = (roof.get("ms_per_launch", 0.0) / (ms / args.steps)) if roof else None
        roof["peak_source"] = peak_src
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, world),
            "updates_per_s": world * args.steps / (ms * 1e-3) / world,
            "per_step_ms": per_step_detail,
            "back_to_back": {"ms_per_step": ms_b2b / args.steps, "value": world * B * args.steps / (ms_b2b * 1e-3),
                             "note": "same steps without the L2 flush, graph replays pipelined"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / n_e2e, "steps": n_e2e,
                    "api": "DDPG.update(step) with host random.sample index stream + metric read-back; "
                           "16 episodes ingested every 40 updates",
                    "device_index_stream": {"ms_per_step": ms_e2e_dev / n_e2e,
                                            "value": world * B * n_e2e / (ms_e2e_dev * 1e-3),
                                            "note": "same call, index_source='device' (rank-local wall clock)"}},
            "gpu_launches": launches, "clocks": clk, "roofline": roof, "rooflines": rooflines, "sweep": sweep,
            "variants": variants, "configs": extra, "dp_parity": parity,
            "cpu_baseline": None if cpu is None else {k_: cpu[k_] for k_ in ("value", "unit", "cores", "kind", "sample")},
            "library": os.path.relpath(gcrl_b200.library_path(), ROOT),
            "kernel_launches_total": int(lib.gcrl_kernel_launches()) - launches0,
        }
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
            log(f"[dump] {len(outputs)} arrays of the last timed step written to {args.dump_outputs}")
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def time_variants(args, data, E, max_len, dev, local, steps=60):
    """updates/s of the other agents behind the same interface (TD3, SAC, TQC) on the same buffer
    contents and shapes, device index stream, metric read-back every step (their update() is synchronous)."""
    import torch
    from gcrl_b200 import SACAgent, TD3Agent, TQCAgent
    out = {}
    T = 50
    for name, cls in (("td3", TD3Agent), ("sac", SACAgent), ("tqc", TQCAgent)):
        try:
            cfg = agent_config(args, max_len)
            cfg.alpha_lr, cfg.alpha_min, cfg.alpha_min_steps = 3e-4, 0.05, 0
            cfg.ac_update_freq = 2 if name == "td3" else 1
            cfg.grad_clip = 1.0
            torch.manual_seed(1898)
            ag = cls(args.obs + args.goal, args.act, cfg, None, 1, 40, index_source="device", device=local)
            for e in range(min(E, 2000)):
                ag.buffer.push_episode(data["s"][e], data["a"][e], data["ns"][e], data["r"][e], data["d"][e],
                                       data["ag"][e], data["fut"][e])
            for i in range(5):
                ag.update(i + 1)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(steps):
                info = ag.update(6 + i)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            assert all(np.isfinite(float(x)) for x in info)
            out[name] = {"updates_per_s": steps / dt, "ms_per_update": dt / steps * 1e3, "batch": args.batch,
                         "hidden": args.hidden, "layers": args.layers}
            del ag
        except Exception as e:   # noqa: BLE001
            out[name] = {"error": str(e)}
    out.update(time_replay_variants(args, data, E, max_len, local))
    return out


def time_replay_variants(args, data, E, max_len, local, steps=100):
    """DDPG.update(step) behind the two non-HER buffers (buffer_type "PER" / "REPLAY", src/agent.py:67-70) on the
    raw transitions of the same synthetic episodes: prioritised draw through numpy.random.choice's exact
    arithmetic + importance-weighted critic loss + priority write-back, and the uniform random.sample draw.
    Wall clock per synchronous update, metric read-back included."""
    import torch
    from gcrl_b200 import DDPG
    out = {}
    for name, btype in (("ddpg_per", "PER"), ("ddpg_replay", "REPLAY")):
        try:
            cfg = agent_config(args, max_len)
            cfg.buffer_type, cfg.alpha, cfg.beta, cfg.beta_end = btype, 0.6, 0.4, 10000
            torch.manual_seed(1898)
            np.random.seed(1898)
            ag = DDPG(args.obs + args.goal, args.act, cfg, None, 1, 40, device=local)
            n_ep = min(E, max_len // 50)
            for lo in range(0, n_ep, 256):
                hi = min(n_ep, lo + 256)
                cat = lambda k: np.concatenate([data[k][e] for e in range(lo, hi)])     # noqa: E731
                ag.buffer.push_rows(cat("s"), cat("a"), cat("r"), cat("ns"), cat("d"))
            for i in range(40):          # the priorities move away from 1.0: the cumsum starts to round
                ag.update(i + 1)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(steps):
                info = ag.update(41 + i)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            assert np.isfinite(float(info[0]))
            rec = {"updates_per_s": steps / dt, "ms_per_update": dt / steps * 1e3, "batch": args.batch,
                   "entries": len(ag.buffer)}
            if btype == "PER":
                rec["cumsum_additions_round"] = bool(ag.buffer.last_sample_info()[1])
            out[name] = rec
            del ag
        except Exception as e:   # noqa: BLE001
            out[name] = {"error": str(e)}
    return out


def main():
    args = parse()
    if args.impl == "reference":
        reference_main(args)
    else:
        gpu_main(args)


if __name__ == "__main__":
    main()

"""torchrun worker for tests/test_dp_gpu.py::test_two_gpu_nccl_run_matches_single_rank: every rank
updates on its own batch with NCCL-averaged gradients; rank 0 also runs a single-rank agent on the
concatenated batch and compares."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "goal-conditioned-rl-framework_b200"))
from tests.helpers import weights_close  # noqa: E402
from tests.test_dp_gpu import rand_batch  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    D, A, H, L, B = 21, 3, 256, 3, 256
    ag = make_agent_on(local, D, A, H, L, B)
    ag.enable_data_parallel()
    single = make_agent_on(local, D, A, H, L, world * B) if rank == 0 else None
    rng = np.random.default_rng(5)
    for step in (39, 40, 41, 42):
        batches = [rand_batch_on(rng, B, D, A, local) for _ in range(world)]   # same stream on every rank
        info = ag.update(step, batch=batches[rank])
        if rank == 0:
            want = single.update(step, batch=tuple(torch.cat(parts) for parts in zip(*batches)))
            np.testing.assert_allclose(np.array([float(x) for x in info]), np.array([float(x) for x in want]),
                                       rtol=5e-5, atol=2e-6)
    # replicas identical across ranks, and equal to the single-rank run within tolerance
    flat = torch.cat([torch.from_numpy(w).reshape(-1) for w, _ in ag.actor.layers() + ag.critic.layers()]).cuda()
    gathered = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(gathered, flat)
    for g in gathered[1:]:
        assert torch.equal(g, gathered[0])
    if rank == 0:
        for (w, b), (ws, bs) in zip(ag.actor.layers() + ag.critic.layers() + ag.target_critic.layers(),
                                    single.actor.layers() + single.critic.layers() + single.target_critic.layers()):
            assert weights_close(w, ws, 1e-3, 4) and weights_close(b, bs, 1e-3, 4)
    tqc_section(rank, world, local)
    p2p_section(rank, world, local)
    normaliser_section(rank, world, local)
    if rank == 0:
        print("DP_OK", flush=True)
    dist.barrier()
    dist.destroy_process_group()


def normaliser_section(rank, world, local):
    """RunningNormalizer.update as a collective over NCCL: per-rank observation batches, identical replicas, and
    equal to the oracle on the concatenated batch to float64 rounding."""
    from gcrl_b200 import RunningNormalizer
    from oracle import her as OH
    dim = 19
    nz = RunningNormalizer(dim, device=local)
    nz.enable_data_parallel()
    single = OH.RunningNormalizerOracle(dim)
    rng = np.random.default_rng(17)
    for step in range(4):
        parts = [rng.standard_normal((2 + r, dim)) * (1 + step) + 0.5 * r for r in range(world)]   # same stream everywhere
        nz.update(parts[rank])
        single.update(np.concatenate(parts, 0))
    np.testing.assert_allclose(nz.mean, single.mean, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(nz.var, single.var, rtol=1e-12, atol=1e-12)
    flat = torch.from_numpy(np.concatenate([nz.mean, nz.var])).cuda(local)
    gathered = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(gathered, flat)
    for g in gathered[1:]:
        assert torch.equal(g, gathered[0]), "normaliser replicas diverged"


def p2p_section(rank, world, local):
    """The same parity rule with the gradients averaged over NVLink peer memory (enable_peer_data_parallel):
    N ranks on per-rank batches == one rank on the concatenated batch within the fp32 tolerance, replicas
    bit-identical, for DDPG and TD3."""
    from gcrl_b200 import TD3Agent
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC, NET_CRITIC2
    from oracle import ddpg as OD
    from tests.test_ddpg_gpu import make_config
    D, A, H, L, B = 21, 3, 256, 3, 256
    dev = torch.device("cuda", local)
    for algo in ("ddpg", "td3"):
        def build(batch):
            if algo == "ddpg":
                return make_agent_on(local, D, A, H, L, batch)
            ag = TD3Agent(D, A, make_config(hidden_dim=H, layer_count=L, batch_size=batch, grad_clip=0.5, ac_update_freq=2),
                          None, 1, 40, device=local)
            r = np.random.default_rng(3)
            ag._set_layers(NET_ACTOR, OD.init_mlp(r, D, H, A, L))
            ag._set_layers(NET_CRITIC, OD.init_mlp(r, D + A, H, 1, L))
            ag._set_layers(NET_CRITIC2, OD.init_mlp(r, D + A, H, 1, L))
            ag.update_target_network()
            return ag
        ag = build(B)
        ag.enable_peer_data_parallel()
        single = build(world * B) if rank == 0 else None
        rng = np.random.default_rng(9)
        for step in (39, 40, 41, 42):
            batches = [rand_batch_on(rng, B, D, A, local) for _ in range(world)]
            noises = [torch.from_numpy(rng.standard_normal((B, A)).astype(np.float32)).to(dev) for _ in range(world)]
            kw = {"noise": noises[rank]} if algo == "td3" else {}
            info = ag.update(step, batch=batches[rank], **kw)
            if rank == 0:
                kw1 = {"noise": torch.cat(noises)} if algo == "td3" else {}
                want = single.update(step, batch=tuple(torch.cat(parts) for parts in zip(*batches)), **kw1)
                np.testing.assert_allclose(np.array([float(x) for x in info]), np.array([float(x) for x in want]),
                                           rtol=5e-5, atol=2e-6)
        nets = [ag.actor, ag.target_actor] + ([ag.critic, ag.target_critic] if algo == "ddpg" else
                                              [ag.critic_1, ag.critic_2, ag.target_critic_1, ag.target_critic_2])
        flat = torch.cat([torch.from_numpy(w).reshape(-1) for n in nets for w, _ in n.layers()]).to(dev)
        gathered = [torch.empty_like(flat) for _ in range(world)]
        dist.all_gather(gathered, flat)
        for g in gathered[1:]:
            assert torch.equal(g, gathered[0]), f"{algo}: peer-averaged replicas diverged"
        if rank == 0:
            snets = [single.actor] + ([single.critic] if algo == "ddpg" else [single.critic_1, single.critic_2])
            pnets = [ag.actor] + ([ag.critic] if algo == "ddpg" else [ag.critic_1, ag.critic_2])
            for pn, sn in zip(pnets, snets):
                for (w, b), (ws, bs) in zip(pn.layers(), sn.layers()):
                    assert weights_close(w, ws, 1e-3, 4) and weights_close(b, bs, 1e-3, 4), algo
        dist.barrier()
        del ag


def tqc_section(rank, world, local):
    """TQC over NCCL: every rank on its own batch and noise; replicas (weights, log_alpha, BatchNorm running
    statistics) must stay bit-identical across ranks.  With sync-BN (the default) the ranks must also equal ONE rank
    on the concatenated batch at the weights_close tolerance (SURVEY 8(e))."""
    from oracle import ddpg as OD
    from oracle import sac as OS
    from gcrl_b200 import TQCAgent
    from tests.helpers import assert_sac_actor_close, weights_close
    from tests.test_sac_gpu import actor_params, assert_running_stats_close, load_initial, sac_config
    D, A, H, L, B = 22, 3, 64, 3, 128
    dev = torch.device("cuda", local)
    for sync_bn in (True, False):
        rng = np.random.default_rng(7)
        actor0, stats0 = OS.init_sac_actor(rng, D, H, A, L, head_scale=0.1, log_std_bias=-1.0)
        critics0 = [OD.init_mlp(rng, D + A, H, 1, L) for _ in range(5)]

        def make(batch):
            cfg = sac_config(hidden_dim=H, layer_count=L, batch_size=batch, grad_clip=0.5, tau=0.05, alpha_min_steps=0,
                             alpha_lr=1e-2)
            a = TQCAgent(D, A, cfg, None, 1, 2, device=local)
            load_initial(a, actor0, stats0, critics0)
            return a
        ag = make(B)
        ag.enable_data_parallel(sync_bn=sync_bn)
        single = make(world * B) if (sync_bn and rank == 0) else None
        nsteps = 4
        for step in range(1, nsteps + 1):
            per_rank = []
            for _ in range(world):
                b = rand_batch_on(rng, B, D, A, local)
                e = [torch.from_numpy(rng.standard_normal((B, A)).astype(np.float32)).to(dev) for _ in range(2)]
                per_rank.append((b, e))
            b, e = per_rank[rank]
            info = ag.update(step, batch=b, eps_next=e[0], eps_cur=e[1])
            assert len(info) in (6, 9) and all(np.isfinite(float(x)) for x in info)
            if single is not None:
                cat = tuple(torch.cat([pr[0][k] for pr in per_rank]) for k in range(5))
                e0 = torch.cat([pr[1][0] for pr in per_rank])
                e1 = torch.cat([pr[1][1] for pr in per_rank])
                want = single.update(step, batch=cat, eps_next=e0, eps_cur=e1)
                np.testing.assert_allclose([float(x) for x in info[:2]], [float(x) for x in want[:2]], rtol=2e-5,
                                           atol=1e-6, err_msg="sync-BN critic losses (averaged over ranks) vs one rank")
        parts = [torch.from_numpy(w).reshape(-1) for v in ag._critic_views + ag._target_views for w, _ in v.layers()]
        parts += [torch.from_numpy(np.concatenate([x.reshape(-1) for x in ag.actor.bn(l)])) for l in range(L)]
        parts += [torch.from_numpy(ag.actor.linear(l)[0]).reshape(-1) for l in range(L + 2)]
        parts.append(torch.tensor([ag.get_log_alpha()]))
        flat = torch.cat(parts).to(dev)
        gathered = [torch.empty_like(flat) for _ in range(world)]
        dist.all_gather(gathered, flat)
        for g in gathered[1:]:
            assert torch.equal(g, gathered[0]), f"TQC replicas diverged (sync_bn={sync_bn})"
        if single is not None:
            (p0, s0), (ps, ss) = actor_params(ag), actor_params(single)
            assert_sac_actor_close(p0, ps, 1e-3, nsteps)
            assert_running_stats_close(p0, s0, ps, ss)
            for v0, vs in zip(ag._critic_views + ag._target_views, single._critic_views + single._target_views):
                for (w, b_), (ws, bs) in zip(v0.layers(), vs.layers()):
                    assert weights_close(w, ws, 1e-3, nsteps) and weights_close(b_, bs, 1e-3, nsteps), "sync-BN critic"
            assert abs(ag.get_log_alpha() - single.get_log_alpha()) <= 1e-6
        dist.barrier()
        del ag, single


def make_agent_on(dev, D, A, H, L, B):
    from gcrl_b200 import DDPG
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC
    from oracle import ddpg as OD
    from tests.test_ddpg_gpu import make_config
    ag = DDPG(D, A, make_config(hidden_dim=H, layer_count=L, batch_size=B, grad_clip=0.5), None, 1, 40, device=dev)
    rng = np.random.default_rng(3)
    ag._set_layers(NET_ACTOR, OD.init_mlp(rng, D, H, A, L))
    ag._set_layers(NET_CRITIC, OD.init_mlp(rng, D + A, H, 1, L))
    ag.update_target_network()
    return ag


def rand_batch_on(rng, B, D, A, dev):
    return tuple(t.to(torch.device("cuda", dev)) for t in (x.cpu() for x in rand_batch(rng, B, D, A)))


if __name__ == "__main__":
    main()

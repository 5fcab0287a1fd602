"""GPU: a weight write made between two updates reaches the weight copies the next update reads.

Agent X runs one update, then a write (set_layer / set_critic_layer / set_actor_linear, hard_update or soft_update),
then a second update on batch b2.  Agent Y, built from the same init, is given X's weights after the write through
the set-layer entry points and runs one update on b2 with the same noise.  What an update computes before its first
optimiser step -- critic loss, TD, Q and the critic gradient norms -- depends on the weights and the batch only, so
the two must agree bit for bit.  A transposed copy (W^T) or TF32 hi / lo halves that missed the write would make X's
differ.

Engines (use_tc in agent.cu / sac.cu): DDPG at B = 256 runs the row-slab kernels, which read W^T; DDPG at B = 2048
and precision 1 runs tcgen05, which reads the halves of p and W^T; SAC / TQC at B = 128 and precision 2 run tcgen05
for every network.  Both agents replay captured graphs, as update() does by default.
"""
import numpy as np
import pytest

from oracle import ddpg as OD
from oracle import sac as OS
from tests import test_sac_gpu as T
from tests.test_fused_variants_gpu import init_nets, make_agent, make_batch

pytestmark = pytest.mark.gpu

DDPG_SHAPE = dict(D=21, A=3, H=128, L=2)
SAC_SHAPE = dict(D=10, A=3, H=64, L=3)      # L = 3: W^T of hidden layers 1 and 2


def to_device(batch):
    import torch
    return tuple(torch.from_numpy(x).cuda() for x in batch)


def assert_bits_equal(mx, my, picks, label):
    for name, k in picks.items():
        x, y = np.float32(mx[k]), np.float32(my[k])
        assert x.view(np.uint32) == y.view(np.uint32), (label, name, float(x), float(y))


# ---- DDPG ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("write", ["set_layer", "hard_update", "soft_update"])
@pytest.mark.parametrize("B, precision", [(256, 1), (2048, 1)], ids=["rowslab-B256", "tcgen05-B2048"])
def test_ddpg_write_between_updates_reaches_next_update(B, precision, write, monkeypatch):
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC, NET_T_ACTOR, NET_T_CRITIC
    monkeypatch.delenv("GCRL_FUSED_R", raising=False)
    monkeypatch.delenv("GCRL_B200_NO_FUSED", raising=False)
    D, A, H, L = (DDPG_SHAPE[k] for k in "DAHL")
    rng = np.random.default_rng(11)
    nets = init_nets(rng, "ddpg", D, A, H, L)
    b1, b2 = make_batch(rng, B, D, A), make_batch(rng, B, D, A)
    fresh = init_nets(rng, "ddpg", D, A, H, L) + init_nets(rng, "ddpg", D, A, H, L)

    X = make_agent("ddpg", B, nets, monkeypatch, D, A, H, L, graphs=True, precision=precision)
    X.update(1, batch=to_device(b1))
    if write == "set_layer":
        for net, params in zip((NET_ACTOR, NET_CRITIC, NET_T_ACTOR, NET_T_CRITIC), fresh):
            X._set_layers(net, params)
    elif write == "hard_update":
        X.update_target_network(hard_update=True)
    else:
        X.update_target_network(hard_update=False, tau=0.5)
    Y = make_agent("ddpg", B, nets, monkeypatch, D, A, H, L, graphs=True, precision=precision)
    for net in X._all_nets():
        Y._set_layers(net, X._get_layers(net))
    mx = X.update(2, batch=to_device(b2))
    my = Y.update(2, batch=to_device(b2))
    # (critic_loss, actor_loss, td, q, critic_grad_norm, actor_grad_norm)
    assert_bits_equal(mx, my, {"critic_loss": 0, "td": 2, "q": 3, "critic_grad_norm": 4}, (B, write))


# ---- SAC / TQC ----------------------------------------------------------------------------------------------
def make_sac(algo, B, seed):
    """An agent whose updates leave alpha alone (alpha_min_steps): its log_alpha copies to another agent exactly."""
    from gcrl_b200 import SACAgent, TQCAgent
    D, A, H, L = (SAC_SHAPE[k] for k in "DAHL")
    rng = np.random.default_rng(seed)
    cfg = T.sac_config(hidden_dim=H, layer_count=L, batch_size=B, grad_clip=0.5, tau=0.05, alpha_min_steps=10)
    actor0, stats0 = OS.init_sac_actor(rng, D, H, A, L, head_scale=0.1, log_std_bias=-1.0)
    critics0 = [OD.init_mlp(rng, D + A, H, 1, L) for _ in range(2 if algo == "sac" else 5)]
    ag = (SACAgent if algo == "sac" else TQCAgent)(D, A, cfg, None, 1, 2, precision=2)
    T.load_initial(ag, actor0, stats0, critics0)
    return ag


def copy_sac(src, dst):
    L = src.config.layer_count
    for layer in range(L + 2):
        dst.actor.set_linear(layer, *src.actor.linear(layer))
    for layer in range(L):
        dst.actor.set_bn(layer, *src.actor.bn(layer))
    for views in ("_critic_views", "_target_views"):
        for s, d in zip(getattr(src, views), getattr(dst, views)):
            d.set_layers(s.layers())
    dst.set_log_alpha(src.get_log_alpha())


@pytest.mark.parametrize("write", ["set_critic_layer", "set_actor_linear", "hard_update"])
@pytest.mark.parametrize("algo", ["sac", "tqc"])
def test_sac_write_between_updates_reaches_next_update(algo, write, monkeypatch):
    import torch
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    B = 128
    D, A, H, L = (SAC_SHAPE[k] for k in "DAHL")
    rng = np.random.default_rng(23)
    b1, b2 = make_batch(rng, B, D, A), make_batch(rng, B, D, A)
    eps = [torch.from_numpy(rng.standard_normal((B, A)).astype(np.float32)).cuda() for _ in range(4)]

    X = make_sac(algo, B, seed=5)
    X.update(1, batch=to_device(b1), eps_next=eps[0], eps_cur=eps[1])
    if write == "set_critic_layer":
        for views in (X._critic_views, X._target_views):
            for v in views:
                v.set_layers(OD.init_mlp(rng, D + A, H, 1, L))
    elif write == "set_actor_linear":
        for layer in range(L + 2):
            w, b = X.actor.linear(layer)
            X.actor.set_linear(layer, rng.uniform(-0.3, 0.3, w.shape).astype(np.float32),
                               rng.uniform(-0.1, 0.1, b.shape).astype(np.float32))
    else:
        X.update_target_network()
    Y = make_sac(algo, B, seed=5)
    copy_sac(X, Y)
    mx = X.update(2, batch=to_device(b2), eps_next=eps[2], eps_cur=eps[3])
    my = Y.update(2, batch=to_device(b2), eps_next=eps[2], eps_cur=eps[3])
    # (critic1_loss, critic2_loss, actor_loss, td, q, critic1_grad_norm, critic2_grad_norm, ...); TQC: means over the
    # critics, and its q is taken after the critic step (the mean over the stepped critics)
    picks = {"critic1_loss": 0, "critic2_loss": 1, "td": 3, "critic1_grad_norm": 5, "critic2_grad_norm": 6}
    if algo == "sac":
        picks["q"] = 4
    assert_bits_equal(mx, my, picks, (algo, write))

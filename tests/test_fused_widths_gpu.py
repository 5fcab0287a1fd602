"""GPU: the two instances of the row-slab update kernels (csrc/fused.cu).

Every row-slab kernel exists twice: h256:: with H = 256 fixed at compile time, and anyh:: for every width.  The
launcher takes h256:: at H = 256 unless GCRL_FUSED_GENERIC=1.  Both run the same sums in the same order, so
  * at H = 256 they must leave bit-identical metrics and weights, for DDPG and TD3 at every rows-per-CTA
    variant (R = 2, 4, 8, the 2-CTA cluster split among them);
  * an odd width (H = 200) at B = 301 and 1021 runs anyh:: and is checked against the NumPy oracle with the
    tolerances of smoke().
"""
import re
import types

import numpy as np
import pytest

from oracle import ddpg as OD
from tests.test_fused_variants_gpu import (PUSH, STEPS, all_weights, first_difference, init_nets, launched_kernels,
                                           make_agent, make_batch, run_updates, set_rows_per_cta)

pytestmark = pytest.mark.gpu


def instances(names):
    return {m.group(1) for n in names for m in re.finditer(r"(h256|anyh)::fused_(critic|actor)_kernel", n)}


@pytest.mark.parametrize("algo", ["ddpg", "td3"])
@pytest.mark.parametrize("B,R", [(256, None), (256, 4), (517, None), (1000, None)], ids=["B256", "B256R4", "B517", "B1000"])
def test_h256_instance_matches_generic(B, R, algo, monkeypatch):
    rng = np.random.default_rng(B + 17)
    nets = init_nets(rng, algo, **PUSH)
    batches = [make_batch(rng, B, PUSH["D"], PUSH["A"]) for _ in STEPS]
    noises = [rng.standard_normal((B, PUSH["A"])).astype(np.float32) for _ in STEPS]
    set_rows_per_cta(monkeypatch, R)
    got = {}
    for generic in (False, True):
        if generic:
            monkeypatch.setenv("GCRL_FUSED_GENERIC", "1")
        else:
            monkeypatch.delenv("GCRL_FUSED_GENERIC", raising=False)
        ag = make_agent(algo, B, nets, monkeypatch, **PUSH)
        info = []
        names = launched_kernels(lambda: info.extend(run_updates(ag, algo, batches, noises)))
        assert instances(names) == {"anyh" if generic else "h256"}, sorted(names)
        got[generic] = (info, all_weights(ag))
    assert got[False][0] == got[True][0]
    assert first_difference(got[False][1], got[True][1]) is None


@pytest.mark.parametrize("B", [301, 1021])
def test_odd_width_matches_oracle(B, monkeypatch):
    import torch
    from gcrl_b200 import DDPG
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC
    monkeypatch.delenv("GCRL_FUSED_R", raising=False)
    monkeypatch.delenv("GCRL_FUSED_GENERIC", raising=False)
    monkeypatch.setenv("GCRL_B200_NO_GRAPH", "1")
    D, A, H, L = 21, 3, 200, 3
    rng = np.random.default_rng(B)
    cfg = types.SimpleNamespace(
        hidden_dim=H, layer_count=L, actor_lr=1e-3, actor_lr_min=1e-3, ac_scheduler_steps=1,
        critic_lr=1e-3, critic_lr_min=1e-3, cr_scheduler_steps=1, buffer_type="HER", max_len=100_000,
        alpha=1.0, batch_size=B, gamma=0.98, ac_update_freq=1, noise_std=0.2, noise_clamp=0.5,
        policy_noise=0.0, grad_clip=10.0, beta=1.0, beta_end=1, k_future=4, max_eps_len=50, tau=0.05)
    agent = DDPG(D, A, cfg, None, 1, 40)
    actor0, critic0 = OD.init_mlp(rng, D, H, A, L), OD.init_mlp(rng, D + A, H, 1, L)
    agent._set_layers(NET_ACTOR, actor0)
    agent._set_layers(NET_CRITIC, critic0)
    agent.update_target_network()
    orc = OD.DDPGOracle(actor0, critic0, gamma=cfg.gamma, tau=cfg.tau, grad_clip=cfg.grad_clip,
                        actor_lr=cfg.actor_lr, critic_lr=cfg.critic_lr)
    for step in (39, 40):
        batch = make_batch(rng, B, D, A)
        info = []
        names = launched_kernels(lambda: info.extend(
            agent.update(step, batch=tuple(torch.from_numpy(x).cuda() for x in batch))))
        assert instances(names) == {"anyh"}, sorted(names)
        want = orc.update_on_batch(step, *batch)
        np.testing.assert_allclose(np.array([float(x) for x in info]), np.array(want), rtol=5e-5, atol=2e-6)
    for (w, _), (rw, _) in zip(agent.critic.layers() + agent.actor.layers(), orc.critic + orc.actor):
        assert np.max(np.abs(w - rw)) <= 1e-5 * np.max(np.abs(rw)) + 5e-6

"""CPU: the quantile-critic TQC reference (tests/tqc_quantile_reference.py) against a float64 torch-autograd
restatement of sb3-contrib's TQC (``quantile_huber_loss`` with ``sum_over_quantiles=False``, the sorted and truncated
target, the untruncated actor loss), on random inputs with ties and with d = 0; and TQCAgent's argument checks, which
must refuse bad values before anything touches a device."""
import types

import numpy as np
import pytest

from tests import tqc_quantile_reference as R


def sb3_quantile_huber_loss(current, target):
    """sb3-contrib common/utils.py quantile_huber_loss(current [B, n, M], target [B, 1, K], sum_over_quantiles=False)
    with an optional per-sample weight folded in before the mean (prioritised replay)."""
    import torch
    M = current.shape[-1]
    cum_prob = ((torch.arange(M, dtype=torch.float64) + 0.5) / M).view(1, 1, -1, 1)
    delta = target.unsqueeze(-2) - current.unsqueeze(-1)
    adelta = delta.abs()
    huber = torch.where(adelta > 1, adelta - 0.5, delta ** 2 * 0.5)
    return (cum_prob - (delta.detach() < 0).double()).abs() * huber          # [B, n, M, K]


def sb3_target(next_quantiles, next_log_prob, r, d, gamma, ent_coef, drop_per_net):
    """sb3-contrib TQC.train: sort the pooled atoms, keep quantiles_total - drop_per_net * n_critics."""
    import torch
    B, n, M = next_quantiles.shape
    z, _ = torch.sort(next_quantiles.reshape(B, -1))
    z = z[:, :n * M - drop_per_net * n]
    z = z - ent_coef * next_log_prob.reshape(-1, 1)
    return r + (1 - d) * gamma * z


def rand_case(rng, B, n, M, ties):
    z = rng.standard_normal((n, B, M)).astype(np.float32)
    zt = (rng.standard_normal((n, B, M)) * 1.5).astype(np.float32)
    if ties:                          # many equal atoms within a row, across critics and between Z and the targets
        z = np.round(z * 2) / 2
        zt = np.round(zt * 2) / 2
        zt[:, :, : M // 2] = zt[:1, :, : M // 2]
    logp = (rng.standard_normal((B, 1)) * 0.3).astype(np.float32)
    r = -(rng.random((B, 1)) > 0.3).astype(np.float32)
    d = (rng.random((B, 1)) < 0.2).astype(np.float32)
    return z.astype(np.float32), zt.astype(np.float32), logp, r, d


CASES = [(7, 5, 5, 0, False), (33, 5, 25, 2, False), (16, 5, 25, 2, True), (9, 5, 1, 0, False), (12, 3, 8, 0, True),
         (5, 5, 51, 7, True)]


@pytest.mark.parametrize("B,n,M,drop,ties", CASES)
def test_target_loss_and_gradients_match_sb3_restatement(B, n, M, drop, ties):
    import torch
    rng = np.random.default_rng(B * 100 + M)
    z, zt, logp, r, d = rand_case(rng, B, n, M, ties)
    gamma, alpha = 0.98, np.float32(0.37)
    y = R.quantile_target(zt, logp, r, d, gamma, alpha, drop)
    assert y.shape == (B, n * (M - drop))
    assert np.all(np.diff(y * np.where(d > 0, 0, 1), axis=1) >= -1e-6)       # sorted (rows with done are constant)
    y64 = sb3_target(torch.from_numpy(zt.transpose(1, 0, 2)).double(), torch.from_numpy(logp).double(),
                     torch.from_numpy(r).double(), torch.from_numpy(d).double(), gamma, float(alpha), drop)
    np.testing.assert_allclose(y, y64.numpy(), rtol=1e-6, atol=1e-6)
    for w in (None, rng.uniform(0.1, 1.0, (B, 1)).astype(np.float32)):
        cur = torch.from_numpy(z.transpose(1, 0, 2)).double().requires_grad_(True)        # [B, n, M]
        pair = sb3_quantile_huber_loss(cur, torch.from_numpy(y).double().unsqueeze(1))
        if w is not None:
            pair = pair * torch.from_numpy(w).double().view(B, 1, 1, 1)
        loss = pair.mean()                              # sb3: one joint mean over the critics
        loss.backward()
        got = [R.quantile_huber(z[i], y, w) for i in range(n)]
        # per-critic losses: their mean is sb3's joint loss; each critic's gradient is n times sb3's share
        np.testing.assert_allclose(np.mean([g[0] for g in got]), loss.item(), rtol=2e-6)
        for i in range(n):
            np.testing.assert_allclose(got[i][0], pair[:, i].mean().item(), rtol=2e-6)
            np.testing.assert_allclose(got[i][1], n * cur.grad[:, i].numpy(), rtol=2e-5,
                                       atol=2e-6 * float(np.abs(got[i][1]).max()) + 1e-12)
            td = np.abs(z[i].astype(np.float64).mean(1, keepdims=True) - y.astype(np.float64).mean(1, keepdims=True))
            np.testing.assert_allclose(got[i][2], td, rtol=1e-5, atol=1e-6)


def test_actor_gradient_per_atom_matches_sb3_actor_loss():
    """sb3-contrib: qf_pi = critic(obs, a).mean(dim=2).mean(dim=1); loss = (ent_coef * log_prob - qf_pi).mean():
    every atom receives -1 / (B n M), the constant the reference and the kernels use."""
    import torch
    B, n, M = 11, 5, 25
    rng = np.random.default_rng(3)
    atoms = torch.from_numpy(rng.standard_normal((B, n, M))).requires_grad_(True)
    logp = torch.from_numpy(rng.standard_normal((B, 1)))
    loss = (0.3 * logp - atoms.mean(dim=2).mean(dim=1, keepdim=True)).mean()
    loss.backward()
    np.testing.assert_allclose(atoms.grad.numpy(), -1.0 / (B * n * M), rtol=1e-12)
    ref = float(np.mean(0.3 * logp.numpy() - atoms.detach().numpy().reshape(B, -1).mean(1, keepdims=True)))
    np.testing.assert_allclose(loss.item(), ref, rtol=1e-12)


def test_reference_update_runs_and_moves_every_critic():
    """Three reference updates (actor and alpha steps included) on a small shape: finite metrics, every critic's
    head [M, H] moved, the targets Polyak-averaged toward them."""
    from oracle import ddpg as OD
    from oracle import sac as OS
    D, A, H, L, B, M = 7, 2, 16, 2, 9, 5
    rng = np.random.default_rng(0)
    actor0, stats0 = OS.init_sac_actor(rng, D, H, A, L, head_scale=0.1, log_std_bias=-1.0)
    critics0 = [OD.init_mlp(rng, D + A, H, M, L) for _ in range(5)]
    orc = R.QuantileTQCOracle(actor0, stats0, critics0, n_quantiles=M, drop_per_net=2, act_dim=A, gamma=0.98,
                              tau=0.05, grad_clip=0.5, actor_lr=1e-3, critic_lr=1e-3, alpha_lr=1e-2,
                              alpha_min_steps=0, gradient_step=2)
    for step in (1, 2, 3):
        s = rng.standard_normal((B, D)).astype(np.float32)
        batch = (s, rng.uniform(-1, 1, (B, A)).astype(np.float32), -(rng.random((B, 1)) > 0.3).astype(np.float32),
                 s + np.float32(0.1), np.zeros((B, 1), np.float32))
        info = orc.update_on_batch(step, *batch, rng.standard_normal((B, A)).astype(np.float32),
                                   rng.standard_normal((B, A)).astype(np.float32))
        assert len(info) == 9 and all(np.isfinite(info))
    assert orc.last_y.shape == (B, 5 * (M - 2))
    for c, c0, t in zip(orc.critics, critics0, orc.target_critics):
        assert c[-1][0].shape == (M, H) and not np.array_equal(c[-1][0], c0[-1][0])
        assert not np.array_equal(t[-1][0], c0[-1][0])


# ---- TQCAgent argument checks: no device needed -----------------------------------------------------------------
BAD = [dict(n_quantiles=0), dict(n_quantiles=-3), dict(n_quantiles=52), dict(n_quantiles=2.5), dict(n_quantiles=True),
       dict(n_quantiles="25"), dict(n_quantiles=25, top_quantiles_to_drop_per_net=25),
       dict(n_quantiles=25, top_quantiles_to_drop_per_net=-1), dict(n_quantiles=5, top_quantiles_to_drop_per_net=1.0),
       dict(n_quantiles=1, top_quantiles_to_drop_per_net=1)]


@pytest.mark.parametrize("kw", BAD, ids=[str(sorted(k.items())) for k in BAD])
def test_tqc_agent_refuses_bad_quantile_arguments_before_any_device_call(kw):
    from gcrl_b200 import TQCAgent
    with pytest.raises(ValueError):
        TQCAgent(10, 3, types.SimpleNamespace(), None, 1, 2, **kw)


def test_valid_quantile_arguments_pass_the_checks():
    from gcrl_b200 import TQCAgent
    assert TQCAgent._check_quantiles(None, 2) == (None, 0)
    assert TQCAgent._check_quantiles(25, 2) == (25, 2)
    assert TQCAgent._check_quantiles(np.int64(51), 0) == (51, 0)
    assert TQCAgent._check_quantiles(1, 0) == (1, 0)


def test_sac_agent_takes_no_quantile_arguments():
    from gcrl_b200 import SACAgent
    for kw in (dict(n_quantiles=25), dict(top_quantiles_to_drop_per_net=2)):
        with pytest.raises(TypeError):
            SACAgent(10, 3, types.SimpleNamespace(), None, 1, 2, **kw)

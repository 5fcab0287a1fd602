"""GPU: TQC with quantile critics (``TQCAgent(n_quantiles=M, top_quantiles_to_drop_per_net=d)``, csrc/sac.cu
quantile_target_kernel / quantile_huber_kernel, gcrl_sac_create_quantile) against the NumPy reference
(tests/tqc_quantile_reference.py) and against itself.

Tolerances are the SAC / TQC odd-shape ones (tests/test_sac_gpu.py): metrics rel 5e-5 (times sqrt(B / 256) above
256 rows) + abs 2e-6, log_alpha rel 1e-5, and every weight, bias and target
weight within Adam's hard bound 2 lr n (assert_within_adam_bound says why not tests.helpers.weights_close); the
tensor-core engine against the fp32 one at 4x those (tests/test_sac_tc_gpu.py).  Every other comparison is bit for
bit: update_many against the update() loop, eager launches against graph replay, a saved and reloaded agent
against the one it was saved from."""
import ctypes as C

import numpy as np
import pytest

from tests import tqc_quantile_reference as R
from tests.helpers import bits
from tests.test_sac_gpu import actor_params, load_initial, sac_config

pytestmark = pytest.mark.gpu

ENG = 4.0


def make_pair(B, H, L, D, A, M, drop, seed=5, precision=0, reference=True, n=5, **over):
    """A quantile TQCAgent with n critics and the reference on the same seeded initial networks."""
    from gcrl_b200 import TQCAgent
    from oracle import ddpg as OD
    from oracle import sac as OS
    rng = np.random.default_rng(seed)
    cfg = sac_config(hidden_dim=H, layer_count=L, batch_size=B, grad_clip=0.5, tau=0.05, alpha_min_steps=1,
                     alpha_lr=1e-2, **over)
    actor0, stats0 = OS.init_sac_actor(rng, D, H, A, L, head_scale=0.1, log_std_bias=-1.0)
    critics0 = [OD.init_mlp(rng, D + A, H, M, L) for _ in range(n)]

    class _TQC8(TQCAgent):
        N_CRITICS = 8
    cls = {5: TQCAgent, 8: _TQC8}[n]
    ag = cls(D, A, cfg, None, 1, 2, n_quantiles=M, top_quantiles_to_drop_per_net=drop, precision=precision)
    load_initial(ag, actor0, stats0, critics0)
    orc = None
    if reference:
        orc = R.QuantileTQCOracle(actor0, stats0, critics0, n_quantiles=M, drop_per_net=drop, act_dim=A,
                                  gamma=cfg.gamma, tau=cfg.tau, grad_clip=cfg.grad_clip, actor_lr=cfg.actor_lr,
                                  critic_lr=cfg.critic_lr, alpha_lr=1e-2, alpha_min_steps=1, gradient_step=2)
    return ag, orc, rng


def rand_batch(rng, B, D, A):
    s = rng.standard_normal((B, D)).astype(np.float32)
    ns = (s + 0.1 * rng.standard_normal((B, D))).astype(np.float32)
    a = rng.uniform(-1, 1, (B, A)).astype(np.float32)
    r = -(rng.random((B, 1)) > 0.3).astype(np.float32)
    d = (rng.random((B, 1)) < 0.1).astype(np.float32)
    e1 = rng.standard_normal((B, A)).astype(np.float32)
    e2 = rng.standard_normal((B, A)).astype(np.float32)
    return (s, a, r, ns, d), e1, e2


def run_update(ag, step, batch, e1, e2):
    import torch
    return ag.update(step, batch=tuple(torch.from_numpy(x).cuda() for x in batch),
                     eps_next=torch.from_numpy(e1).cuda(), eps_cur=torch.from_numpy(e2).cuda())


def state(ag):
    p, s = actor_params(ag)
    out = [x for pair in p + s for x in pair]
    for v in ag._critic_views + ag._target_views:
        out += [x for pair in v.layers() for x in pair]
    return out + [np.float32(ag.get_log_alpha())]


def assert_same_bits(xs, ys):
    assert len(xs) == len(ys)
    for i, (x, y) in enumerate(zip(xs, ys)):
        assert np.array_equal(bits(x), bits(y)), i


# The actor's hidden layers (Linears in front of BatchNorm and the BatchNorm affine parameters): their gradient leaves
# the BatchNorm backward, n dxhat - sum dxhat - xhat sum(dxhat xhat), whose three terms cancel to the fp32 rounding of
# the batch sums for many elements at wide layers, and AdamW turns each of those into a step of up to lr in a
# direction the summation order decides.  Measured on a B200 against the reference after 3 updates at B = 512,
# H = 512: 24 % of the first Linear's weights outside tests.helpers.weights_close with quantile critics -- and 46 %
# with the scalar TQC critics on the same inputs (the existing suite holds no actor weight of that path at such
# shapes either).
def assert_within_adam_bound(ag, orc, lr, n):
    """Every tensor within Adam's hard bound of the reference: the actor's hidden layers (above) carry AdamW's
    sign-regime noise, and it reaches the critics through the sampled actions; gradient entries of the critics at the
    fp32 noise level of their batch sums do the same on their own (measured on a B200: a few hundred elements of a
    512 x 25 first critic layer after one update at B = 512, H = 512).  The metrics of every step, which carry every
    loss, gradient norm, TD error and Q value, stay at the stated tolerance."""
    params, _ = actor_params(ag)
    mine = [x for pair in params for x in pair]
    ref = [x for pair in orc.actor for x in pair]
    for views, nets in ((ag._critic_views, orc.critics), (ag._target_views, orc.target_critics)):
        for view, net in zip(views, nets):
            mine += [x for pair in view.layers() for x in pair]
            ref += [x for pair in net for x in pair]
    for i, (x, rx) in enumerate(zip(mine, ref)):
        assert x.shape == rx.shape
        bound = 2.0 * lr * n + 1e-5 * float(np.max(np.abs(rx)))
        assert float(np.max(np.abs(np.asarray(x, np.float64) - rx))) <= bound, i
    np.testing.assert_allclose(ag.get_log_alpha(), float(orc.log_alpha), rtol=1e-5, atol=1e-8)


# ---- 1. three updates against the reference ----------------------------------------------------------------------
# (B, H, L, D, A, M, drop, critics).  The target kernel sorts n M keys in a warp at KPL = 1, 2, 4, 8 keys per lane
# (n M up to 32, 64, 128, 256): M = 12 runs KPL 2, M = 51 KPL 8 with a head two 32-wide fp32 tiles tall (d = 50
# keeps K = 5 targets, fewer than a warp's lanes), eight critics of 32 atoms fill the 256 keys and every loss slot.
# B = 10000 is more rows than the 64 x 148 warps of the capped grids of the target and row-mean kernels.
SHAPES = [(33, 64, 1, 7, 1, 5, 0, 5), (256, 256, 3, 21, 3, 25, 2, 5), (512, 512, 3, 22, 4, 25, 2, 5),
          (64, 64, 2, 10, 2, 1, 0, 5), (4608, 64, 2, 10, 2, 25, 2, 5), (256, 64, 2, 10, 2, 12, 2, 5),
          (512, 256, 2, 22, 3, 51, 0, 5), (512, 256, 2, 22, 3, 51, 50, 5), (10000, 64, 2, 10, 2, 25, 2, 5),
          (256, 64, 2, 10, 2, 32, 0, 8)]


@pytest.mark.parametrize("B,H,L,D,A,M,drop,n", SHAPES,
                         ids=[f"B{s[0]}_H{s[1]}_M{s[5]}_d{s[6]}" + (f"_n{s[7]}" if s[7] != 5 else "") for s in SHAPES])
def test_updates_match_reference(B, H, L, D, A, M, drop, n):
    """Actor and alpha steps included (alpha from step 2); M = 1 is the quantile rule with one atom (tau 0.5, Huber),
    not the scalar MSE path; B = 4608 runs the per-critic backward above the ensemble's batch limit."""
    ag, orc, rng = make_pair(B, H, L, D, A, M, drop, n=n)
    for step in (1, 2, 3):
        batch, e1, e2 = rand_batch(rng, B, D, A)
        want = np.array(orc.update_on_batch(step, *batch, e1, e2), np.float64)
        got = run_update(ag, step, batch, e1, e2)
        assert len(got) == 9
        rtol = 5e-5 * max(1.0, (B / 256.0) ** 0.5)
        np.testing.assert_allclose(np.array([float(x) for x in got]), want, rtol=rtol, atol=2e-6)
        np.testing.assert_allclose(ag.get_log_alpha(), float(orc.log_alpha), rtol=1e-5, atol=1e-8)
    assert_within_adam_bound(ag, orc, ag.config.critic_lr, 3)


# ---- 2. prioritised replay ---------------------------------------------------------------------------------------
def test_prioritised_weights_and_td_rows_match_reference():
    """The batch and importance weights a PER buffer drew: the weighted quantile loss, every metric and the
    per-sample TD array [B, 1] (max over the critics of |mean_k Z - mean_j y|) against the reference."""
    import torch
    from gcrl_b200.parallel import device_tensor
    from tests.test_per_gpu import rand_rows
    B, H, L, D, A, M, drop = 256, 64, 2, 22, 3, 25, 2
    ag, orc, rng = make_pair(B, H, L, D, A, M, drop, buffer_type="PER", max_len=4096, alpha=0.6, beta=0.4,
                             beta_end=100)
    ag.buffer.push_rows(*rand_rows(rng, 3000, D, A))
    for step in (1, 2, 3):
        e1 = torch.randn((B, A), device="cuda")
        e2 = torch.randn((B, A), device="cuda")
        got = ag.update(step, eps_next=e1, eps_cur=e2)
        s, a, r, ns, d = (t.detach().cpu().numpy().astype(np.float32) for t in ag._replay_out)
        w = device_tensor(ag._per_ptrs()[0].value, B, ag.device_index).cpu().numpy().reshape(B, 1)
        assert np.all(w > 0) and (step == 1 or np.ptp(w) > 0)     # new rows enter at the maximum priority
        want = orc.update_on_batch(step, s.reshape(B, D), a.reshape(B, A), r.reshape(B, 1), ns.reshape(B, D),
                                   d.reshape(B, 1), e1.cpu().numpy(), e2.cpu().numpy(), weights=w)
        assert isinstance(got[3], np.ndarray) and got[3].shape == (B, 1)
        np.testing.assert_allclose(got[3], want[3], rtol=5e-5, atol=2e-6)
        rest = [0, 1, 2, 4, 5, 6, 7, 8]
        np.testing.assert_allclose(np.array([float(got[i]) for i in rest]), np.array([float(want[i]) for i in rest]),
                                   rtol=5e-5, atol=2e-6)
    assert_within_adam_bound(ag, orc, ag.config.critic_lr, 3)


# ---- 3. the tensor-core engine -----------------------------------------------------------------------------------
def test_precision2_matches_precision0():
    """B = 2048, H = 256: hidden layers on tcgen05 (precision 2; the quantile head stays on the fp32 tiles) against
    the fp32 engine on the same weights and inputs: metrics of every step at the tensor-core engine's tolerance, the
    weights within Adam's hard bound; tcgen05 kernels ran."""
    from types import SimpleNamespace
    from tests.test_sac_tc_gpu import _tc_kernels_ran
    B, H, L, D, A, M, drop = 2048, 256, 3, 22, 3, 25, 2
    a0, _, rng = make_pair(B, H, L, D, A, M, drop, precision=0, reference=False)
    a2, _, _ = make_pair(B, H, L, D, A, M, drop, precision=2, reference=False)
    lr = a0.config.critic_lr

    def as_ref(ag):
        p, s_ = actor_params(ag)
        return SimpleNamespace(actor=p, actor_stats=s_, critics=[v.layers() for v in ag._critic_views],
                               target_critics=[v.layers() for v in ag._target_views], log_alpha=ag.get_log_alpha())
    for step in (1, 2, 3):
        batch, e1, e2 = rand_batch(rng, B, D, A)
        want = run_update(a0, step, batch, e1, e2)
        box = []
        assert _tc_kernels_ran(lambda: box.append(run_update(a2, step, batch, e1, e2))) > 0
        np.testing.assert_allclose(np.array([float(x) for x in box[0]]), np.array([float(x) for x in want]),
                                   rtol=ENG * 2e-5 * (B / 256.0) ** 0.5, atol=ENG * 1e-6)
    assert_within_adam_bound(a2, as_ref(a0), lr * ENG, 3)


# ---- 4. update_many against the update() loop --------------------------------------------------------------------
def _quantile_agent(B, kind, index_source="host", M=25, drop=2, hidden=64):
    import torch
    from gcrl_b200 import TQCAgent
    max_len = 2 * B + 100
    cfg = sac_config(hidden_dim=hidden, batch_size=B, max_len=max_len, buffer_type=kind, alpha=0.6, ac_update_freq=2,
                     alpha_min_steps=50, alpha_lr=1e-2, actor_lr=1e-3, actor_lr_min=1e-4, ac_scheduler_steps=30,
                     critic_lr=1e-3, critic_lr_min=1e-4, cr_scheduler_steps=25, beta=0.4, beta_end=100)
    torch.manual_seed(5)
    return TQCAgent(22, 3, cfg, None, 1, 40, index_source=index_source, n_quantiles=M,
                    top_quantiles_to_drop_per_net=drop)


@pytest.mark.parametrize("kind,index_source", [("HER", "host"), ("HER", "device"), ("REPLAY", "host"),
                                               ("PER", "host")])
def test_update_many_equals_the_loop_bitwise(kind, index_source, monkeypatch):
    from tests.test_replay_update_many_gpu import buffer_state, push
    from tests.test_sac_update_many_gpu import assert_same_state, episodes_for, loop_vs_many, one_more_update
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    B = 256
    agents = [_quantile_agent(B, kind, index_source) for _ in range(2)]
    for ag in agents:
        if kind == "HER":
            for ep in episodes_for(B):
                ag.buffer.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], ep["fut"])
        else:
            push(ag, 2 * B + 100 + B // 2 + 37, 4)
    a_loop, a_many = agents
    for steps in (list(range(37, 82)), [5, 5, 40, 3]):
        loop_vs_many(a_loop, a_many, steps)
        assert_same_state(a_loop, a_many)
        if kind != "HER":
            for x, y in zip(buffer_state(a_loop), buffer_state(a_many)):
                assert np.array_equal(bits(x), bits(y))
    one_more_update(a_loop, a_many)
    assert_same_state(a_loop, a_many)


# ---- 5. eager launches against graph replay ----------------------------------------------------------------------
@pytest.mark.parametrize("B", [256, 4608])
def test_eager_equals_graph_replay_bitwise(B, monkeypatch):
    H, L, D, A, M, drop = 64, 2, 10, 2, 25, 2
    monkeypatch.setenv("GCRL_B200_NO_GRAPH", "1")
    eager, _, rng = make_pair(B, H, L, D, A, M, drop, reference=False)
    monkeypatch.delenv("GCRL_B200_NO_GRAPH")
    graph, _, _ = make_pair(B, H, L, D, A, M, drop, reference=False)
    for step in (1, 2, 3, 4):
        batch, e1, e2 = rand_batch(rng, B, D, A)
        r1 = run_update(eager, step, batch, e1, e2)
        r2 = run_update(graph, step, batch, e1, e2)
        assert_same_bits([np.float32(x) for x in r1], [np.float32(x) for x in r2])
    assert_same_bits(state(eager), state(graph))


# ---- 6. checkpoints ----------------------------------------------------------------------------------------------
def test_save_weights_round_trip_and_cross_loading_refused(tmp_path):
    import torch
    from gcrl_b200 import TQCAgent
    B, H, L, D, A, M, drop = 128, 64, 2, 10, 2, 25, 2
    ag, _, rng = make_pair(B, H, L, D, A, M, drop, reference=False)
    cfg = ag.config
    fresh = tmp_path / "fresh"
    ag.save_weights(str(fresh))
    sd = torch.load(str(fresh / "critic_0.pth"))
    assert tuple(sd[f"net.{2 * L}.weight"].shape) == (M, H) and tuple(sd[f"net.{2 * L}.bias"].shape) == (M,)
    twin = TQCAgent(D, A, cfg, str(fresh), 1, 2, n_quantiles=M, top_quantiles_to_drop_per_net=drop)
    assert_same_bits(state(ag), state(twin))
    obs = rng.standard_normal((17, D)).astype(np.float32)
    assert_same_bits([ag.select_action(obs, eval_action=True)], [twin.select_action(obs, eval_action=True)])
    batch, e1, e2 = rand_batch(rng, B, D, A)          # the same next update: fresh moments on both sides
    assert_same_bits([np.float32(x) for x in run_update(ag, 1, batch, e1, e2)],
                     [np.float32(x) for x in run_update(twin, 1, batch, e1, e2)])
    assert_same_bits(state(ag), state(twin))
    trained = tmp_path / "trained"
    ag.save_weights(str(trained))
    again = TQCAgent(D, A, cfg, str(trained), 1, 2, n_quantiles=M, top_quantiles_to_drop_per_net=drop)
    for v1, v2 in zip(ag._critic_views, again._critic_views):
        assert_same_bits([x for p in v1.layers() for x in p], [x for p in v2.layers() for x in p])
    assert_same_bits([ag.select_action(obs, eval_action=True)], [again.select_action(obs, eval_action=True)])
    scalar = TQCAgent(D, A, cfg, None, 1, 2)
    scalar_dir = tmp_path / "scalar"
    scalar.save_weights(str(scalar_dir))
    with pytest.raises(ValueError):
        TQCAgent(D, A, cfg, str(scalar_dir), 1, 2, n_quantiles=M)
    with pytest.raises(ValueError):
        TQCAgent(D, A, cfg, str(fresh), 1, 2)
    with pytest.raises(ValueError):
        TQCAgent(D, A, cfg, str(fresh), 1, 2, n_quantiles=M - 1)


# ---- 7. which kernels run ----------------------------------------------------------------------------------------
def test_profiler_sees_the_quantile_kernels_and_no_scalar_target():
    from torch.profiler import ProfilerActivity, profile
    import torch
    B, H, L, D, A, M, drop = 256, 64, 2, 10, 2, 25, 2
    ag, _, rng = make_pair(B, H, L, D, A, M, drop, reference=False)
    batch, e1, e2 = rand_batch(rng, B, D, A)
    run_update(ag, 1, batch, e1, e2)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run_update(ag, 2, batch, e1, e2)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    for k in ("quantile_target_kernel", "quantile_huber_kernel"):
        assert any(k in n for n in names), k
    assert not any("sac_target_kernel" in n for n in names)
    assert not any("actor_trunc_kernel" in n for n in names)


# ---- 8. data parallelism is refused ------------------------------------------------------------------------------
def test_data_parallel_refused():
    from gcrl_b200._lib import ERR_INVALID, lib
    B, H, L, D, A, M, drop = 64, 64, 1, 10, 2, 5, 1
    ag, _, _ = make_pair(B, H, L, D, A, M, drop, reference=False)
    for sync_bn in (True, False):
        with pytest.raises(ValueError, match="quantile"):
            ag.enable_data_parallel(allreduce_mean=lambda t: None, sync_bn=sync_bn, world=1, rank=0)
    st = ag._stream()
    assert lib.gcrl_sac_set_sync_bn(ag._h, 2, 0) == ERR_INVALID
    assert b"quantile" in lib.gcrl_last_error()
    nul = (None,) * 5
    assert lib.gcrl_sac_update_phase(ag._h, 0, None, B, None, *nul, None, None, 1e-3, 1e-3, 1, st) == ERR_INVALID
    assert b"quantile" in lib.gcrl_last_error()
    coll = C.c_int(0)
    assert lib.gcrl_sac_update_segment(ag._h, 0, None, B, None, *nul, None, None, 1e-3, 1e-3, 1, C.byref(coll),
                                       st) == ERR_INVALID
    assert b"quantile" in lib.gcrl_last_error()
    # the agent still trains
    rng = np.random.default_rng(1)
    batch, e1, e2 = rand_batch(rng, B, D, A)
    assert all(np.isfinite(float(x)) for x in run_update(ag, 1, batch, e1, e2))

"""GPU parity: the DDPG update (csrc/agent.cu, mlp.cu, optim.cu) through the C ABI versus
fixtures dumped from the unmodified reference ``DDPG.update`` (src/agent.py:1378-1404) and
versus the NumPy oracle.

Tolerance (north_star: "within a stated fp32 tolerance (e.g. rel 1e-5)"):
  metrics (losses, td, q, grad norms)   rel 2e-5 + abs 1e-6
  Bellman targets y, Q                  rel 1e-5 (norm-wise) per tensor
  post-update weights                   tests.helpers.weights_close (rel 1e-5 norm-wise + Adam
                                        eps-regime allowance, documented there)
"""
import types

import numpy as np
import pytest

from oracle import ddpg as OD
from tests.helpers import (DDPG_CASES, DDPG_LARGE_CASES, ddpg_params_from_golden, golden_update_inputs, load, rel_err,
                           weight_error_report, weights_close)

pytestmark = pytest.mark.gpu


def make_config(g=None, **over):
    base = dict(hidden_dim=64, layer_count=3, actor_lr=1e-3, actor_lr_min=1e-3, ac_scheduler_steps=1,
                critic_lr=1e-3, critic_lr_min=1e-3, cr_scheduler_steps=1, buffer_type="HER",
                max_len=100000, alpha=1.0, batch_size=64, gamma=0.98, ac_update_freq=1, noise_std=0.2,
                noise_clamp=0.5, policy_noise=0.2, grad_clip=10.0, beta=1.0, beta_end=1, k_future=4,
                max_eps_len=50, tau=0.05)
    if g is not None:
        D, A, H, L, B, seed, ac_T, cr_T, freq = (int(x) for x in g["meta"])
        gamma, tau, clip, alr, clr, alr_min, clr_min = (float(x) for x in g["hp"])
        base.update(hidden_dim=H, layer_count=L, batch_size=B, gamma=gamma, tau=tau, grad_clip=clip,
                    actor_lr=alr, critic_lr=clr, actor_lr_min=alr_min, critic_lr_min=clr_min,
                    ac_scheduler_steps=ac_T, cr_scheduler_steps=cr_T, ac_update_freq=freq)
    base.update(over)
    return types.SimpleNamespace(**base)


def make_agent_from_golden(g):
    from gcrl_b200 import DDPG
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC
    D, A, H, L, B, seed = (int(x) for x in g["meta"][:6])
    ag = DDPG(D, A, make_config(g), None, 1, 40)
    rng = np.random.default_rng(seed)
    actor0 = OD.init_mlp(rng, D, H, A, L)
    critic0 = OD.init_mlp(rng, D + A, H, 1, L)
    ag._set_layers(NET_ACTOR, actor0)
    ag._set_layers(NET_CRITIC, critic0)
    ag.update_target_network()
    return ag, rng


def batch_to_device(g, si):
    import torch
    return tuple(torch.from_numpy(g[f"s{si}_batch_{k}"]).cuda() for k in ("s", "a", "r", "ns", "d"))


@pytest.mark.parametrize("case", DDPG_CASES)
def test_update_matches_reference_fixture(case):
    g = load("ddpg_" + case)
    ag, _ = make_agent_from_golden(g)
    lr = max(float(g["hp"][3]), float(g["hp"][4]))
    for si, step in enumerate(g["steps"]):
        info = ag.update(int(step), batch=batch_to_device(g, si))
        ref = g[f"s{si}_info"]
        assert len(info) == len(ref), "tuple arity (6 with the actor step, else 4)"
        np.testing.assert_allclose(np.array([float(x) for x in info]), ref, rtol=2e-5, atol=1e-6)
        np.testing.assert_allclose([ag.critic_scheduler.lr, ag.actor_scheduler.lr], g[f"s{si}_lr"],
                                   rtol=1e-12)
        if f"s{si}_actor.base_net.0.weight" in g.files:
            for tag, net in (("actor", ag.actor), ("critic", ag.critic),
                             ("target_actor", ag.target_actor), ("target_critic", ag.target_critic)):
                for (w, b), (rw, rb) in zip(net.layers(), ddpg_params_from_golden(g, si, tag)):
                    assert weights_close(w, rw, lr, si + 1), (case, si, tag, rel_err(w, rw))
                    assert weights_close(b, rb, lr, si + 1), (case, si, tag, rel_err(b, rb))


@pytest.mark.parametrize("precision", [1, 0])
@pytest.mark.parametrize("case", DDPG_LARGE_CASES)
def test_large_batch_update_matches_reference_fixture(case, precision, capsys):
    """Batches of 2048 and 8192 on the PickAndPlace shape against the UNMODIFIED reference (fixtures written by
    tests/golden/make_golden.py::large_batch_cases; batches regenerated from the seed and pinned by checksum):
    the default agent (precision 1: hidden-layer GEMMs on tcgen05 with the 3xTF32 split) and the fp32 FFMA tile
    engine (precision 0).  Metrics every step (batch means over B terms: rel 2e-5 * sqrt(B / 256)), all four
    networks after the last step (weights_close); the observed errors are printed."""
    import torch
    from gcrl_b200 import DDPG
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC
    g = load("ddpg_" + case)
    D, A, H, L, B, seed = (int(x) for x in g["meta"][:6])
    (actor0, critic0), batches = golden_update_inputs(g)
    ag = DDPG(D, A, make_config(g), None, 1, 40, precision=precision)
    ag._set_layers(NET_ACTOR, actor0)
    ag._set_layers(NET_CRITIC, critic0)
    ag.update_target_network()
    # The oracle runs alongside ONLY to bound the conditioning of this batch: LeakyReLU' jumps at 0, so hidden
    # units whose pre-activation is zero to the engine's rounding (fp32 tiles ~5e-7, 3xTF32 ~2e-6 per layer; the
    # deltas below are ~10x that) may take either slope, which moves the gradient norms (slack) and, through
    # Adam, individual weights (per-element allowance) -- oracle/ddpg.py::_flip_track.  Everything else is held
    # to the reference's own numbers.
    cfg = make_config(g)
    orc = OD.DDPGOracle([[w.copy(), b.copy()] for w, b in actor0], [[w.copy(), b.copy()] for w, b in critic0],
                        gamma=cfg.gamma, tau=cfg.tau, grad_clip=cfg.grad_clip, actor_lr=cfg.actor_lr, critic_lr=cfg.critic_lr)
    orc.flip_delta = 2e-5 if precision else 5e-6
    rtol = 2e-5 * max(1.0, (B / 256.0) ** 0.5)
    n = len(g["steps"])
    worst = 0.0
    lines = []
    failures = []
    critic_flips = False
    for si, step in enumerate(g["steps"]):
        info = ag.update(int(step), batch=tuple(torch.from_numpy(x).cuda() for x in batches[si]))
        orc.update_on_batch(int(step), *batches[si])
        got, ref = np.array([float(x) for x in info]), g[f"s{si}_info"]
        assert len(got) == len(ref)
        rel = np.abs(got - ref) / (np.abs(ref) + 1e-6)
        tol = np.full(len(ref), rtol)
        tol[4] += orc.last_critic_flip_slack           # critic gradient norm
        tol[5] += orc.last_actor_flip_slack            # actor gradient norm
        critic_flips = critic_flips or orc.last_critic_flip_slack > 0
        lines.append(f"  step {int(step)}: metric rel errors " + " ".join(f"{x:.1e}" for x in rel) +
                     f"   (flip slack: critic norm {orc.last_critic_flip_slack:.1e}, actor norm {orc.last_actor_flip_slack:.1e})")
        worst = max(worst, float(rel[:4].max()))
        if not np.all(np.abs(got - ref) <= tol * np.abs(ref) + 1e-6):
            failures.append((int(step), got.tolist(), ref.tolist(), tol.tolist()))
    lr = max(float(g["hp"][3]), float(g["hp"][4]))
    lines.insert(0, f"{case} precision={precision}: worst loss / td / q rel err {worst:.2e} (allowed {rtol:.2e})")
    for tag, net in (("actor", ag.actor), ("critic", ag.critic), ("target_actor", ag.target_actor),
                     ("target_critic", ag.target_critic)):
        allow = orc.flip_allowance if "actor" in tag else orc.flip_allowance_critic
        scale = cfg.tau * n if tag.startswith("target") else 1.0           # Polyak passes at most tau per step on
        for li, ((w, b), (rw, rb)) in enumerate(zip(net.layers(), ddpg_params_from_golden(g, n - 1, tag))):
            mx, p9999, tol, used = weight_error_report(w, rw, lr, n)
            lines.append(f"  {tag}.{li}.weight: max {mx:.2e}, 99.99 % {p9999:.2e}, base allowance {tol:.2e} ({100 * used:.1f} % used), "
                         f"median flip allowance {float(np.median(allow[li][0])) * scale:.1e}")
            frac = 5e-3 if ("actor" in tag and critic_flips) else 2e-4     # indirect effect of the stepped critic, see the odd-shape test
            if not (weights_close(w, rw, lr, n, extra=allow[li][0] * scale, outlier_frac=frac) and
                    weights_close(b, rb, lr, n, extra=allow[li][1] * scale, outlier_frac=frac)):
                failures.append((tag, li, rel_err(w, rw), rel_err(b, rb)))
    with capsys.disabled():
        print("\n" + "\n".join(lines))
    assert not failures, failures


@pytest.mark.parametrize("B,H,L,D,A", [(1, 64, 3, 10, 3), (33, 100, 2, 22, 3), (1000, 256, 3, 23, 4),
                                       (4096, 512, 3, 22, 3), (777, 64, 1, 7, 1),
                                       # one batch per rows-per-CTA variant of the row-slab kernels (148 SMs),
                                       # each with a ragged last slab: R = 4; R = 8 as 2-CTA clusters; R = 8
                                       (301, 256, 3, 21, 3), (517, 256, 3, 21, 3), (1021, 256, 3, 21, 3),
                                       # R = 8 at H = 512: 194.5 KB of shared memory, the largest that fits
                                       (517, 512, 3, 21, 3),
                                       # K0 = 27 padded to 28; H = 100 leaves one column warp (16-way K split)
                                       (301, 100, 2, 23, 4)])
def test_update_matches_oracle_odd_shapes(B, H, L, D, A):
    """Ragged shapes (B not a tile multiple, H not a multiple of 16, A in 1..4), 4 updates
    spanning a Polyak step, versus the NumPy oracle on identical weights and batches."""
    import torch
    from gcrl_b200 import DDPG
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC
    rng = np.random.default_rng(B * 7 + H)
    cfg = make_config(hidden_dim=H, layer_count=L, batch_size=B, grad_clip=0.5, tau=0.05)
    ag = DDPG(D, A, cfg, None, 1, 40, precision=0)
    actor0, critic0 = OD.init_mlp(rng, D, H, A, L), OD.init_mlp(rng, D + A, H, 1, L)
    ag._set_layers(NET_ACTOR, actor0)
    ag._set_layers(NET_CRITIC, critic0)
    ag.update_target_network()
    orc = OD.DDPGOracle(actor0, critic0, gamma=cfg.gamma, tau=cfg.tau, grad_clip=cfg.grad_clip,
                        actor_lr=cfg.actor_lr, critic_lr=cfg.critic_lr)
    orc.flip_delta = 5e-6
    critic_flips = False
    for si, step in enumerate((39, 40, 41, 42)):
        s = rng.standard_normal((B, D)).astype(np.float32)
        ns = (s + 0.1 * rng.standard_normal((B, D))).astype(np.float32)
        a = rng.uniform(-1, 1, (B, A)).astype(np.float32)
        r = -(rng.random((B, 1)) > 0.3).astype(np.float32)
        d = (rng.random((B, 1)) < 0.1).astype(np.float32)
        want = orc.update_on_batch(step, s, a, r, ns, d)
        got = ag.update(step, batch=tuple(torch.from_numpy(x).cuda() for x in (s, a, r, ns, d)))
        # batch means / gradient norms are fp32 sums over B terms evaluated in a different order than
        # BLAS: the summation-order noise grows like sqrt(B) (rel 5e-5 at B <= 256)
        rtol = np.full(6, 5e-5 * max(1.0, (B / 256.0) ** 0.5))
        # actor gradient norm: plus the oracle's own bound for hidden units whose pre-activation
        # is zero to fp32 rounding (LeakyReLU' jumps there; oracle/ddpg.py::_actor_flip_slack)
        rtol[5] += orc.last_actor_flip_slack
        rtol[4] += orc.last_critic_flip_slack
        critic_flips = critic_flips or orc.last_critic_flip_slack > 0
        got, want = np.array([float(x) for x in got]), np.array(want)
        assert np.all(np.abs(got - want) <= rtol * np.abs(want) + 2e-6), (step, got, want, rtol)
    # A LeakyReLU sign flip of a pre-activation that is zero to fp32 rounding changes one batch row's whole
    # gradient contribution; Adam's per-element normalisation amplifies that for the small-gradient elements.
    # The oracle bounds the effect PER ELEMENT (DDPGOracle._flip_track: the rows it saw within flip_delta of
    # zero, carried through Adam's moments); every other element stays under weights_close's own tolerance.
    n = 4
    for name, net, ref in (("actor", ag.actor, orc.actor), ("critic", ag.critic, orc.critic),
                           ("target_actor", ag.target_actor, orc.target_actor),
                           ("target_critic", ag.target_critic, orc.target_critic)):
        allow = orc.flip_allowance if "actor" in name else orc.flip_allowance_critic
        scale = cfg.tau * n if name.startswith("target") else 1.0          # Polyak passes at most tau per step on
        # The actor's gradient also depends on the STEPPED critic: where the critic's own weights moved inside their
        # flip allowance, the actor's small-gradient elements can change Adam direction -- an indirect effect the
        # per-element bound does not carry; those few elements (<= 0.5 %) are held to Adam's hard bound only.
        frac = 5e-3 if ("actor" in name and critic_flips) else 2e-4
        for li, ((w, b), (rw, rb)) in enumerate(zip(net.layers(), ref)):
            ew, eb = allow[li][0] * scale, allow[li][1] * scale
            assert weights_close(w, rw, 1e-3, n, extra=ew, outlier_frac=frac), (name, li, rel_err(w, rw))
            assert weights_close(b, rb, 1e-3, n, extra=eb, outlier_frac=frac), (name, li, rel_err(b, rb))


@pytest.mark.parametrize("B,H,L,D,A", [(2048, 256, 3, 21, 3), (5000, 64, 2, 23, 4), (1100, 512, 3, 22, 3)])
def test_tensor_core_update_matches_fp32_update(B, H, L, D, A, monkeypatch, capsys):
    """precision=2 (tcgen05, 3xTF32 split, forced for small batches) versus precision=0 (fp32 FFMA) on identical weights and
    batches, and versus the NumPy oracle: metrics rel 5e-5 * sqrt(B/256) like the fp32 path.  The first update of each
    agent runs under torch.profiler, which must show that engine's kernels."""
    import torch
    from gcrl_b200 import DDPG
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC
    from tests.test_engine_edges_gpu import check_engine
    from tests.test_fused_variants_gpu import launched_kernels
    monkeypatch.setenv("GCRL_B200_NO_GRAPH", "1")          # read at creation: every kernel a launch of its own
    rng = np.random.default_rng(B + H)
    cfg = make_config(hidden_dim=H, layer_count=L, batch_size=B, grad_clip=0.5, tau=0.05)
    actor0, critic0 = OD.init_mlp(rng, D, H, A, L), OD.init_mlp(rng, D + A, H, 1, L)
    agents = []
    for precision in (0, 2):
        ag = DDPG(D, A, cfg, None, 1, 40, precision=precision)
        ag._set_layers(NET_ACTOR, actor0)
        ag._set_layers(NET_CRITIC, critic0)
        ag.update_target_network()
        agents.append(ag)
    orc = OD.DDPGOracle(actor0, critic0, gamma=cfg.gamma, tau=cfg.tau, grad_clip=cfg.grad_clip,
                        actor_lr=cfg.actor_lr, critic_lr=cfg.critic_lr)
    # pre-activations carry ~2e-6 relative error per 3xTF32 layer (fp32 tiles: 5e-7), so units within
    # 2e-5 of zero may take either LeakyReLU slope (oracle/ddpg.py::_actor_flip_slack)
    orc.flip_delta = 2e-5
    rtol = np.full(6, 5e-5 * max(1.0, (B / 256.0) ** 0.5))
    steps = (39, 40, 41)     # the step-40 Polyak update in the middle
    critic_flips = False
    for si, step in enumerate(steps):
        s = rng.standard_normal((B, D)).astype(np.float32)
        ns = (s + 0.1 * rng.standard_normal((B, D))).astype(np.float32)
        a = rng.uniform(-1, 1, (B, A)).astype(np.float32)
        r = -(rng.random((B, 1)) > 0.3).astype(np.float32)
        d = (rng.random((B, 1)) < 0.1).astype(np.float32)
        want = np.array(orc.update_on_batch(step, s, a, r, ns, d))
        tol = rtol.copy() * (si + 1)          # the three implementations drift apart step by step
        tol[5] += orc.last_actor_flip_slack
        tol[4] += orc.last_critic_flip_slack
        critic_flips = critic_flips or orc.last_critic_flip_slack > 0
        batch = tuple(torch.from_numpy(x).cuda() for x in (s, a, r, ns, d))
        got = []
        for ag, engine, precision in zip(agents, ("tiles", "tc"), (0, 2)):
            info = []
            names = launched_kernels(lambda: info.extend(ag.update(step, batch=batch)))
            if si == 0:
                check_engine(names, engine, f"DDPG B={B} H={H} precision={precision}", capsys)
            got.append(np.array([float(x) for x in info]))
        for g in got:
            assert np.all(np.abs(g - want) <= tol * np.abs(want) + 2e-6), (step, g, want, tol)
    # post-update weights of all four networks: tensor cores vs fp32 tiles vs oracle.  The critic carries no
    # LeakyReLU-flip sensitivity beyond weights_close; the actor's allowance is per element (flip_allowance)
    n = len(steps)
    fp32, tc = agents
    for name, a0, a1, ref in (("actor", fp32.actor, tc.actor, orc.actor), ("critic", fp32.critic, tc.critic, orc.critic),
                              ("target_actor", fp32.target_actor, tc.target_actor, orc.target_actor),
                              ("target_critic", fp32.target_critic, tc.target_critic, orc.target_critic)):
        extra = orc.flip_allowance if "actor" in name else orc.flip_allowance_critic
        scale = cfg.tau * n if name.startswith("target") else 1.0      # Polyak passes at most tau per step on
        frac = 5e-3 if ("actor" in name and critic_flips) else 2e-4     # indirect effect of the stepped critic, see the odd-shape test
        for li, ((w0, b0), (w1, b1), (rw, rb)) in enumerate(zip(a0.layers(), a1.layers(), ref)):
            ew, eb = extra[li][0] * scale, extra[li][1] * scale
            # the 3xTF32 engine's stated tolerance is 4x the fp32 engine's (~2e-6 vs ~5e-7 relative error per layer)
            kw = dict(rtol=4e-5, extra=None, outlier_frac=frac)
            assert weights_close(w1, rw, 4e-3, n, **{**kw, "extra": ew}), (name, li, "tc vs oracle")
            assert weights_close(b1, rb, 4e-3, n, **{**kw, "extra": eb}), (name, li, "tc vs oracle")
            assert weights_close(w1, w0, 4e-3, n, **{**kw, "extra": ew}), (name, li, "tc vs fp32")
            assert weights_close(b1, b0, 4e-3, n, **{**kw, "extra": eb}), (name, li, "tc vs fp32")


def test_checkpoint_load_and_forward_matches_reference():
    """state_dict key names / layout of the shipped Reach checkpoint (src/model.py:32-37) and
    actor / critic forward versus the reference's own outputs."""
    import torch
    from gcrl_b200 import DDPG
    g = load("checkpoint_reach")
    ag = DDPG(10, 3, make_config(hidden_dim=64, layer_count=3, batch_size=64), None, 1, 40)
    ag.actor.load_state_dict({k[6:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("actor.")})
    ag.critic.load_state_dict({k[7:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("critic.")})
    act = ag._actor_forward(g["x"])
    np.testing.assert_allclose(act, g["act"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(ag.q_values(g["x"], act), g["q"], rtol=1e-5, atol=1e-6)
    sd = ag.actor.state_dict()
    assert sorted(sd) == sorted(k[6:] for k in g.files if k.startswith("actor."))
    for k, v in sd.items():
        assert np.array_equal(v.numpy(), g["actor." + k])
    # eval-mode select_action applies the reference's second tanh (src/agent.py:1364-1366)
    np.testing.assert_allclose(ag.select_action(g["x"], eval_action=True), np.tanh(g["act"]), rtol=1e-5,
                               atol=1e-6)


def test_save_weights_round_trip(tmp_path):
    import torch
    from gcrl_b200 import DDPG
    ag = DDPG(10, 3, make_config(), None, 1, 40)
    ag.save_weights(str(tmp_path / "w"))
    sd = torch.load(str(tmp_path / "w" / "actor.pth"))
    assert list(sd) == [f"base_net.{i}.{p}" for i in (0, 2, 4, 6) for p in ("weight", "bias")]
    sc = torch.load(str(tmp_path / "w" / "critic.pth"))
    assert list(sc) == [f"net.{i}.{p}" for i in (0, 2, 4, 6) for p in ("weight", "bias")]
    ag2 = DDPG(10, 3, make_config(), str(tmp_path / "w"), 1, 40)
    for (w, b), (w2, b2) in zip(ag.actor.layers() + ag.critic.layers(), ag2.actor.layers() + ag2.critic.layers()):
        assert np.array_equal(w, w2) and np.array_equal(b, b2)
    for (w, b), (w2, b2) in zip(ag2.actor.layers(), ag2.target_actor.layers()):
        assert np.array_equal(w, w2) and np.array_equal(b, b2)         # hard sync at init (:1251-1253)


def synthetic_episodes(seed, n, D, A, G, T=50, k=4):
    """Seeded episodes in the layout of tests.helpers.her_episodes: the last G state features are the desired
    goal, ``fut`` holds apply_her's future offsets (randint(t + 1, T - 1), k per step)."""
    rng = np.random.default_rng(seed)
    eps = []
    for _ in range(n):
        obs = rng.standard_normal((T + 1, D)).astype(np.float32)
        ag = np.cumsum(rng.normal(0, 0.05, (T + 1, G)), 0).astype(np.float32)
        fut = np.zeros((T, k), np.uint8)
        for t in range(T - 1):
            fut[t] = rng.integers(t + 1, T, k)
        eps.append({"s": obs[:-1], "a": rng.uniform(-1, 1, (T, A)).astype(np.float32), "ns": obs[1:],
                    "r": -(rng.random(T) > 0.2).astype(np.float32), "d": np.zeros(T, np.float32),
                    "ag": ag[1:], "fut": fut})
    return eps


def test_update_from_buffer_equals_sample_then_update():
    """The fused sample+update call == sample() followed by update(batch) on the same indices,
    bit for bit (same kernels, same order)."""
    from gcrl_b200 import DDPG
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC
    from tests.helpers import her_episodes
    g = load("her_push_evict")
    D, A = 22, 3
    agents = []
    for _ in range(2):
        ag = DDPG(D, A, make_config(hidden_dim=64, batch_size=128, max_len=777), None, 1, 40)
        rng = np.random.default_rng(1)
        ag._set_layers(NET_ACTOR, OD.init_mlp(rng, D, 64, A, 3))
        ag._set_layers(NET_CRITIC, OD.init_mlp(rng, D + A, 64, 1, 3))
        ag.update_target_network()
        for ep in her_episodes(g):
            ag.buffer.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], ep["fut"])
        agents.append(ag)
    rng = np.random.default_rng(2)
    for step in (39, 40, 41):
        idx = rng.permutation(len(agents[0].buffer))[:128]
        i1 = agents[0].update(step, indices=idx)
        i2 = agents[1].update(step, batch=agents[1].buffer.sample(128, indices=idx))
        assert [float(x) for x in i1] == [float(x) for x in i2]
    for n1, n2 in ((agents[0].actor, agents[1].actor), (agents[0].critic, agents[1].critic)):
        for (w, b), (w2, b2) in zip(n1.layers(), n2.layers()):
            assert np.array_equal(w, w2) and np.array_equal(b, b2)


@pytest.mark.parametrize("B,algo", [(128, "td3"), (301, "ddpg"), (301, "td3"), (517, "ddpg"), (517, "td3"),
                                    (1021, "ddpg"), (1021, "td3")])
def test_update_from_buffer_equals_sample_then_update_every_variant(B, algo):
    """test_update_from_buffer_equals_sample_then_update (B = 128, DDPG) at the batches that reach every
    rows-per-CTA variant of the critic kernel's in-kernel sampler (148 SMs: R = 2, 4, 8 as 2-CTA clusters, 8 with
    a ragged last slab), for DDPG and TD3: bit for bit in metrics and in the weights of every network.  TD3's
    critic-2 launch reuses the dense batch the critic-1 launch drew, and both agents get the same noise."""
    import torch
    from gcrl_b200 import DDPG, TD3Agent
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC, NET_CRITIC2
    from tests.helpers import her_episodes
    D, A, G = 22, 3, 3
    if B <= 777:
        episodes, max_len = her_episodes(load("her_push_evict")), 777
    else:             # the fixture's store is too small: seeded episodes, pushed until the store has evicted
        max_len = 2 * B + 100
        episodes = synthetic_episodes(B, max_len // 200 + 3, D, A, G)        # ~250 entries each (T = 50, k = 4)
    cls = DDPG if algo == "ddpg" else TD3Agent
    agents = []
    for _ in range(2):
        cfg = make_config(hidden_dim=64, batch_size=B, max_len=max_len, ac_update_freq=1 if algo == "ddpg" else 2)
        ag = cls(D, A, cfg, None, 1, 40)
        rng = np.random.default_rng(1)
        ag._set_layers(NET_ACTOR, OD.init_mlp(rng, D, 64, A, 3))
        ag._set_layers(NET_CRITIC, OD.init_mlp(rng, D + A, 64, 1, 3))
        if algo == "td3":
            ag._set_layers(NET_CRITIC2, OD.init_mlp(rng, D + A, 64, 1, 3))
        ag.update_target_network()
        growth = []
        for ep in episodes:
            n = len(ag.buffer)
            ag.buffer.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], ep["fut"])
            growth.append(len(ag.buffer) - n)
        # synthetic episodes all add the same number of entries until the store is full and evicts
        assert len(ag.buffer) >= B and (B <= 777 or (min(growth) < max(growth) and len(ag.buffer) >= 2 * B))
        agents.append(ag)
    rng = np.random.default_rng(2)
    for step in (39, 40, 41):
        idx = rng.permutation(len(agents[0].buffer))[:B]
        kw = {"noise": torch.randn((B, A), device="cuda")} if algo == "td3" else {}
        i1 = agents[0].update(step, indices=idx, **kw)
        i2 = agents[1].update(step, batch=agents[1].buffer.sample(B, indices=idx), **kw)
        assert [float(x) for x in i1] == [float(x) for x in i2]
    for n1, n2 in zip(agents[0]._all_nets(), agents[1]._all_nets()):
        for (w, b), (w2, b2) in zip(agents[0]._get_layers(n1), agents[1]._get_layers(n2)):
            assert np.array_equal(w, w2) and np.array_equal(b, b2)


def test_update_is_deterministic_run_to_run():
    import torch
    g = load("ddpg_push_h256")
    outs = []
    for _ in range(2):
        ag, _ = make_agent_from_golden(g)
        infos = [ag.update(int(step), batch=batch_to_device(g, si)) for si, step in enumerate(g["steps"])]
        outs.append((infos, [w.copy() for w, _ in ag.critic.layers() + ag.actor.layers()]))
    assert [[float(x) for x in i] for i in outs[0][0]] == [[float(x) for x in i] for i in outs[1][0]]
    for w1, w2 in zip(outs[0][1], outs[1][1]):
        assert np.array_equal(w1, w2)
    torch.cuda.synchronize()


def test_predrawn_host_indices_keep_the_reference_random_stream():
    """update() pre-draws the next call's positions while the GPU works; every consumer of the global
    ``random`` stream must still see exactly the reference's interleaving of sample / randint / random."""
    import random
    from gcrl_b200 import DDPG
    from tests.helpers import her_episodes
    g = load("her_reach_small")
    ag = DDPG(10, 3, make_config(batch_size=32, max_len=100000), None, 2, 40)
    eps = her_episodes(g)
    for ep in eps[:6]:
        ag.buffer.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], ep["fut"])
    random.seed(7)
    expect_rng = random.Random(7)
    n = len(ag.buffer)
    seen = []
    real_take = ag._take_predrawn
    ag._take_predrawn = lambda B: seen.append(list(real_take(B))) or seen[-1]
    script = ["u", "u", "r", "u", "p", "u", "u", "r", "r", "u"]
    step = 1
    for op in script:
        if op == "u":
            ag.update(step)
            step += 1
            assert seen[-1] == expect_rng.sample(range(n), 32)
        elif op == "r":                      # another consumer (select_action's random.random, :1348)
            assert random.random() == expect_rng.random()
        else:                                # an episode commit changes len(buffer): the pre-draw is void
            ep = eps[6]
            ag.buffer.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], ep["fut"])
            n = len(ag.buffer)
    assert random.random() == expect_rng.random()


@pytest.mark.parametrize("algo", ["ddpg", "td3"])
def test_true_resume_is_bit_identical(tmp_path, algo):
    """save_checkpoint / load_checkpoint (weights, targets, Adam moments + step counts, schedulers): a
    resumed agent makes bit-identical updates; the reference's own checkpoint (weights only) cannot."""
    import torch
    from gcrl_b200 import DDPG, TD3Agent
    cls = DDPG if algo == "ddpg" else TD3Agent
    D, A, B = 22, 3, 128
    cfg = make_config(hidden_dim=64, batch_size=B, actor_lr=1e-3, actor_lr_min=1e-4, ac_scheduler_steps=5,
                      critic_lr=2e-3, critic_lr_min=5e-4, cr_scheduler_steps=3, ac_update_freq=2)
    rng = np.random.default_rng(11)

    def batch():
        s = rng.standard_normal((B, D)).astype(np.float32)
        return tuple(torch.from_numpy(x).cuda() for x in (
            s, rng.uniform(-1, 1, (B, A)).astype(np.float32), -(rng.random((B, 1)) > 0.3).astype(np.float32),
            (s + 0.1 * rng.standard_normal((B, D))).astype(np.float32), (rng.random((B, 1)) < 0.1).astype(np.float32)))
    batches = [batch() for _ in range(8)]
    noises = [torch.randn((B, A), device="cuda") for _ in range(8)]
    kw = (lambda i: {"noise": noises[i]}) if algo == "td3" else (lambda i: {})
    torch.manual_seed(5)
    a1 = cls(D, A, cfg, None, 1, 40)
    for i in range(4):
        a1.update(37 + i, batch=batches[i], **kw(i))
    a1.save_checkpoint(str(tmp_path / "ck"))
    ref = [a1.update(41 + i, batch=batches[4 + i], **kw(4 + i)) for i in range(4)]
    torch.manual_seed(99)                                   # different initial weights: everything must come from the file
    a2 = cls(D, A, cfg, None, 1, 40)
    a2.load_checkpoint(str(tmp_path / "ck"))
    got = [a2.update(41 + i, batch=batches[4 + i], **kw(4 + i)) for i in range(4)]
    assert [[float(x) for x in r] for r in ref] == [[float(x) for x in g] for g in got]
    for n1, n2 in zip((a1.actor, a1.target_actor), (a2.actor, a2.target_actor)):
        for (w, b), (w2, b2) in zip(n1.layers(), n2.layers()):
            assert np.array_equal(w, w2) and np.array_equal(b, b2)


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["ddpg", "td3"])
def test_exploration_select_action_consumes_the_reference_generators(algo):
    """select_action(eval_action=False), src/agent.py:1345-1360 (DDPG) / :253-263 (TD3): DDPG first draws
    random.random() and, below 0.2, returns clip(np.random.randn(n, A)); otherwise both add
    np.random.normal(0, noise_std) to the (DDPG: twice-tanh'd) actor output and clip.  Seeded alike, the product
    must consume both global generators exactly like that and return those values."""
    import random
    from gcrl_b200 import DDPG, TD3Agent
    cls = DDPG if algo == "ddpg" else TD3Agent
    D, A, n = 10, 3, 5
    ag = cls(D, A, make_config(hidden_dim=64, layer_count=3, batch_size=64, noise_std=0.3), None, 1, 40)
    rng = np.random.default_rng(2)
    xs = [rng.standard_normal((n, D)).astype(np.float32) for _ in range(40)]
    det = [np.asarray(ag.select_action(x, eval_action=True)) for x in xs]       # consumes no generator
    random.seed(11)
    np.random.seed(11)
    got = [np.asarray(ag.select_action(x)) for x in xs]
    end_state = (random.random(), np.random.random_sample())
    random.seed(11)
    np.random.seed(11)
    branches = 0
    for x, d_, g_ in zip(xs, det, got):
        if algo == "ddpg" and random.random() < 0.2:
            want = np.clip(np.random.randn(n, A), a_min=-1, a_max=1)
            branches += 1
        else:
            # DDPG's eval output carries the reference's second tanh; TD3's is the raw actor output, tanh'd here
            base = d_ if algo == "ddpg" else np.tanh(d_)
            want = np.clip(base + np.random.normal(0, 0.3, size=base.shape), -1, 1)
        np.testing.assert_allclose(g_, want, rtol=1e-6, atol=1e-6)
    assert (random.random(), np.random.random_sample()) == end_state
    assert algo == "td3" or 0 < branches < 40


def test_failed_update_leaves_step_counters_untouched():
    """An update that fails (under-filled buffer; TD3 without its noise tensor) must not advance Adam's step
    counters: the Python schedulers do not step on an exception either, and every later bias correction would
    be off by one (csrc/agent.cu::AdamStepGuard)."""
    import ctypes as C
    from gcrl_b200 import DDPG
    from gcrl_b200._lib import GcrlError, check, lib
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC
    from tests.helpers import her_episodes
    ag = DDPG(10, 3, make_config(batch_size=64, max_len=100000), None, 2, 40, index_source="device")
    ep = her_episodes(load("her_reach_small"))[2]                  # a 7-step episode: 31 entries < 64
    ag.buffer.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], ep["fut"])

    def steps():
        out = []
        for net in (NET_ACTOR, NET_CRITIC):
            t = C.c_int()
            check(lib.gcrl_agent_get_adam_step(ag._h, net, C.byref(t)))
            out.append(t.value)
        return out

    before, lr_before = steps(), (ag.critic_scheduler.last_epoch, ag.actor_scheduler.last_epoch)
    with pytest.raises((AssertionError, GcrlError)):
        ag.update(1)
    with pytest.raises((AssertionError, GcrlError)):          # GCRL_ERR_UNDERFILLED surfaces as the reference's assert
        check(lib.gcrl_agent_update_from_buffer(ag._h, ag.buffer.handle, 64, None, None, 1e-3, 1e-3, 3, None, None))
    assert steps() == before
    assert (ag.critic_scheduler.last_epoch, ag.actor_scheduler.last_epoch) == lr_before
    # ... and a valid update afterwards advances both by exactly one
    for e in her_episodes(load("her_reach_small")):
        ag.buffer.push_episode(e["s"], e["a"], e["ns"], e["r"], e["d"], e["ag"], e["fut"])
    ag.update(1)
    assert steps() == [before[0] + 1, before[1] + 1]


def test_public_soft_update_matches_the_reference_rule():
    """DDPG.update_target_network(hard_update=False, tau) (src/agent.py:1259-1271) and TD3Agent.update_actor /
    update_critic (:117-132) outside update(): theta_t <- tau theta + (1 - tau) theta_t in fp32, bit for bit."""
    from gcrl_b200 import DDPG, TD3Agent
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC
    rng = np.random.default_rng(5)
    D, A, H, L = 10, 3, 64, 2
    ag = DDPG(D, A, make_config(hidden_dim=H, layer_count=L), None, 1, 40)
    t_before = [[w.copy(), b.copy()] for w, b in ag.target_actor.layers() + ag.target_critic.layers()]
    ag._set_layers(NET_ACTOR, OD.init_mlp(rng, D, H, A, L))
    ag._set_layers(NET_CRITIC, OD.init_mlp(rng, D + A, H, 1, L))
    src = ag.actor.layers() + ag.critic.layers()
    tau = 0.05
    ag.update_target_network(hard_update=False, tau=tau)
    for (tw, tb), (w, b), (gw, gb) in zip(t_before, src, ag.target_actor.layers() + ag.target_critic.layers()):
        want_w = (np.float32(tau) * w + np.float32(1 - tau) * tw).astype(np.float32)
        want_b = (np.float32(tau) * b + np.float32(1 - tau) * tb).astype(np.float32)
        np.testing.assert_allclose(gw, want_w, rtol=2e-7, atol=1e-9)      # one fused multiply-add may replace mul + add
        np.testing.assert_allclose(gb, want_b, rtol=2e-7, atol=1e-9)
    td = TD3Agent(D, A, make_config(hidden_dim=H, layer_count=L), None, 1, 40)
    a0 = [w.copy() for w, _ in td.target_actor.layers()]
    c0 = [w.copy() for w, _ in td.target_critic_2.layers()]
    td._set_layers(NET_ACTOR, OD.init_mlp(rng, D, H, A, L))
    td.update_critic(0.3)                                  # actor target untouched; critic targets blend equal weights
    assert all(np.array_equal(x, y) for x, (y, _) in zip(a0, td.target_actor.layers()))
    assert all(np.allclose(x, y, rtol=2e-7, atol=0) for x, (y, _) in zip(c0, td.target_critic_2.layers()))
    td.update_actor(0.3)
    assert not np.array_equal(a0[0], td.target_actor.layers()[0][0])

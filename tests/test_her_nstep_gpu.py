"""GPU: n-step rows of the HER store (csrc/her.cu ``her_sample_kernel<..., NSTEP = true>``) against the restatement
of tests/her_nstep_reference.py, and every update engine trained from them.  "Bit-exact" is every field, the sign
of a -0.0 reward included.

  1. the sampler at every goal selection, eager and online, host and device positions, n in {1, 2, 3, 5, 60},
     gamma 0.98 and 0.6 (below the exactness bound of the done encoding), G = 3 and 6, episodes of 1, 2, 50 steps
     and early-terminated ones, a wrapped transition ring and a partly evicted oldest episode; both sampler tiles;
  2. update() from an n-step buffer == update(batch=...) on the restatement's rows (row-slab, fp32 tiles, tcgen05,
     SAC, TQC, quantile TQC), and one DDPG case against oracle/ddpg.py;
  3. update_many == the update() loop; 4. resume; 5. at B = 256 an n-step buffer takes the standalone sampler
     launch and n_step = 1 keeps the in-kernel sampler (counted launches).
"""
import random

import numpy as np
import pytest

from oracle.index_stream import feistel_positions
from tests import her_nstep_reference as NR
from tests.helpers import bits
from tests.test_her_nstep_cpu import make_episodes

pytestmark = pytest.mark.gpu

STRATEGIES = ["future", "final", "episode"]
TS = [1, 2, 50, 50, 3, 17, 50, 1, 50, 9, 2, 50, 50, 30]
K = 4
SEED = 1898


def assert_bits(got, ref, what):
    got = np.asarray(got, np.float32).reshape(np.shape(ref))
    assert np.array_equal(bits(got), bits(ref)), what


def ring_capacity(Ts, entries, max_len):
    """The least transition ring that holds every live window of the pushes (so that it wraps)."""
    total, need, ends = 0, 0, []
    for T, E in zip(Ts, entries):
        total += E
        ends.append((total, T))
        first_live = total - min(total, max_len)
        need = max(need, sum(T_ for end, T_ in ends if end > first_live))
    return need


def make_buffer(strategy, online, index_source, n, gamma, G, Ts, rng, max_len=None, **kw):
    from gcrl_b200 import HERBuffer
    eps = make_episodes(rng, Ts, 5, G, 2)
    entries = [T if online else (T - 1) * (K + 1) + 1 for T in Ts]
    max_len = max_len or int(0.8 * sum(entries)) + 1
    cap = ring_capacity(Ts, entries, max_len)
    random.seed(17)
    extra = {} if n is None else dict(n_step=n, gamma=gamma)
    buf = HERBuffer(max_len, 255, 1, k_future=K, index_source=index_source, seed=SEED, cap_transitions=cap,
                    goal_selection_strategy=strategy, online_sampling=online, **extra, **kw)
    for ep in eps:
        buf.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"])
    assert cap < sum(Ts)                                           # the ring wrapped
    return buf


def positions(buf, B, rng):
    epoch = buf.draw_epoch
    if buf.index_source == "host":
        return rng.integers(0, len(buf), B), epoch
    return feistel_positions(np.arange(B), len(buf), SEED, epoch), epoch


def restated(buf, pos, epoch, n, gamma):
    live = buf.state_dict()["episodes"]
    Ts = [ep["s"].shape[0] for ep in live]
    if buf.online_sampling:
        tags = NR.online_tags(Ts, len(buf), pos, SEED, epoch, buf.k_future, buf.goal_selection_strategy)
    else:
        deque = NR.eager_tags(Ts, [ep["fut"] for ep in live], buf.k_future, len(buf))
        tags = [deque[int(p)] for p in pos]
    return NR.nstep_rows(live, tags, n, gamma), tags


def sample(buf, B, pos):
    idx = pos if buf.index_source == "host" else None
    return [x.cpu().numpy() for x in buf.sample(B, indices=idx)]


# ---- 1. the sampler -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 2, 3, 5, 60])
@pytest.mark.parametrize("online", [False, True])
@pytest.mark.parametrize("strategy", STRATEGIES)
def test_sampler_equals_the_restatement(strategy, online, n):
    """Each case draws host positions at (gamma, G) = (0.98, 3) and device positions at (0.6, 6), and the reverse
    pairing at odd n, so every strategy, mode and n meets both discounts, both goal widths and both index streams."""
    rng = np.random.default_rng(n)
    pairs = [(0.98, 3), (0.6, 6)] if n % 2 == 0 else [(0.6, 6), (0.98, 3)]
    for index_source, (gamma, G) in zip(("host", "device"), pairs):
        buf = make_buffer(strategy, online, index_source, n, gamma, G, TS, rng)
        for B in (len(buf) // 2, len(buf)):
            pos, epoch = positions(buf, B, rng)
            got = sample(buf, B, pos)
            (ref, tags) = restated(buf, pos, epoch, n, gamma)
            assert any(j > 0 for _, _, j, _ in tags) and any(j == 0 for _, _, j, _ in tags)
            for x, y, key in zip(got, ref, "s a r ns d".split()):
                assert_bits(x, y, (index_source, B, key))


@pytest.mark.parametrize("online,index_source", [(False, "host"), (True, "device")])
def test_sampler_on_the_wide_tile(online, index_source):
    """B = 65 536: 128 samples per CTA."""
    rng = np.random.default_rng(3)
    B, n, gamma = 65536, 3, 0.98
    buf = make_buffer("future", online, index_source, n, gamma, 3, [50] * 1700 + [7, 1, 50], rng)
    pos, epoch = positions(buf, B, rng)
    got = sample(buf, B, pos)
    ref, _ = restated(buf, pos, epoch, n, gamma)
    for x, y, key in zip(got, ref, "s a r ns d".split()):
        assert_bits(x, y, key)


@pytest.mark.parametrize("online", [False, True])
def test_explicit_one_step_equals_the_default_buffer(online):
    b1 = make_buffer("future", online, "device", 1, 0.98, 3, TS, np.random.default_rng(5))
    b0 = make_buffer("future", online, "device", None, None, 3, TS, np.random.default_rng(5))
    for _ in range(2):
        for x, y in zip(b1.sample_host(len(b1)), b0.sample_host(len(b0))):
            assert_bits(x, y, "n_step=1")


def test_n_step_is_fixed_once_pushed():
    from gcrl_b200 import _lib
    buf = make_buffer("future", False, "device", 3, 0.98, 3, TS[:3], np.random.default_rng(1))
    assert _lib.lib.gcrl_her_set_n_step(buf.handle, 2, 0.98) != 0
    assert _lib.lib.gcrl_her_set_n_step(buf.handle, 3, 0.98) != 0


# ---- 2. updates ------------------------------------------------------------------------------------------------
D, A, G = 22, 3, 3


def nstep_agent(algo, B, n, index_source="device", online=False, hidden=64, max_len=None, cfg=None, **kw):
    import torch
    from gcrl_b200 import DDPG, SACAgent, TD3Agent, TQCAgent
    from tests.test_sac_gpu import sac_config
    max_len = max_len or 2 * B + 100
    cfg = cfg or sac_config(hidden_dim=hidden, batch_size=B, max_len=max_len, ac_update_freq=2, actor_lr=1e-3,
                     actor_lr_min=1e-4, ac_scheduler_steps=30, critic_lr=1e-3, critic_lr_min=1e-4,
                     cr_scheduler_steps=25, beta=0.4, beta_end=100, alpha_min_steps=50, alpha_lr=1e-2)
    torch.manual_seed(5)
    random.seed(6)
    cls = {"ddpg": DDPG, "td3": TD3Agent, "sac": SACAgent, "tqc": TQCAgent}[algo]
    ag = cls(D, A, cfg, None, 1, 40, index_source=index_source, online_sampling=online, n_step=n, **kw)
    per_ep = 50 if online else 49 * (K + 1) + 1
    Ts = [50] * (max_len // per_ep + 3)
    Ts[1] = 7
    for ep in make_episodes(np.random.default_rng(B), Ts, D - G, G, A):
        ag.buffer.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"])
    assert len(ag.buffer) == max_len
    return ag


def agent_state(ag):
    from tests.test_her_strategies_gpu import agent_state as state
    return state(ag)


def launches(fn):
    """Kernel launches of fn() (the library's own counter; the agent runs eager launches, GCRL_B200_NO_GRAPH=1)."""
    import torch
    from gcrl_b200._lib import lib
    torch.cuda.synchronize()
    before = int(lib.gcrl_kernel_launches())
    fn()
    torch.cuda.synchronize()
    return int(lib.gcrl_kernel_launches()) - before


@pytest.mark.parametrize("algo,B,kw", [("ddpg", 256, {}), ("td3", 256, {}), ("ddpg", 1500, {}), ("td3", 1500, {}),
                                       ("ddpg", 4096, {}), ("sac", 256, {}), ("tqc", 256, {}),
                                       ("tqc", 256, dict(n_quantiles=25, top_quantiles_to_drop_per_net=2))])
def test_update_from_the_buffer_equals_the_update_on_the_restated_rows(algo, B, kw):
    import torch
    from tests.test_update_many_gpu import same_results, seed_all
    n, gamma = 3, 0.98
    a1 = nstep_agent(algo, B, n, **kw)
    a2 = nstep_agent(algo, B, n, **kw)
    for step in (39, 40, 41):
        pos, epoch = positions(a1.buffer, B, None)
        rows, _ = restated(a1.buffer, pos, epoch, n, gamma)
        seed_all()
        r1 = [a1.update(step)]
        seed_all()
        batch = tuple(torch.from_numpy(x).cuda() for x in rows)
        r2 = a2.update(step, batch=batch)
        same_results(r1, [r2])
    for i, (x, y) in enumerate(zip(agent_state(a1), agent_state(a2))):
        assert np.array_equal(bits(x), bits(y)), i


def test_ddpg_n_step_update_matches_the_oracle():
    """One DDPG update from an n-step buffer against oracle/ddpg.py on the restated rows (odd shape tolerance)."""
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC
    from oracle import ddpg as OD
    from tests.test_ddpg_gpu import make_config
    B, n, gamma, H, L = 301, 5, 0.98, 64, 3
    ag = nstep_agent("ddpg", B, n, cfg=make_config(hidden_dim=H, layer_count=L, batch_size=B, max_len=2 * B + 100))
    rng = np.random.default_rng(0)
    actor0, critic0 = OD.init_mlp(rng, D, H, A, L), OD.init_mlp(rng, D + A, H, 1, L)
    ag._set_layers(NET_ACTOR, actor0)
    ag._set_layers(NET_CRITIC, critic0)
    ag.update_target_network()
    c = ag.config
    orc = OD.DDPGOracle(actor0, critic0, gamma=gamma, tau=c.tau, grad_clip=c.grad_clip, actor_lr=c.actor_lr,
                        critic_lr=c.critic_lr)
    pos, epoch = positions(ag.buffer, B, None)
    rows, _ = restated(ag.buffer, pos, epoch, n, gamma)
    assert (rows[4] > 0).any() and (rows[4] < 1).any()               # n-step done encodings in the batch
    info = ag.update(40)
    want = orc.update_on_batch(40, *rows)
    np.testing.assert_allclose(np.array([float(x) for x in info]), np.array(want), rtol=5e-5, atol=2e-6)
    for (w, _), (rw, _) in zip(ag.critic.layers() + ag.actor.layers(), orc.critic + orc.actor):
        assert np.max(np.abs(w - rw)) <= 1e-5 * np.max(np.abs(rw)) + 5e-6


# ---- 3. update_many --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo,index_source,online", [("ddpg", "host", False), ("ddpg", "device", False),
                                                      ("tqc", "host", False), ("tqc", "device", False),
                                                      ("ddpg", "device", True)])
def test_update_many_equals_the_loop(algo, index_source, online):
    from tests import test_sac_update_many_gpu as SM
    from tests import test_update_many_gpu as UM
    steps = list(range(1, 41))
    a_loop = nstep_agent(algo, 256, 3, index_source, online)
    a_many = nstep_agent(algo, 256, 3, index_source, online)
    mod = SM if algo == "tqc" else UM
    mod.loop_vs_many(a_loop, a_many, steps)
    mod.assert_same_state(a_loop, a_many)
    mod.one_more_update(a_loop, a_many)


# ---- 4. resume -------------------------------------------------------------------------------------------------
def test_resume_of_an_n_step_buffer_is_bit_identical():
    from gcrl_b200 import HERBuffer
    rng = np.random.default_rng(9)
    buf = make_buffer("episode", True, "device", 5, 0.98, 3, TS, rng)
    buf.sample_host(100)
    sd = buf.state_dict()
    assert sd["n_step"] == 5
    fresh = HERBuffer(buf.max_mem_len, 255, 1, k_future=K, index_source="device", seed=SEED,
                      cap_transitions=buf.cap_transitions, goal_selection_strategy="episode", online_sampling=True,
                      n_step=5, gamma=0.98)
    fresh.load_state_dict(sd)
    for x, y in zip(buf.sample_host(len(buf)), fresh.sample_host(len(fresh))):
        assert_bits(x, y, "resumed")
    for other in (dict(n_step=3, gamma=0.98), dict(n_step=5, gamma=0.9), {}):
        b = HERBuffer(buf.max_mem_len, 255, 1, k_future=K, index_source="device", seed=SEED,
                      goal_selection_strategy="episode", online_sampling=True, **other)
        with pytest.raises(ValueError):
            b.load_state_dict(sd)


# ---- 5. which sampler runs at B = 256 -------------------------------------------------------------------------
@pytest.mark.parametrize("algo", ["ddpg", "td3"])
def test_b256_sampler_path(algo, monkeypatch):
    """n_step = 1 keeps the row-slab critic kernel's in-kernel sampler; an n-step buffer launches the standalone
    sampler beside the same update kernels: exactly the launches of the one-step update with the in-kernel sampler
    switched off (GCRL_B200_NO_FUSED_SAMPLER=1), one more than with it on."""
    monkeypatch.setenv("GCRL_B200_NO_GRAPH", "1")
    one = nstep_agent(algo, 256, 1)
    nstep = nstep_agent(algo, 256, 3)
    monkeypatch.setenv("GCRL_B200_NO_FUSED_SAMPLER", "1")
    standalone = nstep_agent(algo, 256, 1)
    for step in (40, 41):                                          # with and without the actor phase
        n_one, n_nstep, n_standalone = (launches(lambda: ag.update(step)) for ag in (one, nstep, standalone))
        assert n_nstep == n_standalone == n_one + 1, (step, n_one, n_nstep, n_standalone)

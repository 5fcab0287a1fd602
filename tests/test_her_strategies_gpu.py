"""GPU: goal-selection strategies and online relabelling of the HER store (csrc/her.cu, csrc/her_device.cuh)
against the references of tests/her_strategy_reference.py (built on oracle/her.py).  "Bit-exact" is every field, the -0.0 sign of a relabelled reward included.

  1. eager "final" / "episode": push() under a seeded ``random`` -> the full dump equals the strategy-aware
     eager deque and the interpreter's stream ends where the oracle's does; device-drawn offsets lie in the
     strategy's range; offsets outside it are refused;
  2. online sampler == online_relabel_sample at host and Feistel positions, for sample() and sample_host();
  3. online draw statistics: relabel fraction, uniform goal step, no future / final relabel at t = T-1;
  4. every update engine (row-slab in-kernel sampler, fp32 tiles + sampler launch, tcgen05, TQC) samples the rows
     the standalone sampler returns at the same positions and epoch;
  5. update_many == the update() loop on an online buffer (DDPG, TD3, SAC, TQC);
  6. checkpoint resume of an online "episode" buffer, and refusal of a checkpoint with another goal selection.
"""
import random

import numpy as np
import pytest

from oracle import her as OH
from oracle.index_stream import feistel_positions
from tests import her_strategy_reference as HS
from tests.helpers import bits

pytestmark = pytest.mark.gpu

STRATEGIES = ["future", "final", "episode"]


def make_episodes(rng, Ts, O, G, A):
    """Seeded episodes: the last G state columns are the desired goal; achieved goals wander around it so that
    relabelled rewards take both values."""
    eps = []
    for T in Ts:
        dg = rng.normal(0, 0.05, G).astype(np.float32)
        obs = rng.standard_normal((T + 1, O)).astype(np.float32)
        s = np.concatenate([obs, np.tile(dg, (T + 1, 1))], 1).astype(np.float32)
        ag = (dg + np.cumsum(rng.normal(0, 0.02, (T + 1, G)), 0)).astype(np.float32)
        d = np.zeros(T, np.float32)
        d[-1] = 1.0
        eps.append({"s": s[:-1], "ns": s[1:], "a": rng.uniform(-1, 1, (T, A)).astype(np.float32),
                    "r": -(rng.random(T) > 0.2).astype(np.float32), "d": d, "dg": np.tile(dg, (T, 1)),
                    "ag": ag[1:]})
    return eps


def push_steps(buf, ep):
    for t in range(ep["s"].shape[0]):
        buf.push(0, ep["s"][t], ep["a"][t], ep["ns"][t], ep["r"][t], bool(ep["d"][t]), ep["dg"][t], ep["ag"][t])


def assert_bits(got, ref, what):
    got = np.asarray(got, np.float32).reshape(np.asarray(ref).shape)
    assert np.array_equal(bits(got), bits(ref)), what


def dump(buf):
    n = len(buf)
    return buf.sample_host(n, indices=np.arange(n))


# ---- 1. eager final / episode ---------------------------------------------------------------------------------
TS = [1, 2, 5, 50, 3, 17, 50, 1, 33, 49, 2, 50, 8]


@pytest.mark.parametrize("strategy", ["final", "episode"])
@pytest.mark.parametrize("k", [0, 1, 4, 8])
def test_eager_push_equals_the_strategy_aware_deque(strategy, k):
    from gcrl_b200 import HERBuffer
    eps = make_episodes(np.random.default_rng(k), TS, 7, 3, 3)
    total = sum((T - 1) * (k + 1) + 1 for T in TS)
    max_len = int(0.7 * total) + 3                                 # the oldest episodes are (partly) evicted
    random.seed(100 + k)
    buf = HERBuffer(max_len, 50, 1, k_future=k, goal_selection_strategy=strategy)
    for ep in eps:
        push_steps(buf, ep)
    st_product = random.getstate()
    random.seed(100 + k)
    orc = HS.eager_oracle(max_len, 50, 1, k, strategy)
    for ep in eps:
        push_steps(orc, ep)
    assert random.getstate() == st_product
    assert len(buf) == len(orc) == max_len
    for got, ref, key in zip(dump(buf), OH.collate(list(orc.buffer)), "s a r ns d".split()):
        assert_bits(got, ref, key)


@pytest.mark.parametrize("strategy", STRATEGIES)
def test_device_drawn_offsets_lie_in_the_strategy_range(strategy):
    from gcrl_b200 import HERBuffer
    k = 4
    eps = make_episodes(np.random.default_rng(3), TS, 7, 3, 3)
    buf = HERBuffer(10 ** 5, 50, 1, k_future=k, index_source="device", goal_selection_strategy=strategy)
    st = random.getstate()
    for ep in eps:
        buf.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"])
    assert random.getstate() == st
    parts = []
    for ep, stored in zip(eps, buf.state_dict()["episodes"]):
        T = ep["s"].shape[0]
        fut = stored["fut"][:T - 1].astype(np.int64)
        lo = {"future": np.arange(1, T)[:, None], "final": T - 1, "episode": 0}[strategy]
        assert (fut >= lo).all() and (fut <= T - 1).all()
        if strategy == "episode" and T > 2:
            assert len(np.unique(fut)) > 1
        parts.append(OH.materialise_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], stored["fut"], k))
    for got, i, key in zip(dump(buf), (0, 1, 2, 3, 4), "s a r ns d".split()):
        assert_bits(got, np.concatenate([p[i] for p in parts]), key)


@pytest.mark.parametrize("strategy", STRATEGIES)
def test_offsets_outside_the_strategy_range_are_refused(strategy):
    from gcrl_b200 import HERBuffer
    ep = make_episodes(np.random.default_rng(4), [6], 7, 3, 3)[0]
    T, k = 6, 2
    bad = {"future": 1, "final": T - 2, "episode": T}[strategy]     # offset of step 1
    fut = np.full((T, k), T - 1, np.uint8)
    fut[1, 0] = bad
    buf = HERBuffer(1000, 50, 1, k_future=k, goal_selection_strategy=strategy)
    with pytest.raises(ValueError):
        buf.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], fut)
    fut[1, 0] = T - 1                                               # inside every strategy's range
    buf.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], fut)
    assert len(buf) == (T - 1) * (k + 1) + 1
    online = HERBuffer(1000, 50, 1, k_future=k, goal_selection_strategy=strategy, online_sampling=True)
    with pytest.raises(ValueError):
        online.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], fut)


def test_bad_arguments_and_late_goal_selection_are_refused():
    import ctypes as C

    from gcrl_b200 import HERBuffer
    from gcrl_b200._lib import check, lib
    with pytest.raises(ValueError):
        HERBuffer(1000, 50, 1, goal_selection_strategy="random")
    with pytest.raises(ValueError):
        HERBuffer(1000, 50, 1, online_sampling="yes")
    ep = make_episodes(np.random.default_rng(5), [4], 7, 3, 3)[0]
    buf = HERBuffer(1000, 50, 1, k_future=4, index_source="device")
    with pytest.raises(ValueError):                                 # online needs a K = 0 store
        check(lib.gcrl_her_set_goal_selection(buf._h or _create(buf, ep), 0, 4))
    buf.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"])
    with pytest.raises(ValueError):                                 # after a commit
        check(lib.gcrl_her_set_goal_selection(buf._h, 1, 0))
    with pytest.raises(ValueError):
        check(lib.gcrl_her_set_goal_selection(buf._h, 3, 0))
    assert C.c_uint64(lib.gcrl_her_get_draw_epoch(buf._h)).value == 0


def _create(buf, ep):
    buf._ensure(ep["s"].shape[1], ep["a"].shape[1], ep["ag"].shape[1])
    return buf._h


# ---- 2. online sampler against the oracle ---------------------------------------------------------------------
@pytest.mark.parametrize("threshold", [0.05, 0.11])
@pytest.mark.parametrize("O,G", [(7, 3), (5, 6)])
@pytest.mark.parametrize("index_source", ["host", "device"])
@pytest.mark.parametrize("strategy", STRATEGIES)
def test_online_sampler_equals_the_oracle(strategy, index_source, O, G, threshold):
    from gcrl_b200 import HERBuffer
    rng = np.random.default_rng(10 * STRATEGIES.index(strategy) + G + (index_source == "host"))
    k, A, max_len, seed = 4, 3, 300, 1234
    Ts = [1, 2, 50] + [int(x) for x in rng.integers(1, 51, 30)] + [50, 1, 2]
    eps = make_episodes(rng, Ts, O, G, A)
    buf = HERBuffer(max_len, 50, 1, threshold=threshold, k_future=k, index_source=index_source, seed=seed,
                    cap_transitions=max_len + 60, goal_selection_strategy=strategy, online_sampling=True)
    assert buf.draw_epoch == 0
    committed = []
    for ci, ep in enumerate(eps):
        buf.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"])
        committed.append(ep)
        if len(buf) < 200 or ci % 6:
            continue
        assert len(buf) == min(sum(e["s"].shape[0] for e in committed), max_len)
        for call in range(2):
            B = 200 if call == 0 else len(buf)
            epoch = buf.draw_epoch
            pos = rng.integers(0, len(buf), B) if index_source == "host" else \
                feistel_positions(np.arange(B), len(buf), seed, epoch)
            idx = pos if index_source == "host" else None
            if call == 0:
                got = [x.cpu().numpy() for x in buf.sample(B, indices=idx)]
            else:
                *got, used = buf.sample_host(B, indices=idx, return_indices=True)
                assert np.array_equal(used, pos)
            assert buf.draw_epoch == epoch + 1
            ref, rel = HS.online_relabel_sample(committed, max_len, pos, seed, epoch, k, strategy, threshold)
            assert rel.any()
            for x, y, key in zip(got, ref, "s a r ns d".split()):
                assert_bits(x, y, (ci, call, key))


# ---- 3. online draw statistics ---------------------------------------------------------------------------------
@pytest.mark.parametrize("strategy", STRATEGIES)
def test_online_draw_statistics(strategy):
    from scipy import stats

    from gcrl_b200 import HERBuffer
    T, k, G, O, A, n_eps = 50, 4, 3, 4, 2, 1400
    buf = HERBuffer(T * n_eps, 50, 1, k_future=k, index_source="device", goal_selection_strategy=strategy,
                    online_sampling=True)
    t = np.arange(T, dtype=np.float32)
    s = np.zeros((T, O + G), np.float32)
    s[:, 0] = t
    s[:, O:] = -1.0                                                 # no step index is negative: -1 marks "not relabelled"
    ag = np.stack([t, t, t], 1).astype(np.float32)                  # the goal of step f is (f, f, f)
    zeros = np.zeros(T, np.float32)
    for _ in range(n_eps):
        buf.push_episode(s, np.zeros((T, A), np.float32), s, zeros, zeros, ag)
    B = 65536
    tt, ff = [], []
    for _ in range(16):                                             # 2^20 draws
        out = buf.sample_host(B)
        tt.append(out[0][:, 0].astype(np.int64))
        ff.append(out[0][:, O].astype(np.int64))
    tt, ff = np.concatenate(tt), np.concatenate(ff)
    rel = ff >= 0
    p = k / (k + 1)
    inner = tt < T - 1
    frac = rel[inner].mean()
    assert abs(frac - p) < 5 * np.sqrt(p * (1 - p) / inner.sum()), frac
    if strategy == "episode":
        last = rel[~inner].mean()
        assert abs(last - p) < 5 * np.sqrt(p * (1 - p) / (~inner).sum()), last
    else:
        assert not rel[~inner].any()
    lo = {"future": tt + 1, "final": np.full_like(tt, T - 1), "episode": np.zeros_like(tt)}[strategy]
    assert (ff[rel] >= lo[rel]).all() and (ff[rel] <= T - 1).all()
    if strategy == "final":
        assert (ff[rel] == T - 1).all()
        return
    t0 = 10
    sel = rel & (tt == t0)
    lo0 = t0 + 1 if strategy == "future" else 0
    counts = np.bincount(ff[sel] - lo0, minlength=T - lo0)
    assert counts.size == T - lo0
    assert stats.chisquare(counts).pvalue > 1e-5, counts


# ---- 4. every update engine samples the same rows ---------------------------------------------------------------
D, A, G = 22, 3, 3


def online_agent(algo, B, index_source="host", strategy="future", hidden=64, max_len=None):
    import torch
    from gcrl_b200 import DDPG, SACAgent, TD3Agent, TQCAgent
    from tests.test_sac_gpu import sac_config
    max_len = max_len or 2 * B + 100
    cfg = sac_config(hidden_dim=hidden, batch_size=B, max_len=max_len, ac_update_freq=2, actor_lr=1e-3,
                      actor_lr_min=1e-4, ac_scheduler_steps=30, critic_lr=1e-3, critic_lr_min=1e-4,
                      cr_scheduler_steps=25, beta=0.4, beta_end=100, alpha_min_steps=50, alpha_lr=1e-2)
    torch.manual_seed(5)
    cls = {"ddpg": DDPG, "td3": TD3Agent, "sac": SACAgent, "tqc": TQCAgent}[algo]
    ag = cls(D, A, cfg, None, 1, 40, index_source=index_source, goal_selection_strategy=strategy,
             online_sampling=True)
    for ep in make_episodes(np.random.default_rng(B), [50] * (max_len // 50 + 3), D - G, G, A):
        ag.buffer.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"])
    assert len(ag.buffer) == max_len
    return ag


def agent_state(ag):
    if hasattr(ag, "_critic_views"):
        from tests.test_sac_update_many_gpu import sac_state
        return sac_state(ag)
    from tests.test_fused_variants_gpu import all_weights
    w = all_weights(ag)
    return [w[key] for key in sorted(w)]


@pytest.mark.parametrize("index_source", ["host", "device"])
@pytest.mark.parametrize("algo,B", [("ddpg", 256), ("ddpg", 1536), ("ddpg", 4096), ("tqc", 256)])
def test_update_from_the_buffer_equals_the_update_on_the_sampled_rows(algo, B, index_source):
    from tests.test_update_many_gpu import same_results, seed_all
    a1 = online_agent(algo, B, index_source, strategy="episode")
    a2 = online_agent(algo, B, index_source, strategy="episode")
    for step in (39, 40, 41):
        seed_all()
        r1 = a1.update(step)
        seed_all()
        batch = a2.buffer.sample(B)
        r2 = a2.update(step, batch=batch)
        same_results([r1], [r2])
        assert a1.buffer.draw_epoch == a2.buffer.draw_epoch == step - 38
    for i, (x, y) in enumerate(zip(agent_state(a1), agent_state(a2))):
        assert np.array_equal(bits(x), bits(y)), i


# ---- 5. update_many == the update() loop ---------------------------------------------------------------------
@pytest.mark.parametrize("index_source", ["host", "device"])
@pytest.mark.parametrize("algo,B", [("ddpg", 256), ("ddpg", 1536), ("td3", 256), ("sac", 256), ("tqc", 256)])
def test_update_many_equals_the_loop_on_an_online_buffer(algo, B, index_source):
    from tests import test_sac_update_many_gpu as SM
    from tests import test_update_many_gpu as UM
    steps = list(range(1, 71))                                      # two graph chunks
    a_loop = online_agent(algo, B, index_source, strategy="future")
    a_many = online_agent(algo, B, index_source, strategy="future")
    mod = SM if algo in ("sac", "tqc") else UM
    mod.loop_vs_many(a_loop, a_many, steps)
    mod.assert_same_state(a_loop, a_many)
    assert a_loop.buffer.draw_epoch == a_many.buffer.draw_epoch == len(steps)
    mod.one_more_update(a_loop, a_many)


# ---- 6. resume ----------------------------------------------------------------------------------------------
def test_resume_of_an_online_episode_buffer_is_bit_identical(tmp_path):
    import torch
    from gcrl_b200 import DDPG
    from tests.test_ddpg_gpu import make_config
    eps = make_episodes(np.random.default_rng(21), [50, 13, 50, 50, 7, 50, 50, 50, 31, 50], D - G, G, A)
    cfg = make_config(hidden_dim=64, batch_size=64, max_len=250)   # the oldest episodes are evicted
    kw = dict(goal_selection_strategy="episode", online_sampling=True)

    def feed(ag, ep, lo=0, hi=None):
        for t in range(lo, ep["s"].shape[0] if hi is None else hi):
            ag.push_her(0, ep["s"][t], ep["a"][t], ep["ns"][t], ep["r"][t], bool(ep["d"][t]), ep["dg"][t], ep["ag"][t])
    torch.manual_seed(1)
    random.seed(77)
    a1 = DDPG(D, A, cfg, None, 1, 40, **kw)
    for ep in eps[:7]:
        feed(a1, ep)
    feed(a1, eps[7], hi=9)                                          # 9 transitions left in the staging deque
    for step in (1, 2, 3):
        a1.update(step)
    a1.save_checkpoint(str(tmp_path / "ck"))

    def rest(ag):
        feed(ag, eps[7], lo=9)
        feed(ag, eps[8])
        out = [[float(x) for x in ag.update(step)] for step in (4, 5, 6)]
        n = len(ag.buffer)
        return out, n, ag.buffer.draw_epoch, [x.copy() for x in ag.buffer.sample_host(n)]
    ref = rest(a1)
    torch.manual_seed(2)
    random.seed(5)
    a2 = DDPG(D, A, cfg, None, 1, 40, **kw)
    a2.load_checkpoint(str(tmp_path / "ck"))
    got = rest(a2)
    assert ref[:3] == got[:3]
    for x, y in zip(ref[3], got[3]):
        assert_bits(x, y, "resumed buffer dump")
    for other in (dict(goal_selection_strategy="future", online_sampling=True),
                  dict(goal_selection_strategy="episode", online_sampling=False), {}):
        a3 = DDPG(D, A, cfg, None, 1, 40, **other)
        with pytest.raises(ValueError):
            a3.load_checkpoint(str(tmp_path / "ck"))

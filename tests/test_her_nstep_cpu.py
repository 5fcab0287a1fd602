"""CPU: the n-step restatement (tests/her_nstep_reference.py) against the unmodified eager oracle and online
sampler at n = 1, against a float64 definition at every n, the exactness of the done encoding, and argument
validation of HERBuffer / the agents' ``n_step``."""
import random
import types

import numpy as np
import pytest

from oracle import her as OH
from tests import her_nstep_reference as NR
from tests import her_strategy_reference as HS
from tests.helpers import bits

STRATEGIES = ["future", "final", "episode"]
TS = [1, 2, 5, 50, 3, 17, 50, 1, 33, 49, 2, 50, 8]


def make_episodes(rng, Ts, O=5, G=3, A=2, terminate_every=3):
    """Seeded episodes, the last G state columns the desired goal; every `terminate_every`-th one ends in done = 1,
    the others are cut off (done = 0 throughout)."""
    eps = []
    for e, T in enumerate(Ts):
        dg = rng.normal(0, 0.05, G).astype(np.float32)
        obs = rng.standard_normal((T + 1, O)).astype(np.float32)
        s = np.concatenate([obs, np.tile(dg, (T + 1, 1))], 1).astype(np.float32)
        ag = (dg + np.cumsum(rng.normal(0, 0.02, (T + 1, G)), 0)).astype(np.float32)
        d = np.zeros(T, np.float32)
        if e % terminate_every == 0:
            d[-1] = 1.0
        eps.append({"s": s[:-1], "ns": s[1:], "a": rng.uniform(-1, 1, (T, A)).astype(np.float32),
                    "r": -(rng.random(T) > 0.2).astype(np.float32), "d": d, "dg": np.tile(dg, (T, 1)),
                    "ag": ag[1:]})
    return eps


def oracle_deque(eps, k, strategy, max_len, seed):
    """The eager oracle's deque after pushing `eps`, and the goal steps its randint returned, per episode."""
    random.seed(seed)
    orc = HS.eager_oracle(max_len, 255, 1, k, strategy)
    drawn = []
    inner = orc._randint
    orc._randint = lambda lo, hi: drawn.append(inner(lo, hi)) or drawn[-1]
    futs = []
    for ep in eps:
        T = ep["s"].shape[0]
        before = len(drawn)
        for t in range(T):
            orc.push(0, ep["s"][t], ep["a"][t], ep["ns"][t], ep["r"][t], t == T - 1, ep["dg"][t], ep["ag"][t])
        futs.append(np.array(drawn[before:], np.int64).reshape(max(T - 1, 0), k) if k else np.zeros((T, 0)))
    return orc, futs


def assert_bits(got, ref, what):
    assert np.array_equal(bits(np.asarray(got, np.float32).reshape(np.shape(ref))), bits(ref)), what


@pytest.mark.parametrize("strategy", STRATEGIES)
@pytest.mark.parametrize("k", [0, 1, 4])
def test_one_step_tags_are_the_eager_oracle_deque(strategy, k):
    eps = make_episodes(np.random.default_rng(k), TS, terminate_every=1)   # the oracle flushes on done
    total = sum((T - 1) * (k + 1) + 1 for T in TS)
    max_len = int(0.7 * total) + 3
    orc, futs = oracle_deque(eps, k, strategy, max_len, 10 + k)
    tags = NR.eager_tags([e["s"].shape[0] for e in eps], futs, k, max_len)
    assert len(tags) == len(orc) == max_len
    for got, ref, key in zip(NR.nstep_rows(eps, tags, 1, 0.98), OH.collate(list(orc.buffer)), "s a r ns d".split()):
        assert_bits(got, ref, key)


@pytest.mark.parametrize("strategy", STRATEGIES)
def test_one_step_online_tags_are_the_online_sampler(strategy):
    eps = make_episodes(np.random.default_rng(7), TS)
    total = sum(TS)
    max_len, seed, k = total - 20, 1234, 4
    pos = np.random.default_rng(1).integers(0, max_len, 300)
    for epoch in (0, 5):
        tags = NR.online_tags(TS, max_len, pos, seed, epoch, k, strategy)
        ref, rel = HS.online_relabel_sample(eps, max_len, pos, seed, epoch, k, strategy)
        assert np.array_equal(rel, np.array([j > 0 for _, _, j, _ in tags]))
        for got, want, key in zip(NR.nstep_rows(eps, tags, 1, 0.98), ref, "s a r ns d".split()):
            assert_bits(got, want, (epoch, key))


def all_tags(Ts, k, rng):
    futs = [np.stack([rng.integers(min(t + 1, T - 1), T, max(k, 1)) for t in range(T)]) for T in Ts]
    return NR.eager_tags(Ts, futs, k, 10 ** 9)


@pytest.mark.parametrize("n", [1, 2, 3, 5, 35, 60, 255])
@pytest.mark.parametrize("gamma", [0.98, 0.6, 1.0])
def test_restatement_against_the_float64_definition(n, gamma):
    """|R - sum gamma^i r_i| <= 2 (k-1) 2^-24 sum gamma^i |r_i| (k rounded products and sums, each relative 2^-24);
    |gamma (1 - d) - gamma^k (1 - done)| <= (k + 2) 2^-24 gamma^k + 2^-25 gamma (p's k-1 roundings, the product with
    gamma, and the 2^-25 of 1 - p when p < 1/2)."""
    rng = np.random.default_rng(n)
    eps = make_episodes(rng, TS)
    for ep in eps:                                   # stored rewards beyond {0, -1}: arbitrary float32 values
        ep["r"] = (ep["r"] * rng.uniform(0.1, 3.0, ep["r"].shape)).astype(np.float32)
    tags = all_tags(TS, 4, rng)
    _, _, R, _, Dn = NR.nstep_rows(eps, tags, n, gamma)
    R64, W64 = NR.float64_definition(eps, tags, n, gamma)
    g = float(np.float32(gamma))
    k = np.array([min(n, eps[e]["s"].shape[0] - t) for e, t, _, _ in tags], np.float64)
    absum = np.array([sum(g ** i * abs(float(NR.sparse_reward(eps[e]["ag"][t + i], eps[e]["ag"][f], 0.05) if j else
                                             eps[e]["r"][t + i])) for i in range(int(kk)))
                      for (e, t, j, f), kk in zip(tags, k)])
    assert (np.abs(R[:, 0].astype(np.float64) - R64) <= 2 * (k - 1) * 2.0 ** -24 * absum).all()
    w = (np.float32(gamma) * (np.float32(1) - Dn[:, 0])).astype(np.float32).astype(np.float64)
    assert (np.abs(w - W64) <= (k + 2) * 2.0 ** -24 * g ** k + 2.0 ** -25 * g).all()


@pytest.mark.parametrize("gamma", [0.98, 0.6, 0.9, 0.5, 1.0])
def test_the_bootstrap_weight_is_exact_while_p_is_at_least_one_half(gamma):
    """gamma (1 - d') == fl(gamma p) bit for bit for p = gamma^(k-1) >= 1/2, and |(1 - d') - p| <= 2^-25 below."""
    g = np.float32(gamma)
    p = np.float32(1)
    for k in range(1, 256):
        d = np.float32(np.float32(1) - np.float32(p * np.float32(np.float32(1) - np.float32(0))))
        one_minus = np.float32(np.float32(1) - d)
        if p >= 0.5:
            assert np.float32(g * one_minus) == np.float32(g * p), k
            assert one_minus == p
        else:
            assert abs(float(one_minus) - float(p)) <= 2.0 ** -25, k
        d_done = np.float32(np.float32(1) - np.float32(p * np.float32(np.float32(1) - np.float32(1))))
        assert d_done == 1.0 and np.float32(g * np.float32(1 - d_done)) == 0.0
        p = np.float32(p * g)
    if gamma == 0.98:      # the documented range of exactness: n <= 35
        p35 = np.float32(1)
        for _ in range(34):
            p35 = np.float32(p35 * g)
        assert p35 >= 0.5 and np.float32(p35 * g) < 0.5


# ---- argument validation ----------------------------------------------------------------------------------------
def test_n_step_arguments_are_checked():
    from gcrl_b200.buffer import _check_n_step
    assert _check_n_step(1, None) == (1, None)
    assert _check_n_step(1, 0.98) == (1, None)
    assert _check_n_step(3, 0.98) == (3, float(np.float32(0.98)))
    assert _check_n_step(np.int64(255), 1.0) == (255, 1.0)
    for n, g in [(0, 0.98), (256, 0.98), (2.0, 0.98), (True, 0.98), ("3", 0.98), (3, None), (3, 0.0), (3, 1.5),
                 (3, -0.5), (3, float("nan"))]:
        with pytest.raises(ValueError):
            _check_n_step(n, g)


def test_replay_buffers_refuse_n_step(monkeypatch):
    from gcrl_b200 import _lib
    from gcrl_b200.agent import _AgentBase
    monkeypatch.setattr(_lib, "require_cuda", lambda: None)
    for bt in ("REPLAY", "PER"):
        cfg = types.SimpleNamespace(buffer_type=bt, max_len=100, alpha=0.6, gamma=0.98)
        with pytest.raises(ValueError, match="n_step"):
            _AgentBase._init_common(object.__new__(_AgentBase), 5, 2, cfg, 1, 40, "host", 0, 1, "future", False, 3)

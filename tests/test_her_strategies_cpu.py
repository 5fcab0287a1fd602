"""CPU: the goal-selection references of tests/her_strategy_reference.py (the eager oracle of oracle/her.py with a
strategy, and the online relabelling restatement) -- what tests/test_her_strategies_gpu.py holds the CUDA store to.

  * with "future" the strategy-aware oracle still reproduces the reference's deque dumps (her_*.npz);
  * "final" consumes nothing from the interpreter's stream and relabels to the last step; "episode" calls
    randint(0, T-1) once per relabelled copy, in apply_her's order (t ascending, then j);
  * the online sampler's coin and goal step follow the stated rule on a hand-built store.
"""
import random

import numpy as np
import pytest

from oracle import her as OH
from oracle.index_stream import splitmix64
from tests import her_strategy_reference as HS
from tests.her_strategy_reference import relabel_hash
from tests.helpers import HER_CASES, bits, her_episodes, load


def push_all(buf, eps):
    for ep in eps:
        T = ep["s"].shape[0]
        for t in range(T):
            buf.push(0, ep["s"][t], ep["a"][t], ep["ns"][t], ep["r"][t], bool(ep["d"][t]), ep["dg"][t], ep["ag"][t])


@pytest.mark.parametrize("case", HER_CASES)
def test_future_strategy_reproduces_the_reference_dump(case):
    g = load("her_" + case)
    O, G, A, k, max_len, nenvs = (int(x) for x in g["meta"])
    eps = her_episodes(g)
    it = iter([int(v) for ep in eps for v in ep["fut"][:ep["s"].shape[0] - 1].reshape(-1)])
    buf = HS.eager_oracle(max_len, 50, 1, k, "future", randint=lambda a, b: next(it))
    push_all(buf, eps)
    assert next(it, None) is None
    s, a, r, ns, d = OH.collate(list(buf.buffer))
    for got, key in ((s, "dump_s"), (a, "dump_a"), (ns, "dump_ns"), (r[:, 0], "dump_r"), (d[:, 0], "dump_d")):
        assert np.array_equal(bits(got), bits(g[key])), key


@pytest.mark.parametrize("strategy", ["final", "episode"])
@pytest.mark.parametrize("k", [0, 1, 4])
def test_final_and_episode_consume_the_stream_as_stated(strategy, k):
    g = load("her_push_evict")
    eps = her_episodes(g)
    calls = []

    def randint(lo, hi):
        calls.append((lo, hi))
        return random.randint(lo, hi)

    random.seed(7)
    buf = HS.eager_oracle(10 ** 6, 50, 1, k, strategy, randint=randint)
    push_all(buf, eps)
    want = [] if strategy == "final" else [(0, ep["s"].shape[0] - 1) for ep in eps
                                           for _ in range((ep["s"].shape[0] - 1) * k)]
    assert calls == want
    # the relabelled copies carry the goal of step T-1 (final) or of the drawn step (episode)
    random.seed(7)
    pos = 0
    entries = list(buf.buffer)
    for ep in eps:
        T = ep["s"].shape[0]
        G = ep["ag"].shape[1]
        for t in range(T):
            pos += 1                                   # the original
            for _ in range(k if t < T - 1 else 0):
                f = T - 1 if strategy == "final" else random.randint(0, T - 1)
                s2, _, _, r2, d2, goal, ag = entries[pos]
                assert np.array_equal(goal, ep["ag"][f]) and np.array_equal(s2[-G:], ep["ag"][f])
                assert bits(r2) == bits(OH.compute_reward(ep["ag"][t], ep["ag"][f])) and d2 is False
                pos += 1
    assert pos == len(entries)


def test_oracle_refuses_an_unknown_strategy():
    with pytest.raises(AssertionError):
        HS.eager_oracle(100, 50, 1, 4, "random")


def test_relabel_hash_is_splitmix_of_key_plus_row():
    key = splitmix64(1898 ^ 0x6A09E667F3BCC909 ^ ((5 * 0xD1B54A32D192ED03) & ((1 << 64) - 1)))
    h = relabel_hash(1898, 5, np.arange(4, dtype=np.uint64))
    assert [int(x) for x in h] == [splitmix64((key + i) & ((1 << 64) - 1)) for i in range(4)]
    assert not np.array_equal(h, relabel_hash(1898, 6, np.arange(4, dtype=np.uint64)))


@pytest.mark.parametrize("strategy", ["future", "final", "episode"])
def test_online_restatement_follows_the_rule(strategy):
    rng = np.random.default_rng(0)
    T, D, A, G, k = 5, 6, 2, 3, 3
    ep = {"s": rng.standard_normal((T, D)).astype(np.float32), "a": rng.standard_normal((T, A)).astype(np.float32),
          "ns": rng.standard_normal((T, D)).astype(np.float32), "r": np.full(T, -1.0, np.float32),
          "d": np.ones(T, np.float32), "ag": np.arange(T * G, dtype=np.float32).reshape(T, G)}
    pos = np.tile(np.arange(T), 40)
    (s, a, r, ns, d), rel = HS.online_relabel_sample([ep], 100, pos, 1898, 3, k, strategy)
    h = relabel_hash(1898, 3, np.arange(len(pos), dtype=np.uint64))
    for i, t in enumerate(pos):
        lo = 0 if strategy == "episode" else t + 1
        want_rel = lo < T and int(h[i]) % (k + 1) != 0
        assert rel[i] == want_rel
        if want_rel:
            f = T - 1 if strategy == "final" else lo + (int(h[i]) >> 32) % (T - lo)
            assert np.array_equal(s[i, -G:], ep["ag"][f]) and np.array_equal(ns[i, -G:], ep["ag"][f])
            assert np.array_equal(s[i, :-G], ep["s"][t, :-G]) and d[i, 0] == 0.0
        else:
            assert np.array_equal(s[i], ep["s"][t]) and r[i, 0] == -1.0 and d[i, 0] == 1.0
    eligible = (pos < T - 1) | (strategy == "episode")
    assert 0.6 < rel[eligible].mean() < 0.9 and not rel[~eligible].any()

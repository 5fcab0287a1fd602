"""NumPy references for the HER store's goal-selection strategies and online relabelling (csrc/her.cu,
csrc/her_device.cuh), built on the unmodified eager oracle (oracle/her.py) and index stream (oracle/index_stream.py).

  * ``eager_oracle``: the reference's eager deque (``HERBufferOracle``) with the relabel goal of each copy chosen by
    a strategy -- "future" ``randint(t+1, T-1)`` (the reference), "final" ``T-1`` (no draw), "episode"
    ``randint(0, T-1)``, one goal per relabelled copy in apply_her's order.  apply_her asks its ``randint`` for
    ``(t+1, T-1)``; the strategy is a wrapper around that call.
  * ``relabel_hash`` / ``online_relabel_sample``: the online sampler, restated.
"""
import random

import numpy as np

from oracle.her import HERBufferOracle
from oracle.index_stream import M64, splitmix64

STRATEGIES = ("future", "final", "episode")


def strategy_randint(strategy, randint=None):
    """apply_her's ``randint(t+1, T-1)`` call -> the strategy's goal index for that copy."""
    assert strategy in STRATEGIES, strategy
    base = randint or random.randint
    if strategy == "final":
        return lambda lo, hi: hi                 # T-1, nothing drawn
    if strategy == "episode":
        return lambda lo, hi: base(0, hi)
    return base


def eager_oracle(max_mem_len, max_eps_len, nenvs, k_future, goal_selection_strategy="future", randint=None):
    return HERBufferOracle(max_mem_len, max_eps_len, nenvs, k_future=k_future,
                           randint=strategy_randint(goal_selection_strategy, randint))


def relabel_hash(seed, epoch, i):
    """Online relabelling's hash of (buffer seed, draw epoch, batch row i) (csrc/her_device.cuh
    ``her_relabel_hash``): splitmix64(splitmix64(seed ^ C ^ epoch * 0xD1B54A32D192ED03) + i), vectorised over i."""
    key = splitmix64(seed ^ 0x6A09E667F3BCC909 ^ ((epoch * 0xD1B54A32D192ED03) & M64))
    with np.errstate(over="ignore"):
        x = (np.asarray(i, np.uint64) + np.uint64(key)).astype(np.uint64)   # wraps mod 2^64
        x = x + np.uint64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def sparse_reward(achieved_goal, desired_goal, threshold):
    """oracle.her.compute_reward's arithmetic rule at any float32 threshold."""
    a = np.asarray(achieved_goal, dtype=np.float32)
    d = np.asarray(desired_goal, dtype=np.float32)
    diff = a - d
    sq = diff * diff
    acc = sq[..., 0]
    for i in range(1, sq.shape[-1]):
        acc = (acc + sq[..., i]).astype(np.float32)
    dist = np.sqrt(acc, dtype=np.float32)
    return -np.array(dist > np.float32(threshold), dtype=np.float32)


def online_relabel_sample(episodes, max_len, positions, seed, epoch, k, strategy, threshold=0.05):
    """Online relabelling sampler (csrc/her_device.cuh ``her_resolve``, online branch), restated.

    ``episodes``: every committed episode in commit order, dicts of s, a, ns, r, d, ag ([T, ...] arrays).  The
    store holds each transition once, so the live window is the last min(total, max_len) transitions and
    position p is transition total - len + p.  Row i of the call with draw epoch ``epoch`` hashes
    h = relabel_hash(seed, epoch, i); it is relabelled iff h % (k + 1) != 0 and the strategy's range
    [lo, T-1] is not empty (lo = t + 1 for future / final, 0 for episode), to the achieved goal of step
    f = T-1 (final) or lo + (h >> 32) % (T - lo): goal columns of s and s' <- ag[f], reward <- the sparse rule on
    (ag[t], ag[f]), done <- 0.  -> (states, actions, rewards, next_states, dones) and the relabel mask.
    """
    Ts = np.array([ep["s"].shape[0] for ep in episodes], np.int64)
    starts = np.cumsum(Ts) - Ts
    total = int(Ts.sum())
    n = min(total, int(max_len))
    ge = total - n + np.asarray(positions, np.int64)
    e = np.searchsorted(starts, ge, side="right") - 1
    S, A, R, NS, Dn, rel = [], [], [], [], [], []
    h = relabel_hash(seed, epoch, np.arange(len(ge), dtype=np.uint64))
    for i, (g, ei) in enumerate(zip(ge, e)):
        ep = episodes[int(ei)]
        t, T = int(g - starts[ei]), int(Ts[ei])
        s, ns = ep["s"][t].astype(np.float32).copy(), ep["ns"][t].astype(np.float32).copy()
        r, d = np.float32(ep["r"][t]), np.float32(ep["d"][t])
        lo = 0 if strategy == "episode" else t + 1
        hi = int(h[i])
        relabel = lo < T and hi % (k + 1) != 0
        if relabel:
            f = T - 1 if strategy == "final" else lo + ((hi >> 32) % (T - lo))
            goal = ep["ag"][f].astype(np.float32)
            G = goal.shape[0]
            s[-G:] = goal
            ns[-G:] = goal
            r = sparse_reward(ep["ag"][t], goal, threshold)
            d = np.float32(0.0)
        S.append(s); NS.append(ns); A.append(ep["a"][t].astype(np.float32))
        R.append(r); Dn.append(d); rel.append(relabel)
    return (np.stack(S), np.stack(A), np.array(R, np.float32)[:, None], np.stack(NS),
            np.array(Dn, np.float32)[:, None]), np.array(rel)

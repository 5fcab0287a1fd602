"""NumPy restatement of the HER store's n-step rows (csrc/her.cu ``her_sample_kernel<..., NSTEP>``).

Every deque entry is tagged (episode, t, j, f) straight from the pushed episodes, in apply_her's order: per step t
the original (j = 0, f = -1), then for t < T-1 the k_future relabelled copies (j = 1..k, goal step f = the copy's
drawn index).  The deque is the last min(total, max_len) tags.  An online store tags row i of a call with its own
relabel draw (her_strategy_reference.online_relabel_sample's rule).  At n = 1 the rows of these tags are the
eager oracle's deque and the online sampler's rows, bit for bit (tests/test_her_nstep_cpu.py); ``nstep_rows`` then
builds the n-step row of each tag in the kernel's float32 order:

  k  = min(n, T - t)
  r  = r_t + gamma*(r_{t+1} + gamma*(... + gamma*r_{t+k-1}))      (each product and sum rounded, from the back)
  s' = ns_{t+k-1}, goal columns <- g for a relabelled row
  d  = 1 - p*(1 - done_{t+k-1}),  p = gamma^(k-1) as k-1 rounded products; done = 0 for a relabelled row
  (k = 1: the one-step row, d = the stored done)

Stored rewards r_{t+i} are used for j = 0; a relabelled row recomputes each for its goal with the sparse rule.
"""
import numpy as np

from tests.her_strategy_reference import relabel_hash, sparse_reward

f32 = np.float32


def eager_tags(Ts, futs, k, max_len):
    """Ts: episode lengths in commit order; futs[e]: [T, >= k] goal steps of episode e's relabelled copies."""
    tags = []
    for e, T in enumerate(Ts):
        for t in range(T):
            tags.append((e, t, 0, -1))
            if t < T - 1:
                tags.extend((e, t, j, int(futs[e][t][j - 1])) for j in range(1, k + 1))
    return tags[len(tags) - min(len(tags), int(max_len)):]


def online_tags(Ts, max_len, positions, seed, epoch, k, strategy):
    """The tags of one online sample call at deque positions ``positions`` with draw epoch ``epoch``."""
    Ts = [int(T) for T in Ts]
    flat = [(e, t) for e, T in enumerate(Ts) for t in range(T)]
    live = flat[len(flat) - min(len(flat), int(max_len)):]
    h = relabel_hash(seed, epoch, np.arange(len(positions), dtype=np.uint64))
    tags = []
    for i, p in enumerate(positions):
        e, t = live[int(p)]
        T = Ts[e]
        lo = 0 if strategy == "episode" else t + 1
        hi = int(h[i])
        if lo < T and hi % (k + 1) != 0:
            tags.append((e, t, 1, T - 1 if strategy == "final" else lo + (hi >> 32) % (T - lo)))
        else:
            tags.append((e, t, 0, -1))
    return tags


def nstep_rows(episodes, tags, n, gamma, threshold=0.05):
    """-> (states, actions, rewards [B, 1], next_states, dones [B, 1]) of the tagged entries at n-step n."""
    gamma = f32(gamma)
    S, A, R, NS, Dn = [], [], [], [], []
    for e, t, j, f in tags:
        ep = episodes[e]
        T = ep["s"].shape[0]
        k = min(int(n), T - t)
        s = ep["s"][t].astype(f32).copy()
        ns = ep["ns"][t + k - 1].astype(f32).copy()
        if j > 0:
            g = ep["ag"][f].astype(f32)
            s[-g.shape[0]:] = g
            ns[-g.shape[0]:] = g
            rs = [f32(sparse_reward(ep["ag"][t + i], g, threshold)) for i in range(k)]
            done = f32(0.0)
        else:
            rs = [f32(ep["r"][t + i]) for i in range(k)]
            done = f32(ep["d"][t + k - 1])
        acc = rs[k - 1]
        for i in range(k - 2, -1, -1):
            acc = f32(rs[i] + f32(gamma * acc))
        if k > 1:
            p = f32(1.0)
            for _ in range(k - 1):
                p = f32(p * gamma)
            done = f32(f32(1.0) - f32(p * f32(f32(1.0) - done)))
        S.append(s); A.append(ep["a"][t].astype(f32)); R.append(acc); NS.append(ns); Dn.append(done)
    return (np.stack(S), np.stack(A), np.array(R, f32)[:, None], np.stack(NS), np.array(Dn, f32)[:, None])


def float64_definition(episodes, tags, n, gamma, threshold=0.05):
    """-> (R, weight) per tag in float64: R = sum_i gamma^i r_{t+i}, weight = gamma^k (1 - done_{t+k-1})."""
    g64 = float(f32(gamma))
    R, W = [], []
    for e, t, j, f in tags:
        ep = episodes[e]
        T = ep["s"].shape[0]
        k = min(int(n), T - t)
        if j > 0:
            rs = [float(sparse_reward(ep["ag"][t + i], ep["ag"][f], threshold)) for i in range(k)]
            done = 0.0
        else:
            rs = [float(ep["r"][t + i]) for i in range(k)]
            done = float(ep["d"][t + k - 1])
        R.append(sum(g64 ** i * r for i, r in enumerate(rs)))
        W.append(g64 ** k * (1.0 - done))
    return np.array(R), np.array(W)

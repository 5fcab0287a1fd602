"""HERBuffer over the device-resident episode store (reference src/buffer.py:92-179)."""
from __future__ import annotations

import ctypes as C
import random
from collections import deque

import numpy as np

from . import _lib
from ._lib import check, lib, np_ptr, vp

_FLUSH_LEN = 50  # the reference flushes on `done or len >= 50` (literal, src/buffer.py:117)
_RANDINT_BOUNDS = {}  # (T, k, strategy) -> (lo, hi) arrays of apply_her's randint calls, in its draw order
_STRATEGIES = {"future": _lib.HER_FUTURE, "final": _lib.HER_FINAL, "episode": _lib.HER_EPISODE}


def _to_np(x, dtype=np.float32):
    if hasattr(x, "detach"):                 # torch tensor (env.py hands device rows)
        x = x.detach().cpu().numpy()
    return np.asarray(x, dtype=dtype)


def _check_n_step(n_step, gamma):
    """-> (n_step, gamma as a float32 value, None when n_step == 1); ValueError on anything else."""
    if isinstance(n_step, (bool, np.bool_)) or not isinstance(n_step, (int, np.integer)) or not 1 <= n_step <= 255:
        raise ValueError(f"n_step must be an integer in [1, 255], got {n_step!r}")
    if n_step == 1:
        return 1, None
    if gamma is None:
        raise ValueError("n_step > 1 needs the discount gamma")
    g = float(np.float32(gamma))
    if not 0.0 < g <= 1.0:
        raise ValueError(f"gamma must be in (0, 1], got {gamma!r}")
    return int(n_step), g


class HERBuffer:
    """Same constructor, ``push`` / ``sample`` / ``__len__`` and attributes as the
    reference class.  Transitions are staged per env on the host and committed to the GPU
    as whole episodes; relabelling, the sparse reward and the gather run in
    csrc/her.cu at sample time.

    index_source:
      "host"   -- future indices come from ``random.randint`` and sample positions from
                  ``random.sample(range(len), B)``: the reference's exact Mersenne-Twister
                  stream (src/buffer.py:124,153), bit-identical batches.
      "device" -- both are drawn on the GPU (no per-call host work).
    ``compute_reward`` (src/env.py:105 assigns the env's function): relabelled rewards are computed on the
    GPU with the sparse Panda rule -(||ag - g||_2 > threshold) as float32.  An assigned callable is therefore
    PROBED on known-answer points around the threshold (as soon as the goal width is known) and must agree
    with that rule exactly; any other reward function raises ``ValueError`` instead of silently training on
    different rewards.  ``threshold`` (default 0.05, src/buffer.py:93) is passed to the kernel.

    goal_selection_strategy (Andrychowicz et al. 2017): the step f whose achieved goal relabels a transition at
    step t of an episode of T steps --
      "future"  -- f in [t+1, T-1] (the reference's strategy, the default);
      "final"   -- f = T-1;
      "episode" -- f in [0, T-1].
    online_sampling:
      False -- each episode is expanded into the reference's deque entries (the original and, for t < T-1,
               ``k_future`` relabelled copies whose f are drawn at commit: ``random.randint`` in apply_her's order
               with the "host" index source, "final" draws nothing).
      True  -- each transition is stored once (``len()`` counts transitions, so ``max_mem_len`` holds
               ``k_future + 1`` times as many episodes) and every sampled row is relabelled with probability
               k_future / (k_future + 1) to a freshly drawn f (none at t = T-1 for "future" / "final"): coin and f
               come from a hash of (seed, draw epoch, batch row), drawn on the GPU whatever the index source.
    n_step (Stable-Baselines3's ``n_steps``; 1, the default, samples one-step rows): a sampled row at step t of an
    episode of T stored steps, with goal g (the original or its relabel), covers the window t .. t+k-1,
    k = min(n_step, T - t).  ``rewards`` is r_t + gamma*(r_{t+1} + gamma*(... + gamma*r_{t+k-1})) in unfused float32
    from the back (relabelled rows recompute every r_{t+i} for g with the sparse rule), ``next_states`` is the next
    state of step t+k-1 (goal columns <- g), and ``dones`` is d' = 1 - gamma**(k-1) * (1 - done_{t+k-1}) (0 for the
    done of relabelled rows; gamma**(k-1) as k-1 rounded float32 products).  Any learner's gamma*(1 - d') is then the
    n-step bootstrap weight gamma**k * (1 - done): bit for bit fl(gamma * gamma**(k-1)) while gamma**(k-1) >= 1/2
    (gamma = 0.98: n_step <= 35), and within 2**-25 of it below.  The window does not stop at the relabel step.
    ``gamma`` in (0, 1] is required when n_step > 1; n_step is in [1, 255].
    """
    goal_selection_strategy = "future"
    online_sampling = False

    def __init__(self, max_mem_len, max_eps_len, nenvs, threshold=0.05, k_future=4, *,
                 index_source="host", seed=1898, cap_transitions=0, device=0,
                 goal_selection_strategy="future", online_sampling=False, n_step=1, gamma=None):
        _lib.require_cuda()
        n_step, gamma = _check_n_step(n_step, gamma)
        if index_source not in ("host", "device"):
            raise ValueError(f"index_source must be 'host' or 'device', got {index_source!r}")
        if goal_selection_strategy not in _STRATEGIES:
            raise ValueError(f"goal_selection_strategy must be one of {sorted(_STRATEGIES)}, "
                             f"got {goal_selection_strategy!r}")
        if not isinstance(online_sampling, (bool, np.bool_)):
            raise ValueError(f"online_sampling must be True or False, got {online_sampling!r}")
        if not 1 <= int(max_eps_len) <= 255:
            raise ValueError(f"max_eps_len must be in [1, 255] (future offsets are stored as uint8), got {max_eps_len}")
        if float(threshold) < 0:
            raise ValueError(f"threshold must be >= 0, got {threshold}")
        self.max_mem_len = int(max_mem_len)
        self.episodes = [deque(maxlen=max_eps_len) for _ in range(nenvs)]
        self.device_index = int(device)
        self.device = f"cuda:{self.device_index}"
        self.threshold = threshold
        self.k_future = int(k_future)
        self._compute_reward = None
        self._reward_checked = True
        self.obs_normalizer = None
        self.dg_normalizer = None
        self.index_source = index_source
        self.goal_selection_strategy = goal_selection_strategy
        self.online_sampling = bool(online_sampling)
        self.seed = int(seed)
        self.cap_transitions = int(cap_transitions)
        self.n_step, self.gamma = n_step, gamma
        self._h = None
        self._dims = None

    def __del__(self):
        if getattr(self, "_h", None):
            lib.gcrl_her_destroy(self._h)
            self._h = None

    # -- the injected reward function (src/env.py:105, called at src/buffer.py:166) --------------
    @property
    def compute_reward(self):
        return self._compute_reward

    @compute_reward.setter
    def compute_reward(self, fn):
        self._compute_reward = fn
        self._reward_checked = fn is None
        if fn is not None and self._dims is not None:
            self._check_reward(self._dims[2])

    def _check_reward(self, G):
        """The kernel relabels with -(||a - b||_2 > threshold) as float32 (csrc/her.cu, phase 3).  Probe the
        assigned callable on points whose distance is 0, well inside, exactly at and one float32 step either side
        of the threshold, and well outside; it must return that rule's values (0 / -1)."""
        thr = np.float32(self.threshold)
        dists = np.array([0.0, 0.5 * thr, np.nextafter(thr, np.float32(0)), thr, np.nextafter(thr, np.float32(1)),
                          2.0 * thr + 0.1], np.float32)
        a = np.zeros((len(dists), G), np.float32)
        b = np.zeros((len(dists), G), np.float32)
        b[:, 0] = dists                      # ||a - b|| is exactly dists[i] (one non-zero coordinate)
        want = -(dists > thr).astype(np.float32)
        try:
            got = np.stack([np.asarray(self._compute_reward(a[i], b[i], {}), np.float32).reshape(()) for i in range(len(dists))])
        except Exception as e:   # noqa: BLE001
            raise ValueError(f"compute_reward could not be evaluated on [{G}]-vectors: {e!r}") from e
        if not np.array_equal(got, want):
            raise ValueError(
                "HERBuffer.compute_reward is not the sparse rule -(||achieved - goal||_2 > threshold) "
                f"(threshold {float(thr)}): on distances {dists.tolist()} it returned {got.tolist()}, the GPU "
                f"relabel computes {want.tolist()}.  Only that reward is relabelled on the device; pass the matching "
                "`threshold` to HERBuffer, or use a sparse-reward task.")
        self._reward_checked = True

    # -- handle ---------------------------------------------------------------------------
    def _ensure(self, D, A, G):
        if self._h is None:
            h = vp()
            # an online store holds each transition once: the K = 0 entry mapping, relabelled at sample time
            check(lib.gcrl_her_create(C.byref(h), self.device_index, self.max_mem_len, self.cap_transitions, D, G, A,
                                      self._stored_k(), self.seed))
            self._h, self._dims = h, (D, A, G)
            check(lib.gcrl_her_set_threshold(h, float(self.threshold)))
            check(lib.gcrl_her_set_goal_selection(h, _STRATEGIES[self.goal_selection_strategy],
                                                  self.k_future if self.online_sampling else 0))
            if self.n_step > 1:
                check(lib.gcrl_her_set_n_step(h, self.n_step, self.gamma))
        elif self._dims != (D, A, G):
            raise ValueError(f"transition shape changed: {self._dims} -> {(D, A, G)}")
        if not self._reward_checked:
            self._check_reward(G)

    def _stored_k(self):
        return 0 if self.online_sampling else self.k_future

    @property
    def handle(self):
        return self._h

    @property
    def draw_epoch(self):
        """Sample calls drawn so far on the device index stream (online sampling: every sample call)."""
        return int(lib.gcrl_her_get_draw_epoch(self._h)) if self._h else 0

    def _stream(self):
        return _lib.current_stream(self.device_index)

    # -- reference API --------------------------------------------------------------------
    def push(self, idx, state, action, next_state, reward, done, desired_goal, achieved_goal):
        ep = self.episodes[idx]
        ep.append((_to_np(state), _to_np(action), _to_np(next_state), np.float32(reward),
                   bool(done), _to_np(achieved_goal)))
        if done or len(ep) >= _FLUSH_LEN:
            self._commit(ep)
            ep.clear()

    def push_episode(self, s, a, ns, r, d, ag, fut=None):
        """Commit a whole episode at once (arrays [T,...]); fut [T,k] uint8 or None."""
        s = np.ascontiguousarray(s, np.float32)
        a = np.ascontiguousarray(a, np.float32)
        ns = np.ascontiguousarray(ns, np.float32)
        r = np.ascontiguousarray(r, np.float32).reshape(-1)
        d = np.ascontiguousarray(d, np.float32).reshape(-1)
        ag = np.ascontiguousarray(ag, np.float32)
        T = s.shape[0]
        if self.online_sampling and fut is not None:
            raise ValueError("an online-sampling HERBuffer draws relabel goals at sample time: fut must be None")
        self._ensure(s.shape[1], a.shape[1], ag.shape[1])
        k = self._stored_k()
        if fut is None and self.index_source == "host" and k > 0:
            fut = self._draw_future(T)
        fptr = None
        if fut is not None and k > 0:
            fut = np.ascontiguousarray(fut, np.uint8).reshape(T, -1)[:, :k]
            fut = np.ascontiguousarray(fut)
            fptr = np_ptr(fut)
        check(lib.gcrl_her_push_episode(self._h, T, np_ptr(s), np_ptr(a), np_ptr(ns), np_ptr(r),
                                        np_ptr(d), np_ptr(ag), fptr, self._stream()))

    def _draw_future(self, T):
        """random.randint(t+1, T-1) in apply_her's order (src/buffer.py:145-153); "episode" draws
        random.randint(0, T-1) in the same order, "final" takes T-1 and draws nothing."""
        k, strategy = self.k_future, self.goal_selection_strategy
        fut = np.zeros((T, max(k, 1)), np.uint8)
        if T > 1 and k > 0 and strategy == "final":
            fut[:T - 1, :k] = T - 1
        elif T > 1 and k > 0:   # the same (T - 1) * k draws, in the same order, through the C mirror of CPython's MT
            bounds = _RANDINT_BOUNDS.get((T, k, strategy))
            if bounds is None:
                lo = np.repeat(np.arange(1, T, dtype=np.int32), k) if strategy == "future" else \
                    np.zeros((T - 1) * k, np.int32)
                bounds = _RANDINT_BOUNDS[(T, k, strategy)] = (lo, np.full(lo.shape, T - 1, np.int32))
            fut[:T - 1, :k] = _lib.py_randint_seq(*bounds).reshape(T - 1, k)
        return fut

    def _commit(self, ep):
        s, a, ns, r, d, ag = zip(*ep)
        self.push_episode(np.stack(s), np.stack(a), np.stack(ns), np.array(r, np.float32),
                          np.array(d, np.float32), np.stack(ag))

    def sample(self, batch_size: int, indices=None):
        import torch
        assert len(self) >= batch_size, "[ERROR] Not enough in buffer to sample"
        B = int(batch_size)
        D, A, _ = self._dims
        dev = torch.device("cuda", self.device_index)
        out = [torch.empty((B, w), dtype=torch.float32, device=dev) for w in (D, A, 1, D, 1)]
        iptr = None
        if indices is None and self.index_source == "host":
            indices = _lib.py_sample_range(len(self), B)       # == random.sample(deque, B), same MT stream
        if indices is not None:
            indices = np.ascontiguousarray(indices, np.int64)
            iptr = np_ptr(indices)
        check(lib.gcrl_her_sample(self._h, B, iptr, vp(out[0].data_ptr()), vp(out[1].data_ptr()),
                                  vp(out[2].data_ptr()), vp(out[3].data_ptr()),
                                  vp(out[4].data_ptr()), None, self._stream()))
        return tuple(out)                    # states, actions, rewards, next_states, dones

    def sample_host(self, batch_size: int, indices=None, return_indices=False):
        """sample() with NumPy outputs on the host (device->host copies inside the call)."""
        assert len(self) >= batch_size, "[ERROR] Not enough in buffer to sample"
        B = int(batch_size)
        D, A, _ = self._dims
        out = [np.empty((B, w), np.float32) for w in (D, A, 1, D, 1)]
        iptr = None
        if indices is None and self.index_source == "host":
            indices = _lib.py_sample_range(len(self), B)
        if indices is not None:
            indices = np.ascontiguousarray(indices, np.int64)
            iptr = np_ptr(indices)
        used = np.empty(B, np.int64) if return_indices else None
        check(lib.gcrl_her_sample_host(self._h, B, iptr, np_ptr(out[0]), np_ptr(out[1]),
                                       np_ptr(out[2]), np_ptr(out[3]), np_ptr(out[4]),
                                       np_ptr(used) if used is not None else None, self._stream()))
        return (*out, used) if return_indices else tuple(out)

    def __len__(self):
        return int(lib.gcrl_her_len(self._h)) if self._h else 0

    # -- true resume (SURVEY 8f-3): the live window + the per-env staging deques ---------------------------
    def state_dict(self):
        """Every episode that still holds a live entry (oldest first, with the future indices that were
        drawn) and the transitions staged per env.  ``load_state_dict`` on a fresh buffer with the same
        ``max_mem_len`` / ``k_future`` / goal selection reproduces every deque position, so a resumed run samples
        the same batches from the same ``random`` stream.  An online-sampling buffer stores no future indices; it
        records its draw epoch instead, so the resumed run draws the same relabels."""
        eps = []
        if self._h:
            D, A, G = self._dims
            k = self._stored_k()
            for i in range(int(lib.gcrl_her_live_episodes(self._h))):
                T = C.c_int()
                check(lib.gcrl_her_get_episode(self._h, i, C.byref(T), *([None] * 7), self._stream()))
                n = T.value
                arrs = dict(s=np.empty((n, D), np.float32), a=np.empty((n, A), np.float32),
                            ns=np.empty((n, D), np.float32), r=np.empty(n, np.float32), d=np.empty(n, np.float32),
                            ag=np.empty((n, G), np.float32), fut=np.zeros((n, max(k, 1)), np.uint8))
                fut = np.empty((n, k), np.uint8) if k else None
                check(lib.gcrl_her_get_episode(self._h, i, C.byref(T), np_ptr(arrs["s"]), np_ptr(arrs["a"]),
                                               np_ptr(arrs["ns"]), np_ptr(arrs["r"]), np_ptr(arrs["d"]),
                                               np_ptr(arrs["ag"]), np_ptr(fut) if k else None, self._stream()))
                if k:
                    arrs["fut"] = fut
                elif self.online_sampling:
                    arrs["fut"] = None
                eps.append(arrs)
        sd = {"max_mem_len": self.max_mem_len, "k_future": self.k_future, "dims": self._dims, "episodes": eps,
              "staging": [list(ep) for ep in self.episodes]}
        if self.goal_selection_strategy != "future" or self.online_sampling:
            sd.update(goal_selection_strategy=self.goal_selection_strategy, online_sampling=self.online_sampling)
        if self.online_sampling:
            sd["draw_epoch"] = self.draw_epoch
        if self.n_step > 1:
            sd.update(n_step=self.n_step, gamma=self.gamma)
        return sd

    def load_state_dict(self, sd):
        if sd["max_mem_len"] != self.max_mem_len or sd["k_future"] != self.k_future:
            raise ValueError("buffer checkpoint was written with a different max_mem_len / k_future")
        if (sd.get("goal_selection_strategy", "future") != self.goal_selection_strategy
                or bool(sd.get("online_sampling", False)) != self.online_sampling):
            raise ValueError("buffer checkpoint was written with a different goal_selection_strategy / online_sampling")
        if (int(sd.get("n_step", 1)), sd.get("gamma")) != (self.n_step, self.gamma):
            raise ValueError(f"buffer checkpoint was written with n_step={sd.get('n_step', 1)} / gamma={sd.get('gamma')}, "
                             f"this buffer has n_step={self.n_step} / gamma={self.gamma}")
        if self._h:
            check(lib.gcrl_her_clear(self._h))
        for ep in sd["episodes"]:
            self.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], ep["fut"])
        if self.online_sampling and self._h:
            check(lib.gcrl_her_set_draw_epoch(self._h, int(sd["draw_epoch"])))
        for dq, items in zip(self.episodes, sd["staging"]):
            dq.clear()
            dq.extend(items)

    def compute_termination(self, dg, ag):                 # src/buffer.py:140-141
        return np.linalg.norm(np.asarray(dg) - np.asarray(ag), axis=-1) < self.threshold

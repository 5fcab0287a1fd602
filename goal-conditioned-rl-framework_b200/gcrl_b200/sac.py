"""SAC / TQC agents over the CUDA learner (reference src/agent.py:388-770, 773-1171).

Same constructor arguments, attributes and methods as the reference classes: ``update(step)``
returns the 9-tuple (actor step) or 6-tuple, ``select_action`` is the eval-mode policy sample,
``save_weights`` writes ``actor.pth`` (SACActorModel state_dict keys, BatchNorm buffers
included), ``critic_1/2.pth`` (SAC) or ``critic_{i}.pth`` (TQC) and ``log_alpha.pth``.
The arithmetic runs in ``libgcrl_b200.so`` (csrc/sac.cu); the standard-normal draws behind
``Normal.rsample`` come from torch's CUDA generator (or are passed in by the parity tests).
"""
from __future__ import annotations

import ctypes as C
import os
import random

import numpy as np

from . import _lib
from ._lib import SacConfig, check, lib, np_ptr, vp
from .agent import CosineAnnealingLR, _AgentBase
from .buffer import HERBuffer

ALGO_SAC, ALGO_TQC = 2, 3


def _np(x):
    return np.asarray(x.detach().cpu().numpy() if hasattr(x, "detach") else x, np.float32)


class _SacActorView:
    """``agent.actor``: SACActorModel's state_dict surface (src/model.py:100-116, 143-156)."""

    def __init__(self, agent):
        self._a = agent

    def eval(self):
        return self

    def train(self, mode=True):
        return self

    def linear(self, layer):
        a = self._a
        rows = a.config.hidden_dim if layer < a.config.layer_count else a.ac_dim
        cols = a.obs_dim if layer == 0 else a.config.hidden_dim
        w, b = np.empty((rows, cols), np.float32), np.empty((rows,), np.float32)
        check(lib.gcrl_sac_get_actor_linear(a._h, layer, np_ptr(w), np_ptr(b), a._stream()))
        return w, b

    def set_linear(self, layer, w, b):
        a = self._a
        w, b = np.ascontiguousarray(w, np.float32), np.ascontiguousarray(b, np.float32)
        ew, _ = self.linear(layer)
        if w.shape != ew.shape or b.shape != (ew.shape[0],):
            raise ValueError(f"actor layer {layer}: expected {ew.shape}, got {w.shape}")
        check(lib.gcrl_sac_set_actor_linear(a._h, layer, np_ptr(w), np_ptr(b), a._stream()))

    def bn(self, layer):
        a = self._a
        out = [np.empty((a.config.hidden_dim,), np.float32) for _ in range(4)]
        check(lib.gcrl_sac_get_actor_bn(a._h, layer, *(np_ptr(x) for x in out), a._stream()))
        return out       # weight, bias, running_mean, running_var

    def set_bn(self, layer, weight=None, bias=None, running_mean=None, running_var=None):
        a = self._a
        arrs = [None if x is None else np.ascontiguousarray(x, np.float32)
                for x in (weight, bias, running_mean, running_var)]
        check(lib.gcrl_sac_set_actor_bn(a._h, layer, *(None if x is None else np_ptr(x) for x in arrs),
                                        a._stream()))

    def state_dict(self):
        import torch
        a, sd = self._a, {}
        for l in range(a.config.layer_count):
            w, b = self.linear(l)
            sd[f"base_net.{3 * l}.weight"], sd[f"base_net.{3 * l}.bias"] = torch.from_numpy(w), torch.from_numpy(b)
            g, be, rm, rv = self.bn(l)
            sd[f"base_net.{3 * l + 1}.weight"], sd[f"base_net.{3 * l + 1}.bias"] = torch.from_numpy(g), torch.from_numpy(be)
            sd[f"base_net.{3 * l + 1}.running_mean"] = torch.from_numpy(rm)
            sd[f"base_net.{3 * l + 1}.running_var"] = torch.from_numpy(rv)
            sd[f"base_net.{3 * l + 1}.num_batches_tracked"] = torch.tensor(a._bn_batches)
        L = a.config.layer_count
        for name, layer in (("mean_head", L), ("log_std_head", L + 1)):
            w, b = self.linear(layer)
            sd[f"{name}.weight"], sd[f"{name}.bias"] = torch.from_numpy(w), torch.from_numpy(b)
        return sd

    def load_state_dict(self, sd):
        a = self._a
        for l in range(a.config.layer_count):
            self.set_linear(l, _np(sd[f"base_net.{3 * l}.weight"]), _np(sd[f"base_net.{3 * l}.bias"]))
            k = f"base_net.{3 * l + 1}."
            self.set_bn(l, _np(sd[k + "weight"]), _np(sd[k + "bias"]), _np(sd[k + "running_mean"]),
                        _np(sd[k + "running_var"]))
            if k + "num_batches_tracked" in sd:
                a._bn_batches = int(sd[k + "num_batches_tracked"])
        L = a.config.layer_count
        self.set_linear(L, _np(sd["mean_head.weight"]), _np(sd["mean_head.bias"]))
        self.set_linear(L + 1, _np(sd["log_std_head.weight"]), _np(sd["log_std_head.bias"]))

    def save(self, path):
        import torch
        os.makedirs(os.path.dirname(path), exist_ok=True)
        torch.save(self.state_dict(), path)

    def load(self, weights, device="cpu"):
        import torch
        self.load_state_dict(torch.load(weights, map_location="cpu"))


class _SacCriticView:
    """``agent.critic_1`` / ``agent.critics[i]`` / targets: Critic state_dict surface."""

    def __init__(self, agent, index, target):
        self._a, self._i, self._t = agent, index, int(target)

    def eval(self):
        return self

    def train(self, mode=True):
        return self

    def _shape(self, layer):
        a = self._a
        L, H = a.config.layer_count, a.config.hidden_dim
        return (a._head_width() if layer == L else H, a.obs_dim + a.ac_dim if layer == 0 else H)

    def layers(self):
        a, out = self._a, []
        for layer in range(a.config.layer_count + 1):
            o, i = self._shape(layer)
            w, b = np.empty((o, i), np.float32), np.empty((o,), np.float32)
            check(lib.gcrl_sac_get_critic_layer(a._h, self._i, self._t, layer, np_ptr(w), np_ptr(b), a._stream()))
            out.append((w, b))
        return out

    def set_layers(self, layers):
        a = self._a
        for layer, (w, b) in enumerate(layers):
            w, b = np.ascontiguousarray(w, np.float32), np.ascontiguousarray(b, np.float32)
            if w.shape != self._shape(layer):
                raise ValueError(f"critic layer {layer}: expected {self._shape(layer)}, got {w.shape}")
            check(lib.gcrl_sac_set_critic_layer(a._h, self._i, self._t, layer, np_ptr(w), np_ptr(b), a._stream()))

    def state_dict(self):
        import torch
        sd = {}
        for i, (w, b) in enumerate(self.layers()):
            sd[f"net.{2 * i}.weight"], sd[f"net.{2 * i}.bias"] = torch.from_numpy(w), torch.from_numpy(b)
        return sd

    def load_state_dict(self, sd):
        n = self._a.config.layer_count + 1
        self.set_layers([(_np(sd[f"net.{2 * i}.weight"]), _np(sd[f"net.{2 * i}.bias"])) for i in range(n)])

    def save(self, path):
        import torch
        os.makedirs(os.path.dirname(path), exist_ok=True)
        torch.save(self.state_dict(), path)

    def load(self, weights, device="cpu"):
        import torch
        self.load_state_dict(torch.load(weights, map_location="cpu"))


class _Alpha:
    """``agent.alpha.item()`` (src/env.py:574, 604)."""

    def __init__(self, agent):
        self._a = agent

    def item(self):
        import math
        return math.exp(self._a.get_log_alpha())

    def __float__(self):
        return self.item()


class _SacBase(_AgentBase):
    ALGO = ALGO_SAC
    N_CRITICS, DROP_TOP = 2, 1
    ENTROPY_COEF = 0.2
    _sync_bn = None          # set by enable_data_parallel(sync_bn=True): the BatchNorm statistics all-gather
    _nq, _nq_drop = None, 0  # quantile critics (TQCAgent(n_quantiles=...)): atoms per critic, dropped per critic

    def __init__(self, obs_dim, ac_dim, config, weights, nenvs, gradient_step, *,
                 index_source="host", device=0, max_batch=None, seed=1898, precision=0,
                 goal_selection_strategy="future", online_sampling=False, n_step=1):
        """precision: 0 (default) runs every GEMM on the fp32 FFMA tiles; 1 runs the hidden-layer GEMMs of the
        critics and the actor on the tcgen05 tensor cores (3xTF32 split, the critic ensemble batched into one launch
        per layer) once batch * hidden_dim**2 >= 2048 * 256**2 (2048 rows at hidden_dim 256, 512 at 512, 8192 at
        128); 2 does so for every batch >= 128 (tests).  select_action stays on fp32.
        goal_selection_strategy / online_sampling / n_step: passed to the HER buffer (HERBuffer), n_step with
        config.gamma.  n_step > 1 needs buffer_type "HER" (ValueError otherwise).  The buffer's rows carry the n-step
        reward and a done column whose gamma*(1 - done) is gamma**k*(1 - done), so every update computes the n-step
        target unchanged; SAC / TQC take the entropy term at the bootstrap state only, as Stable-Baselines3 does."""
        self._init_common(obs_dim, ac_dim, config, nenvs, gradient_step, index_source, device, seed,
                          goal_selection_strategy, online_sampling, n_step)
        self.alpha_min = getattr(config, "alpha_min", 0.05)
        self.alpha_min_steps = getattr(config, "alpha_min_steps", 10000)
        self.target_entropy = self._target_entropy(ac_dim)
        cfg = SacConfig(algo=self.ALGO, state_dim=self.obs_dim, act_dim=self.ac_dim,
                        hidden_dim=config.hidden_dim, layer_count=config.layer_count,
                        max_batch=int(max_batch or config.batch_size), n_critics=self.N_CRITICS,
                        drop_top=self.DROP_TOP, gamma=config.gamma, tau=config.tau,
                        grad_clip=config.grad_clip, weight_decay=0.01, entropy_coef=self.ENTROPY_COEF,
                        target_entropy=self.target_entropy, alpha_lr=getattr(config, "alpha_lr", 3e-4),
                        precision=int(precision))
        h = vp()
        if self._nq is None:
            check(lib.gcrl_sac_create(C.byref(h), self.device_index, C.byref(cfg)))
        else:
            check(lib.gcrl_sac_create_quantile(C.byref(h), self.device_index, C.byref(cfg), self._nq, self._nq_drop))
        self._h = h
        self._max_batch = int(max_batch or config.batch_size)
        self._metrics = (C.c_float * 12)()
        self._bn_batches = 0
        self.actor = _SacActorView(self)
        self.alpha = _Alpha(self)
        self._critic_views = [_SacCriticView(self, i, False) for i in range(self.N_CRITICS)]
        self._target_views = [_SacCriticView(self, i, True) for i in range(self.N_CRITICS)]
        self._init_parameters()

    def __del__(self):
        if getattr(self, "_h", None):
            lib.gcrl_sac_destroy(self._h)
            self._h = None

    def _init_parameters(self):
        """xavier_uniform_ weights / bias 0.01 for every Linear, BatchNorm defaults
        (src/model.py:143-146), in the reference's construction order."""
        import torch
        H, L, D, A = self.config.hidden_dim, self.config.layer_count, self.obs_dim, self.ac_dim

        def xavier(o, i):
            w = torch.empty(o, i)
            torch.nn.init.xavier_uniform_(w)
            return w.numpy(), np.full((o,), 0.01, np.float32)

        for l in range(L):
            self.actor.set_linear(l, *xavier(H, D if l == 0 else H))
            self.actor.set_bn(l, np.ones(H, np.float32), np.zeros(H, np.float32), np.zeros(H, np.float32),
                              np.ones(H, np.float32))
        self.actor.set_linear(L, *xavier(A, H))
        self.actor.set_linear(L + 1, *xavier(A, H))
        for view in self._critic_views:
            view.set_layers([xavier(self._head_width() if l == L else H, D + A if l == 0 else H) for l in range(L + 1)])
        self._bn_batches = 0

    def _target_entropy(self, ac_dim):
        raise NotImplementedError

    def _head_width(self):
        """Rows of every critic's last Linear: 1, or n_quantiles for quantile critics."""
        return 1 if self._nq is None else self._nq

    def update_target_network(self):
        check(lib.gcrl_sac_hard_update(self._h, self._stream()))

    def get_log_alpha(self):
        v = C.c_float()
        check(lib.gcrl_sac_get_log_alpha(self._h, C.byref(v), self._stream()))
        return float(v.value)

    def set_log_alpha(self, value):
        check(lib.gcrl_sac_set_log_alpha(self._h, float(value), self._stream()))

    @property
    def log_alpha(self):
        import torch
        return torch.tensor([self.get_log_alpha()], dtype=torch.float32)

    def select_action(self, obs_tensor, eval_action: bool = False):           # :641-647 / :1044-1050
        obs = np.ascontiguousarray(obs_tensor, np.float32).reshape(-1, self.obs_dim)
        out = np.empty((obs.shape[0], self.ac_dim), np.float32)
        # Normal.rsample draws from torch's generator in the reference (src/model.py:135-137), never from NumPy's
        # global stream (which PERBuffer.sample consumes): same generator here, on the agent's device
        eps = None
        if not eval_action:
            import torch
            eps = torch.randn((obs.shape[0], self.ac_dim), dtype=torch.float32, device=self.device).cpu().numpy()
        cap = int(self._max_batch)
        for lo in range(0, obs.shape[0], cap):       # any number of envs: the act scratch holds max_batch rows
            hi = min(obs.shape[0], lo + cap)
            o_, out_ = np.ascontiguousarray(obs[lo:hi]), np.empty((hi - lo, self.ac_dim), np.float32)
            e_ = None if eps is None else np.ascontiguousarray(eps[lo:hi])
            check(lib.gcrl_sac_act(self._h, hi - lo, np_ptr(o_), None if e_ is None else np_ptr(e_), np_ptr(out_),
                                   self._stream()))
            out[lo:hi] = out_
        return out

    def _polyak_now(self, step):
        raise NotImplementedError

    def _per_ptrs(self):
        if self._per is None:
            w, td = vp(), vp()
            check(lib.gcrl_sac_per_buffers(self._h, C.byref(w), C.byref(td)))
            self._per = (w, td)
        return self._per

    # -- data parallel: same GradAverager as DDPG / TD3 over the buffers of gcrl_sac_dp_buffer -------
    def enable_data_parallel(self, process_group=None, allreduce_mean=None, sync_bn=True, *, world=None, rank=None,
                             allgather=None):
        """Gradient averaging between the update phases as for DDPG / TD3, plus -- ``sync_bn=True``, the default --
        BatchNorm batch statistics over the GLOBAL batch, so that N ranks on B rows each equal one rank on the
        concatenated N * B rows (SURVEY 8(e): the reference is single-GPU, src/model.py:103-111 normalises over the
        whole batch).  Every rank must use the same local batch size.  ``sync_bn=False`` keeps local statistics
        (torch DDP's default without SyncBatchNorm: 4 phases, 3 collectives per update instead of 3 + 3 per
        BatchNorm layer) and averages the running statistics after every update.
        ``world`` / ``rank`` / ``allgather(slots_tensor)`` override torch.distributed (tests).  Not available for
        quantile critics (TQCAgent(n_quantiles=...)): ValueError."""
        if self._nq is not None:
            raise ValueError(f"{type(self).__name__}: data parallelism is not available for quantile critics "
                             "(n_quantiles); train on one GPU")
        dp = super().enable_data_parallel(process_group, allreduce_mean)
        self._sync_bn = None
        if not sync_bn:
            check(lib.gcrl_sac_set_sync_bn(self._h, 0, 0))
            return dp
        if world is None:
            import torch.distributed as dist
            world, rank = dist.get_world_size(process_group), dist.get_rank(process_group)
        check(lib.gcrl_sac_set_sync_bn(self._h, int(world), int(rank)))
        slots = self.grad_tensor(4)
        if allgather is None:
            import torch.distributed as dist
            mine = slots.view(int(world), -1)[int(rank)]

            def allgather(t, _mine=mine, _group=process_group):
                dist.all_gather_into_tensor(t, _mine, group=_group)      # in place: row `rank` is the input
        self._sync_bn = lambda: allgather(slots)
        return dp

    def grad_tensor(self, which):
        from .parallel import device_tensor
        ptr, n = vp(), C.c_int64()
        check(lib.gcrl_sac_dp_buffer(self._h, int(which), C.byref(ptr), C.byref(n)))
        return device_tensor(ptr.value, n.value, self.device_index)

    def metrics_tensor(self):
        return self.grad_tensor(3)

    def _flags(self, step):
        """bit0 actor step, bit1 Polyak step, bit2 alpha step (an actor step past alpha_min_steps)."""
        actor_step = step % self.ac_update_freq == 0
        return (1 if actor_step else 0) | (2 if self._polyak_now(step) else 0) \
            | (4 if (actor_step and step > self.alpha_min_steps) else 0)

    def _result(self, step, m):
        """The tuple update(step) returns, from the 12 metric floats of its update."""
        flags = self._flags(step)
        q1l, q2l, acl, td, qv, c1g, c2g, acg, all_ = m[:9]
        td = np.float32(td) if self._last_td is None else self._last_td
        if flags & 1:
            return q1l, q2l, acl, td, qv, c1g, c2g, acg, (all_ if flags & 4 else 0.0)
        return q1l, q2l, td, qv, c1g, c2g

    def update(self, step: int, batch=None, indices=None, eps_next=None, eps_cur=None):
        import torch
        B = self.batch_size if batch is None else batch[0].shape[0]
        actor_step = step % self.ac_update_freq == 0
        if eps_next is None:
            eps_next = torch.randn((B, self.ac_dim), dtype=torch.float32, device=self.device)
        if eps_cur is None and actor_step:
            eps_cur = torch.randn((B, self.ac_dim), dtype=torch.float32, device=self.device)
        flags = self._flags(step)
        lr_c, lr_a = self.critic_scheduler.lr, self.actor_scheduler.lr
        mptr = C.cast(self._metrics, vp)
        en = vp(eps_next.data_ptr())
        ec = vp(eps_cur.data_ptr()) if eps_cur is not None else None
        iptr, bufh, ptrs = None, None, (None,) * 5
        per = False
        if batch is None and not isinstance(self.buffer, HERBuffer):
            batch, per = self._replay_batch(B)           # src/agent.py:661-673 / :1064-1076
            if per:
                flags |= 8
        if batch is None:
            assert len(self.buffer) >= B, "[ERROR] Not enough in buffer to sample"
            if indices is None and self.index_source == "host":
                indices = _lib.py_sample_range(len(self.buffer), B)
            if indices is not None:
                indices = np.ascontiguousarray(indices, np.int64)
                iptr = np_ptr(indices)
            bufh = self.buffer.handle
        else:
            ptrs = tuple(vp(t.data_ptr()) for t in batch)
        if self._dp is not None and self._sync_bn is not None:
            # sync-BN: graph segments, each ending in the collective the C side names (include/gcrl_b200.h)
            st = self._stream()
            coll = C.c_int(0)
            for seg in range(1 << 16):
                check(lib.gcrl_sac_update_segment(self._h, seg, bufh, B, iptr, *ptrs, en, ec, lr_c, lr_a, flags,
                                                  C.byref(coll), st))
                if coll.value == 0:
                    break
                if coll.value == 1:
                    self._sync_bn()                        # all-gather of the BatchNorm partial statistics
                else:
                    self._dp.average((1,) if coll.value == 2 else (0,))
            self._dp.average_metrics()
            check(lib.gcrl_sac_read_metrics(self._h, flags, mptr, st))
        elif self._dp is not None:
            st = self._stream()
            for phase in range(4):
                check(lib.gcrl_sac_update_phase(self._h, phase, bufh, B, iptr, *ptrs, en, ec, lr_c, lr_a, flags, st))
                if phase == 0:
                    self._dp.average((1,))                 # the critic ensemble's gradients, one buffer
                elif phase == 2 and (flags & 1):
                    self._dp.average((0,))                 # actor gradient + alpha's batch mean
            self._dp.average((2,))                         # BatchNorm running statistics
            self._dp.average_metrics()
            check(lib.gcrl_sac_read_metrics(self._h, flags, mptr, st))
        elif batch is None:
            check(lib.gcrl_sac_update_from_buffer(self._h, bufh, B, iptr, en, ec, lr_c, lr_a, flags, mptr,
                                                  self._stream()))
        else:
            check(lib.gcrl_sac_update_batch(self._h, B, *ptrs, en, ec, lr_c, lr_a, flags, mptr, self._stream()))
        self._last_td = self._replay_finish(B) if per else None
        self.critic_scheduler.step()
        self._bn_batches += 1
        if actor_step:
            self.actor_scheduler.step()
            self._bn_batches += 1
        self.beta_scheduler(step)
        return self._result(step, [float(x) for x in self._metrics])

    # -- a training cycle's gradient steps in one call (_AgentBase.update_many) ------------------------------
    _MANY_FNS = ("gcrl_sac_update_many", "gcrl_sac_update_many_replay")
    _METRIC_WIDTH = 12
    _MIN_BATCH = 2              # BatchNorm needs more than one row
    _BN_BATCHES = (1, 2)        # num_batches_tracked grows as update() grows it: 1, or 2 with an actor step

    def _many_noise(self, B, flags):
        """update()'s torch.randn calls for n updates, in step order: (eps_next [n][B][A], eps_cur [n][B][A] or None
        when no update steps the actor)."""
        import torch
        shape = (B, self.ac_dim)
        eps_next, eps_cur = [], []
        for f in flags:
            eps_next.append(torch.randn(shape, dtype=torch.float32, device=self.device))
            eps_cur.append(torch.randn(shape, dtype=torch.float32, device=self.device) if f & 1 else None)
        eps_next = torch.stack(eps_next)
        if not any(f & 1 for f in flags):
            return eps_next, None
        unused = torch.zeros(shape, dtype=torch.float32, device=self.device)    # rows of critic-only steps: never read
        return eps_next, torch.stack([unused if e is None else e for e in eps_cur])

    def _save_log_alpha(self, path):
        import torch
        torch.save(self.log_alpha, os.path.join(path, "log_alpha.pth"))

    def reset(self):
        """SACAgent.reset / TQCAgent.reset (src/agent.py:755-769, :1161-1170): ``module.apply(_init_weights)`` on the
        actor, every critic and every TARGET critic re-draws xavier weights / bias 0.01 for the nn.Linear layers
        only -- BatchNorm affine parameters and running statistics survive, the targets get their OWN draws (they
        are not copies of the online critics afterwards) -- then log_alpha = 0 with a fresh AdamW.  Draw order as
        the reference: actor (hidden Linears, mean head, log-std head), critics, target critics."""
        import torch
        H, L, D, A = self.config.hidden_dim, self.config.layer_count, self.obs_dim, self.ac_dim

        def xavier(o, i):
            w = torch.empty(o, i)
            torch.nn.init.xavier_uniform_(w)
            return w.numpy(), np.full((o,), 0.01, np.float32)

        for l in range(L):
            self.actor.set_linear(l, *xavier(H, D if l == 0 else H))
        self.actor.set_linear(L, *xavier(A, H))
        self.actor.set_linear(L + 1, *xavier(A, H))
        for view in list(self._critic_views) + list(self._target_views):
            view.set_layers([xavier(self._head_width() if l == L else H, D + A if l == 0 else H) for l in range(L + 1)])
        self.set_log_alpha(0.0)          # also re-creates alpha's AdamW state (gcrl_sac_set_log_alpha)

    # -- what the DDPG / TD3 base offers through gcrl_agent_* does not exist for this handle type ---------------
    def _not_for_sac(self, what):
        raise NotImplementedError(
            f"{type(self).__name__}.{what} is not available: SAC / TQC agents checkpoint through save_weights() "
            "(the reference's own format: actor.pth, critic_*.pth, log_alpha.pth -- src/agent.py:701-705, :1102-1106) "
            "and the normalisers' YAML; optimiser moments are not exported for these agents")

    def state_dict(self):
        self._not_for_sac("state_dict")

    def load_state_dict(self, sd):
        self._not_for_sac("load_state_dict")

    def save_checkpoint(self, path):
        self._not_for_sac("save_checkpoint")

    def load_checkpoint(self, path):
        self._not_for_sac("load_checkpoint")

    def hard_update(self):
        self.update_target_network()

    def q_values(self, *a, **k):
        self._not_for_sac("q_values")

    def _actor_forward(self, *a, **k):
        self._not_for_sac("_actor_forward")

    def read_metrics(self):
        self._not_for_sac("read_metrics")

    def enable_peer_data_parallel(self, process_group=None):
        self._not_for_sac("enable_peer_data_parallel (use enable_data_parallel: NCCL between the update phases)")

    def peer_barrier(self):
        self._not_for_sac("peer_barrier")

    def _num_layers(self, net):
        self._not_for_sac("_num_layers")

    def _get_layers(self, net):
        self._not_for_sac("_get_layers")

    def _set_layers(self, net, layers):
        self._not_for_sac("_set_layers")


class SACAgent(_SacBase):
    """Reference src/agent.py:388-770."""
    ALGO = ALGO_SAC
    N_CRITICS, DROP_TOP = 2, 1          # torch.min(Q1, Q2)
    ENTROPY_COEF = 0.2                   # literal at :521, :569 (the learned alpha is never used in a loss)

    def __init__(self, obs_dim, ac_dim, config, weights, nenvs, gradient_step, **kw):
        super().__init__(obs_dim, ac_dim, config, weights, nenvs, gradient_step, **kw)
        self.critic_1, self.critic_2 = self._critic_views
        self.target_critic_1, self.target_critic_2 = self._target_views
        self.train_alpha = False
        if weights:
            self.actor.load(os.path.join(weights, "actor.pth"))
            self.critic_1.load(os.path.join(weights, "critic_1.pth"))
            self.critic_2.load(os.path.join(weights, "critic_2.pth"))
        self.update_target_network()

    def _target_entropy(self, ac_dim):
        return -ac_dim * 0.5             # :423

    def _polyak_now(self, step):
        return step % self.gradient_step == 0     # :681

    def save_weights(self, path: str):   # :701-705
        self.actor.save(os.path.join(path, "actor.pth"))
        self.critic_1.save(os.path.join(path, "critic_1.pth"))
        self.critic_2.save(os.path.join(path, "critic_2.pth"))
        self._save_log_alpha(path)


class TQCAgent(_SacBase):
    """Reference src/agent.py:773-1171 (5 scalar critics, drop the top 2; see SURVEY 0.4).

    ``n_quantiles=None`` (the default) is that agent.  An integer M gives Truncated Quantile Critics as
    sb3-contrib's ``TQC(n_quantiles=M, top_quantiles_to_drop_per_net=d)`` runs them (Kuznetsov et al., 2020):
    every critic ends in an H -> M Linear (M quantile atoms), the target pools the 5 M atoms of the target critics
    at (s', a'), keeps the 5 (M - d) smallest and each critic fits all its atoms to them with the quantile Huber
    loss (kappa 1); the actor maximises the mean of all atoms, without truncation.  Checkpoints hold an [M, H] head
    in ``net.{2L}.weight``; data parallelism is not available for quantile critics."""
    ALGO = ALGO_TQC
    N_CRITICS, DROP_TOP = 5, 2           # getattr defaults, :789-790 (the YAML keys never reach the config)
    ENTROPY_COEF = -1.0                  # use the learned alpha (:928, :978)

    def __init__(self, obs_dim, ac_dim, config, weights, nenvs, gradient_step, *, n_quantiles=None,
                 top_quantiles_to_drop_per_net=2, **kw):
        self._nq, self._nq_drop = self._check_quantiles(n_quantiles, top_quantiles_to_drop_per_net)
        super().__init__(obs_dim, ac_dim, config, weights, nenvs, gradient_step, **kw)
        self.num_critics, self.top_quantiles_to_drop = self.N_CRITICS, self.DROP_TOP
        self.n_quantiles, self.top_quantiles_to_drop_per_net = self._nq, self._nq_drop
        self.critics, self.target_critics = list(self._critic_views), list(self._target_views)
        if weights:
            import torch
            self.actor.load(os.path.join(weights, "actor.pth"))
            for i, critic in enumerate(self.critics):
                p = os.path.join(weights, f"critic_{i}.pth")
                if os.path.exists(p):
                    critic.load(p)
            p = os.path.join(weights, "log_alpha.pth")
            if os.path.exists(p):
                self.set_log_alpha(float(torch.load(p, map_location="cpu").reshape(-1)[0]))
        self.update_target_network()

    @classmethod
    def _check_quantiles(cls, n_quantiles, drop):
        """(M, d) of the quantile critics, or (None, 0); ValueError before anything touches the device."""
        if n_quantiles is None:
            return None, 0

        def whole(x):
            return isinstance(x, (int, np.integer)) and not isinstance(x, (bool, np.bool_))
        if not whole(n_quantiles) or n_quantiles < 1:
            raise ValueError(f"n_quantiles must be None or an integer >= 1, got {n_quantiles!r}")
        if cls.N_CRITICS * int(n_quantiles) > 256:
            raise ValueError(f"n_quantiles = {n_quantiles}: {cls.N_CRITICS} critics x n_quantiles must be <= 256 "
                             f"(n_quantiles <= {256 // cls.N_CRITICS})")
        if not whole(drop) or not 0 <= drop < n_quantiles:
            raise ValueError(f"top_quantiles_to_drop_per_net must be an integer in [0, n_quantiles) = "
                             f"[0, {n_quantiles}), got {drop!r}")
        return int(n_quantiles), int(drop)

    def _target_entropy(self, ac_dim):
        return float(-ac_dim)            # :815

    def _polyak_now(self, step):
        return True                      # :1086

    def save_weights(self, path: str):   # :1102-1106
        self.actor.save(os.path.join(path, "actor.pth"))
        for i, critic in enumerate(self.critics):
            critic.save(os.path.join(path, f"critic_{i}.pth"))
        self._save_log_alpha(path)

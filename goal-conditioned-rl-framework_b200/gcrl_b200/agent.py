"""DDPG / TD3 agents over the CUDA learner (reference src/agent.py:12-386, 1173-1465).

Same constructor arguments, attributes and methods as the reference classes, so
``GoalEnvHER`` (src/env.py) drives them unchanged: ``update(step)`` returns tuples of the
same arity, ``save_weights`` writes ``actor.pth`` / ``critic.pth`` state_dicts with the
reference key names, the normaliser glue is identical.  All arithmetic of the hot path
(sample, relabel, reward, forward, backward, clip, Adam, Polyak) runs in
``libgcrl_b200.so``; this file is host plumbing only.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import random

import numpy as np

from . import _lib
from ._lib import AgentConfig, check, lib, np_ptr, vp
from .buffer import HERBuffer
from .replay import PERBuffer, ReplayBuffer

ALGO_DDPG, ALGO_TD3 = 0, 1
MAX_MANY_STEPS = 64         # GCRL_MAX_MANY_STEPS: updates per n-update graph launch
NET_ACTOR, NET_CRITIC, NET_T_ACTOR, NET_T_CRITIC, NET_CRITIC2, NET_T_CRITIC2 = range(6)


class CosineAnnealingLR:
    """Host scalar schedule = torch.optim.lr_scheduler.CosineAnnealingLR driven by
    ``step()`` once per optimiser step (recursive form; keeps oscillating past T_max
    like torch).  ``lr`` is what the next optimiser step uses (src/agent.py:1203-1212)."""

    def __init__(self, base_lr, T_max, eta_min):
        self.base_lr, self.T_max, self.eta_min = float(base_lr), int(T_max), float(eta_min)
        self.last_epoch = 0
        self.lr = float(base_lr)

    def step(self):
        self.last_epoch += 1
        e, T = self.last_epoch, self.T_max
        if (e - 1 - T) % (2 * T) == 0:
            self.lr = self.lr + (self.base_lr - self.eta_min) * (1 - math.cos(math.pi / T)) / 2
        else:
            self.lr = ((1 + math.cos(math.pi * e / T)) / (1 + math.cos(math.pi * (e - 1) / T))
                       * (self.lr - self.eta_min) + self.eta_min)
        return self.lr


class _NetView:
    """Stand-in for the reference's nn.Module attributes (``agent.actor`` ...): exposes
    ``state_dict`` / ``load_state_dict`` / ``save`` / ``load`` / ``eval`` / ``train`` with
    the reference checkpoint key names (src/model.py:24-37,64-74)."""

    def __init__(self, agent, net_id, prefix):
        self._agent, self._net, self._prefix = agent, net_id, prefix

    def eval(self):
        return self

    def train(self, mode=True):
        return self

    def layers(self):
        return self._agent._get_layers(self._net)

    def state_dict(self):
        import torch
        sd = {}
        for i, (w, b) in enumerate(self.layers()):
            sd[f"{self._prefix}.{2 * i}.weight"] = torch.from_numpy(w)
            sd[f"{self._prefix}.{2 * i}.bias"] = torch.from_numpy(b)
        return sd

    def load_state_dict(self, sd):
        n = self._agent._num_layers(self._net)
        layers = []
        for i in range(n):
            w = sd[f"{self._prefix}.{2 * i}.weight"]
            b = sd[f"{self._prefix}.{2 * i}.bias"]
            layers.append((np.asarray(w.detach().cpu().numpy() if hasattr(w, "detach") else w),
                           np.asarray(b.detach().cpu().numpy() if hasattr(b, "detach") else b)))
        self._agent._set_layers(self._net, layers)

    def save(self, path: str):
        import torch
        os.makedirs(os.path.dirname(path), exist_ok=True)
        torch.save(self.state_dict(), path)

    def load(self, weights: str, device: str = "cpu"):
        import torch
        self.load_state_dict(torch.load(weights, map_location="cpu"))


def _torch_init_mlp(in_dim, hidden, out_dim, layer_count):
    """Initial parameters with the reference's torch RNG consumption (src/model.py:12-27,
    39-42): nn.Linear default init per layer at construction, then xavier_uniform_ + bias
    0.01 over the layers in order."""
    import torch
    dims = [in_dim] + [hidden] * layer_count + [out_dim]
    lin = [torch.nn.Linear(dims[i], dims[i + 1]) for i in range(len(dims) - 1)]
    return _torch_xavier(lin)


def _torch_xavier(lin):
    import torch
    out = []
    for m in lin:
        torch.nn.init.xavier_uniform_(m.weight)
        m.bias.data.fill_(0.01)
        out.append((m.weight.detach().numpy().copy(), m.bias.detach().numpy().copy()))
    return out, lin


class _AgentBase:
    ALGO = ALGO_DDPG
    WEIGHT_DECAY = 0.0

    def __init__(self, obs_dim, ac_dim, config, weights, nenvs, gradient_step, *,
                 index_source="host", device=0, max_batch=None, seed=1898, precision=1,
                 goal_selection_strategy="future", online_sampling=False, n_step=1):
        """precision: 1 (default) runs the hidden-layer GEMMs of batches >= 2048 on the tcgen05 tensor
        cores with the 3xTF32 split (fp32-level accuracy, rel ~2e-6 per layer); 2 does so for every
        batch >= 128; 0 keeps every GEMM on the fp32 FFMA tiles.
        goal_selection_strategy / online_sampling / n_step: passed to the HER buffer (HERBuffer), n_step with
        config.gamma.  n_step > 1 needs buffer_type "HER" (ValueError otherwise).  The buffer's rows carry the n-step
        reward and a done column whose gamma*(1 - done) is gamma**k*(1 - done), so every update computes the n-step
        target unchanged; SAC / TQC take the entropy term at the bootstrap state only, as Stable-Baselines3 does."""
        self._init_common(obs_dim, ac_dim, config, nenvs, gradient_step, index_source, device, seed,
                          goal_selection_strategy, online_sampling, n_step)
        cfg = AgentConfig(algo=self.ALGO, state_dim=self.obs_dim, act_dim=self.ac_dim,
                          hidden_dim=config.hidden_dim, layer_count=config.layer_count,
                          max_batch=int(max_batch or config.batch_size), gamma=config.gamma,
                          tau=config.tau,
                          grad_clip=-1.0 if config.grad_clip is None else config.grad_clip,
                          policy_noise=config.policy_noise, noise_clamp=config.noise_clamp,
                          weight_decay=self.WEIGHT_DECAY, precision=int(precision), reserved=0)
        h = vp()
        check(lib.gcrl_agent_create(C.byref(h), self.device_index, C.byref(cfg)))
        self._h = h
        self._max_batch = int(max_batch or config.batch_size)
        self._metrics = (C.c_float * 8)()

    def _init_common(self, obs_dim, ac_dim, config, nenvs, gradient_step, index_source, device, seed,
                     goal_selection_strategy, online_sampling, n_step):
        _lib.require_cuda()
        self.device_index = int(device)
        self.device = f"cuda:{self.device_index}"
        self.config = config
        self.gradient_step = gradient_step
        self.obs_dim, self.ac_dim = int(obs_dim), int(ac_dim)
        self.index_source = index_source

        if n_step != 1 and config.buffer_type != "HER":
            raise ValueError(f"n_step > 1 needs the HER buffer (its episodes bound the window), got buffer_type "
                             f"{config.buffer_type!r}")
        if config.buffer_type == "HER":
            self.buffer = HERBuffer(config.max_len, config.max_eps_len, nenvs,
                                    k_future=config.k_future, index_source=index_source,
                                    seed=seed, device=device, goal_selection_strategy=goal_selection_strategy,
                                    online_sampling=online_sampling, n_step=n_step, gamma=config.gamma)
        elif config.buffer_type == "PER":                                  # src/agent.py:67-68
            self.buffer = PERBuffer(config.max_len, config.alpha, device=device)
        elif config.buffer_type == "REPLAY":                               # :69-70
            self.buffer = ReplayBuffer(config.max_len, device=device)
        else:
            raise ValueError(f"[ERROR] Invalid Buffer type. Received {config.buffer_type}.")

        self.noise_std = config.noise_std
        self.noise_clamp = config.noise_clamp
        self.policy_noise = config.policy_noise
        self.gamma = config.gamma
        self.batch_size = config.batch_size
        self.ac_update_freq = config.ac_update_freq
        self.grad_clip = config.grad_clip
        self.tau = config.tau
        self.beta = self.beta_start = config.beta
        self.beta_max = 1.0
        self.beta_end = config.beta_end

        self.actor_scheduler = CosineAnnealingLR(config.actor_lr, config.ac_scheduler_steps,
                                                 config.actor_lr_min)
        self.critic_scheduler = CosineAnnealingLR(config.critic_lr, config.cr_scheduler_steps,
                                                  config.critic_lr_min)

    def __del__(self):
        if getattr(self, "_h", None):
            lib.gcrl_agent_destroy(self._h)
            self._h = None

    # -- parameter exchange -------------------------------------------------------------
    def _stream(self):
        return _lib.current_stream(self.device_index)

    def _num_layers(self, net):
        return int(lib.gcrl_agent_num_layers(self._h, net))

    def _get_layers(self, net):
        out = []
        for layer in range(self._num_layers(net)):
            o, i = C.c_int(), C.c_int()
            check(lib.gcrl_agent_layer_shape(self._h, net, layer, C.byref(o), C.byref(i)))
            w = np.empty((o.value, i.value), np.float32)
            b = np.empty((o.value,), np.float32)
            check(lib.gcrl_agent_get_layer(self._h, net, layer, np_ptr(w), np_ptr(b), self._stream()))
            out.append((w, b))
        return out

    def _set_layers(self, net, layers):
        for layer, (w, b) in enumerate(layers):
            o, i = C.c_int(), C.c_int()
            check(lib.gcrl_agent_layer_shape(self._h, net, layer, C.byref(o), C.byref(i)))
            w = np.ascontiguousarray(w, np.float32)
            b = np.ascontiguousarray(b, np.float32)
            if w.shape != (o.value, i.value) or b.shape != (o.value,):
                raise ValueError(f"layer {layer}: expected {(o.value, i.value)}, got {w.shape}")
            check(lib.gcrl_agent_set_layer(self._h, net, layer, np_ptr(w), np_ptr(b), self._stream()))

    def hard_update(self):
        check(lib.gcrl_agent_hard_update(self._h, self._stream()))

    # -- reference API shared by all agents (src/agent.py:1368-1376, 1410-1465) -------------
    def push(self, state, action, reward, next_state, done):
        self.buffer.push(state, action, reward, next_state, done)

    def push_her(self, idx, state, action, next_state, reward, done, desired_goal, achieved_goal):
        self.buffer.push(idx, state, action, next_state, reward, done, desired_goal, achieved_goal)

    def is_buffer_filled(self):
        return len(self.buffer) >= self.batch_size

    def set_train(self):
        pass

    def set_eval(self):
        pass

    def beta_scheduler(self, step: int):
        self.beta = self._beta_at(step)

    def _beta_at(self, step):
        ratio = step / self.beta_end
        return min(self.beta_max, self.beta_start + ratio * (self.beta_max - self.beta_start))

    def update_normalizers(self, obs_list, dg_list, obs_normalize, g_normalize):
        if getattr(self.buffer, "obs_normalizer", None) is not None and obs_list and obs_normalize:
            self.buffer.obs_normalizer.update(np.concatenate(obs_list, axis=0))
        if getattr(self.buffer, "dg_normalizer", None) is not None and dg_list and g_normalize:
            self.buffer.dg_normalizer.update(np.concatenate(dg_list, axis=0))

    def normalize_obs(self, obs, normalize: bool):
        nz = getattr(self.buffer, "obs_normalizer", None)
        return nz.normalize(obs) if (nz is not None and normalize) else obs

    def normalize_goal(self, goal, normalize: bool):
        nz = getattr(self.buffer, "dg_normalizer", None)
        return nz.normalize(goal) if (nz is not None and normalize) else goal

    def normalize_state_batch(self, obs_batch, dg_batch, obs_normalize, g_normalize):
        return np.concatenate([self.normalize_obs(obs_batch, obs_normalize),
                               self.normalize_goal(dg_batch, g_normalize)], axis=-1)

    def _actor_forward(self, obs):
        obs = np.ascontiguousarray(obs, np.float32).reshape(-1, self.obs_dim)
        out = np.empty((obs.shape[0], self.ac_dim), np.float32)
        cap = int(self._max_batch)
        for lo in range(0, obs.shape[0], cap):       # any number of envs: the act scratch holds max_batch rows
            hi = min(obs.shape[0], lo + cap)
            o_, out_ = np.ascontiguousarray(obs[lo:hi]), np.empty((hi - lo, self.ac_dim), np.float32)
            check(lib.gcrl_agent_act(self._h, hi - lo, np_ptr(o_), np_ptr(out_), self._stream()))
            out[lo:hi] = out_
        return out

    def q_values(self, obs, act):
        obs = np.ascontiguousarray(obs, np.float32).reshape(-1, self.obs_dim)
        act = np.ascontiguousarray(act, np.float32).reshape(-1, self.ac_dim)
        out = np.empty((obs.shape[0], 1), np.float32)
        check(lib.gcrl_agent_q(self._h, obs.shape[0], np_ptr(obs), np_ptr(act), np_ptr(out),
                               self._stream()))
        return out

    def _flags(self, step):
        raise NotImplementedError

    # -- data parallel (one process per GPU; SURVEY 8e) -------------------------------------
    _dp = None

    def enable_peer_data_parallel(self, process_group=None):
        """Data parallelism without a collective library on the critical path: the ranks exchange CUDA-IPC
        handles of their flat gradient buffers once (through ``torch.distributed.all_gather_object``), and from
        then on every ``update()`` averages the critic / actor gradients and the batch-mean metrics over NVLink
        peer memory inside the one captured CUDA graph (flag barrier + every rank summing all ranks' buffers in
        rank order).  Same contract as ``enable_data_parallel``: every rank owns its episode shard, samples its
        local batch, and all ranks issue the same sequence of updates; replicas stay bit-identical."""
        import torch.distributed as dist
        rank, world = dist.get_rank(process_group), dist.get_world_size(process_group)
        n = C.c_int()
        check(lib.gcrl_agent_dp_export(self._h, None, C.byref(n)))
        buf = (C.c_ubyte * (64 * n.value))()
        check(lib.gcrl_agent_dp_export(self._h, C.cast(buf, vp), C.byref(n)))
        gathered = [None] * world
        dist.all_gather_object(gathered, bytes(buf), group=process_group)
        blob = b"".join(gathered)
        err = None
        try:
            check(lib.gcrl_agent_dp_connect(self._h, rank, world, C.cast(C.c_char_p(blob), vp)))
        except Exception as e:   # noqa: BLE001  (e.g. CUDA IPC not permitted in this container)
            err = e
        oks = [None] * world                    # all ranks take the same path
        dist.all_gather_object(oks, err is None, group=process_group)
        if not all(oks):
            if err is None:
                raise RuntimeError("a peer rank could not map the gradient buffers (CUDA IPC)")
            raise err
        dist.barrier(group=process_group)
        self._dp = None
        self._peer_dp = (rank, world)

    def peer_barrier(self):
        """One flag barrier over the peer-connected ranks on the current stream (no host synchronisation)."""
        check(lib.gcrl_agent_dp_barrier(self._h, self._stream()))

    def enable_data_parallel(self, process_group=None, allreduce_mean=None):
        """Average gradients over the ranks of ``process_group`` (torch.distributed, NCCL over
        NVLink) between the backward and the optimiser phases of every update.  Each rank keeps
        its own episode shard of the buffer and samples its local minibatch; weights, optimiser
        state and targets stay replicated because every rank applies the same averaged
        gradient.  ``allreduce_mean(tensor)`` overrides the collective (tests)."""
        from .parallel import GradAverager
        self._dp = GradAverager(self, process_group, allreduce_mean)
        return self._dp

    def grad_tensor(self, net):
        """The flat fp32 gradient buffer of a trainable network as a torch tensor (zero copy)."""
        from .parallel import device_tensor
        ptr, n = vp(), C.c_int64()
        check(lib.gcrl_agent_grad_buffer(self._h, net, C.byref(ptr), C.byref(n)))
        return device_tensor(ptr.value, n.value, self.device_index)

    def metrics_tensor(self):
        from .parallel import device_tensor
        ptr = vp()
        check(lib.gcrl_agent_metrics_buffer(self._h, C.byref(ptr)))
        return device_tensor(ptr.value, 8, self.device_index)

    def _trainable_critics(self):
        return (NET_CRITIC,)

    # -- uniform / prioritised replay behind update() (src/agent.py:1380-1394 and the twins in TD3 / SAC / TQC) --
    _per = None
    _replay_out = None
    _last_td = None

    def _per_ptrs(self):
        if self._per is None:
            w, td = vp(), vp()
            check(lib.gcrl_agent_per_buffers(self._h, C.byref(w), C.byref(td)))
            self._per = (w, td)
        return self._per

    def _replay_batch(self, B):
        """Draw the batch of a non-HER buffer into device tensors.  Returns (batch, prioritised?); for a
        PERBuffer the importance weights land in the agent's weight array (read by the critic loss when flags
        bit3 is set) and nothing comes back to the host."""
        buf = self.buffer
        assert len(buf) >= B, "Not enough in buffer to sample"
        buf._flush()
        if self._replay_out is None or self._replay_out[0].shape[0] != B:
            self._replay_out = buf._outputs(B)          # reused: the update copies the batch before it returns
        if isinstance(buf, PERBuffer):
            buf.sample_into(B, self.beta, self._replay_out, self._per_ptrs()[0])
            return tuple(self._replay_out), True
        buf.sample_into(B, self._replay_out)
        return tuple(self._replay_out), False

    def _replay_finish(self, B):
        """buffer.update_priorities(indices, td_error) (:1387) on the device, then the per-sample TD errors the
        reference returns in place of their mean (:1338-1340)."""
        from .parallel import device_tensor
        td_ptr = self._per_ptrs()[1]
        self.buffer.update_priorities_last(B, td_ptr)
        return device_tensor(td_ptr.value, B, self.device_index).cpu().numpy().reshape(B, 1)

    def _run_update(self, step, batch=None, indices=None, noise=None, sync=True):
        """One update; ``batch`` = 5 device tensors (explicit batch) or None (sample from the
        buffer; ``indices`` optional host positions).  Returns the raw 8-float metric vector
        (or None when sync=False)."""
        flags = self._flags(step)
        lr_c, lr_a = self.critic_scheduler.lr, self.actor_scheduler.lr
        mptr = C.cast(self._metrics, vp) if sync else None
        nptr = vp(noise.data_ptr()) if noise is not None else None
        iptr = None
        predraw = False
        per = False
        if batch is None and not isinstance(self.buffer, HERBuffer):
            batch, per = self._replay_batch(self.batch_size)
            if per:
                flags |= 8
        if batch is None:
            B = self.batch_size
            assert len(self.buffer) >= B, "[ERROR] Not enough in buffer to sample"
            if indices is None and self.index_source == "host":
                indices = self._take_predrawn(B)
                predraw = sync
            if indices is not None:
                indices = np.ascontiguousarray(indices, np.int64)
                iptr = np_ptr(indices)
            bufh, ptrs = self.buffer.handle, (None,) * 5
        else:
            B = batch[0].shape[0]
            bufh, ptrs = None, tuple(vp(t.data_ptr()) for t in batch)      # s, a, r, ns, d
        if self._dp is not None:
            st = self._stream()
            for phase in range(4):
                check(lib.gcrl_agent_update_phase(self._h, phase, bufh, B, iptr, *ptrs, nptr, lr_c, lr_a,
                                                  flags, st))
                if phase == 0:
                    self._dp.average(self._trainable_critics())
                elif phase == 2 and (flags & 1):
                    self._dp.average((NET_ACTOR,))
            if sync:
                if predraw:
                    self._predraw(B)       # host work hidden behind the queued phases and all-reduces
                self._dp.average_metrics()
                check(lib.gcrl_agent_read_metrics(self._h, mptr, st))
        elif batch is None:
            if predraw:
                # launch asynchronously, draw the NEXT call's positions while the GPU works, then read back
                check(lib.gcrl_agent_update_from_buffer(self._h, bufh, B, iptr, nptr, lr_c, lr_a, flags, None,
                                                        self._stream()))
                self._predraw(B)
                check(lib.gcrl_agent_read_metrics(self._h, mptr, self._stream()))
            else:
                check(lib.gcrl_agent_update_from_buffer(self._h, bufh, B, iptr, nptr, lr_c, lr_a, flags, mptr,
                                                        self._stream()))
        else:
            check(lib.gcrl_agent_update_batch(self._h, B, *ptrs, nptr, lr_c, lr_a, flags, mptr,
                                              self._stream()))
        self._last_td = self._replay_finish(B) if per else None
        self.critic_scheduler.step()
        if flags & 1:
            self.actor_scheduler.step()
        return [float(x) for x in self._metrics] if sync else None

    # -- true resume (SURVEY 8f-3): everything update() depends on, beyond the reference's weight files ----
    def _all_nets(self):
        return [n for n in range(6) if self._num_layers(n) > 0]

    def _trainable_nets(self):
        return (NET_ACTOR,) + tuple(self._trainable_critics())

    def state_dict(self):
        """Weights of every network (targets included), Adam moments and step counts, both learning-rate
        schedules and the PER beta schedule: restoring it makes the next update() bit-identical to the
        one an uninterrupted run would have made on the same batch."""
        import torch
        out = {"algo": self.ALGO, "nets": {}, "adam": {}, "beta": self.beta}
        for net in self._all_nets():
            out["nets"][net] = [(torch.from_numpy(w), torch.from_numpy(b)) for w, b in self._get_layers(net)]
        for net in self._trainable_nets():
            layers = []
            for layer, (w, b) in enumerate(self._get_layers(net)):
                mw, vw = np.empty_like(w), np.empty_like(w)
                mb, vb = np.empty_like(b), np.empty_like(b)
                check(lib.gcrl_agent_get_adam_layer(self._h, net, layer, np_ptr(mw), np_ptr(mb), np_ptr(vw), np_ptr(vb),
                                                    self._stream()))
                layers.append(tuple(torch.from_numpy(x) for x in (mw, mb, vw, vb)))
            step = C.c_int()
            check(lib.gcrl_agent_get_adam_step(self._h, net, C.byref(step)))
            out["adam"][net] = {"step": int(step.value), "layers": layers}
        for name, sch in (("actor_scheduler", self.actor_scheduler), ("critic_scheduler", self.critic_scheduler)):
            out[name] = {"last_epoch": sch.last_epoch, "lr": sch.lr}
        return out

    def load_state_dict(self, sd):
        if sd["algo"] != self.ALGO:
            raise ValueError("checkpoint belongs to a different agent type")
        for net, layers in sd["nets"].items():
            self._set_layers(int(net), [(w.numpy(), b.numpy()) for w, b in layers])
        for net, st in sd["adam"].items():
            for layer, arrs in enumerate(st["layers"]):
                mw, mb, vw, vb = (np.ascontiguousarray(x.numpy(), np.float32) for x in arrs)
                check(lib.gcrl_agent_set_adam_layer(self._h, int(net), layer, np_ptr(mw), np_ptr(mb), np_ptr(vw),
                                                    np_ptr(vb), self._stream()))
            check(lib.gcrl_agent_set_adam_step(self._h, int(net), int(st["step"])))
        for name in ("actor_scheduler", "critic_scheduler"):
            sch = getattr(self, name)
            sch.last_epoch, sch.lr = int(sd[name]["last_epoch"]), float(sd[name]["lr"])
        self.beta = sd["beta"]

    def save_checkpoint(self, path: str, with_buffer: bool = True):
        """save_weights(path) (the reference's files) plus ``trainer_state.pt`` (targets, Adam, schedulers,
        the interpreter's ``random`` state) and ``buffer_state.pt`` (the replay buffer's live window) for a
        true resume."""
        import torch
        self.save_weights(path)
        st = self.state_dict()
        st["python_random"] = random.getstate()
        st["numpy_random"] = np.random.get_state()        # PERBuffer.sample draws from NumPy's global stream
        torch.save(st, os.path.join(path, "trainer_state.pt"))
        if with_buffer:
            torch.save(self.buffer.state_dict(), os.path.join(path, "buffer_state.pt"))

    def load_checkpoint(self, path: str):
        import torch
        st = torch.load(os.path.join(path, "trainer_state.pt"), map_location="cpu", weights_only=False)
        self.load_state_dict(st)
        bpath = os.path.join(path, "buffer_state.pt")
        if os.path.exists(bpath):
            self.buffer.load_state_dict(torch.load(bpath, map_location="cpu", weights_only=False))
        if "python_random" in st:
            random.setstate(st["python_random"])
        if "numpy_random" in st:
            np.random.set_state(st["numpy_random"])
        self._pre = None

    # -- host index stream: latency hiding without changing the Mersenne-Twister stream ---------------
    # ``random.sample(range(len), B)`` costs ~0.1 ms of host time per update.  The draw for the next
    # update is made while the GPU executes the current one, and the global ``random`` state is put
    # back right away; the next update uses the pre-drawn positions only if the state it finds is
    # exactly the one that was put back (nobody consumed the stream in between, same buffer length and
    # batch), and then advances the state to where its own draw would have left it.  Any other
    # consumer (apply_her's randint, select_action's random.random, a reseed) therefore sees precisely
    # the reference's interleaving.
    _pre = None

    _known_state = None     # the tuple the global generator was just set to (by _take_predrawn), if still current

    def _predraw(self, B):
        if _lib.direct_stream_available():
            return          # drawing in place from the interpreter's generator costs ~6 us: nothing worth hiding
        n = len(self.buffer)
        # right after a successful _take_predrawn the global state IS the tuple it installed: no getstate(),
        # and the C mirror recognises its own tuple and skips the 624-word conversion
        before, self._known_state = self._known_state, None
        if before is None:
            before = random.getstate()
        idx, after = _lib.py_sample_range_from(before, n, B)     # C mirror of random.sample; global state untouched
        self._pre = (before, after, idx, n, B)

    def _take_predrawn(self, B):
        pre, self._pre = self._pre, None
        n = len(self.buffer)
        if pre is None and _lib.direct_stream_available():
            return _lib.py_sample_range(n, B)
        if pre is not None and pre[3] == n and pre[4] == B and random.getstate() == pre[0]:
            random.setstate(pre[1])
            self._known_state = pre[1]
            return pre[2]
        self._known_state = None
        return _lib.py_sample_range(n, B)

    def read_metrics(self):
        check(lib.gcrl_agent_read_metrics(self._h, C.cast(self._metrics, vp), self._stream()))
        return [float(x) for x in self._metrics]

    # -- a training cycle's gradient steps in one call ---------------------------------------------------
    # What the family's n-update calls take: their C functions (HER buffer, REPLAY / PER buffer), the metric floats of
    # an update, the smallest batch, and (SAC / TQC) the BatchNorm batches an update counts without / with an actor step
    _MANY_FNS = ("gcrl_agent_update_many", "gcrl_agent_update_many_replay")
    _METRIC_WIDTH = 8
    _MIN_BATCH = 1
    _BN_BATCHES = None

    def update_many(self, steps):
        """``[self.update(s) for s in steps]``: the same tuples, and afterwards the same state of every network,
        optimiser, schedule, beta, buffer (ring, priorities, last positions), index stream and random generator.
        ``steps`` need not be consecutive.

        DDPG, TD3, SAC and TQC on one GPU issue every 64 steps as ONE CUDA graph launch, whatever the buffer: the
        positions (HER host index stream, ``random.sample`` of REPLAY), the uniforms and beta of every PER draw,
        the learning rates and the noise (TD3 smoothing, SAC / TQC rsample) of all of them are drawn up front in
        the loop's order and travel in one copy each, so no interpreter, launch, priority round trip or metric
        read-back sits between the updates.  With PER, each update's draw reads the priorities the previous one
        wrote; while the ring is still filling, each call issues its updates without a graph.  Both data-parallel
        modes run the loop."""
        steps = [int(s) for s in steps]
        if self._dp is not None or getattr(self, "_peer_dp", None) is not None:
            return [self.update(s) for s in steps]
        out = []
        for lo in range(0, len(steps), MAX_MANY_STEPS):
            out += self._update_chunk(steps[lo:lo + MAX_MANY_STEPS])
        return out

    def _many_noise(self, B, flags):
        """The device noise update() draws for each of these updates, in step order: the tensors the n-update call
        takes (None: a NULL pointer)."""
        return (None,)

    def _step_schedules(self, flags):
        """The learning rates of n updates with these flags: the schedules step as update() steps them.  Returns
        (lr_critic[n], lr_actor[n], the schedules' state before) for _restore_schedules on a refused call."""
        n = len(flags)
        lr_c, lr_a = (C.c_double * n)(), (C.c_double * n)()
        saved = [(sch.last_epoch, sch.lr) for sch in (self.critic_scheduler, self.actor_scheduler)]
        for i, f in enumerate(flags):
            lr_c[i], lr_a[i] = self.critic_scheduler.lr, self.actor_scheduler.lr
            self.critic_scheduler.step()
            if f & 1:
                self.actor_scheduler.step()
        return lr_c, lr_a, saved

    def _restore_schedules(self, saved):
        for sch, (epoch, lr) in zip((self.critic_scheduler, self.actor_scheduler), saved):
            sch.last_epoch, sch.lr = epoch, lr

    def _update_chunk(self, steps):
        """Up to MAX_MANY_STEPS updates in one C call.  update()'s host draws for every step are made up front, each
        generator in step order: the noise, then the positions ``random.sample(range(len), B)`` (REPLAY, HER with the
        host index stream) or the uniforms ``np.random.random_sample(B)`` and the beta each draw uses -- the one
        beta_scheduler(step) left after the update before (PER)."""
        B, n = self.batch_size, len(steps)
        her, per = isinstance(self.buffer, HERBuffer), isinstance(self.buffer, PERBuffer)
        # what update() checks, before any generator is touched
        assert len(self.buffer) >= B, ("[ERROR] " if her else "") + "Not enough in buffer to sample"
        if not self._MIN_BATCH <= B <= self._max_batch:
            raise ValueError(f"batch size {B} outside [{self._MIN_BATCH}, max_batch = {self._max_batch}]")
        flags = [self._flags(s) | (8 if per else 0) for s in steps]
        noise = self._many_noise(B, flags)       # referenced until the call has copied it
        pos = u = beta = None
        if per:
            u = np.stack([np.random.random_sample(B) for _ in steps])
            betas, b = [], self.beta
            for s in steps:
                betas.append(b)
                b = self._beta_at(s)
            beta = np.array(betas, np.float64)
        elif not her or self.index_source == "host":
            self._pre = self._known_state = None        # the host index stream's pre-drawn positions are stale
            nlen = len(self.buffer)
            pos = np.stack([_lib.py_sample_range(nlen, B) for _ in steps])
        cflags = (C.c_int * n)(*flags)
        lr_c, lr_a, saved = self._step_schedules(flags)
        metrics = np.empty((n, self._METRIC_WIDTH), np.float32)
        td = np.empty((n, B), np.float32) if per else None

        def ptr(x):
            return None if x is None else np_ptr(x)
        nptrs = [None if t is None else vp(t.data_ptr()) for t in noise]
        if her:
            fn, draws, tail = self._MANY_FNS[0], (ptr(pos),), ()
        else:
            fn, draws, tail = self._MANY_FNS[1], (ptr(pos), ptr(u), ptr(beta)), (ptr(td),)
        try:
            check(getattr(lib, fn)(self._h, self.buffer.handle, B, n, cflags, *draws, *nptrs, lr_c, lr_a,
                                   np_ptr(metrics), *tail, self._stream()))
        except BaseException:
            self._restore_schedules(saved)
            raise
        return self._many_results(steps, flags, metrics, td)

    def _many_results(self, steps, flags, metrics, td):
        """What update() does after its call, for every step in order: the TD array (PER), the BatchNorm batch count
        (SAC / TQC), beta and the returned tuple."""
        out = []
        for i, (step, f, m) in enumerate(zip(steps, flags, metrics.tolist())):
            self._last_td = td[i].reshape(-1, 1) if td is not None else None
            if self._BN_BATCHES is not None:
                self._bn_batches += self._BN_BATCHES[f & 1]
            self.beta_scheduler(step)
            out.append(self._result(step, m))
        return out


class DDPG(_AgentBase):
    """Reference src/agent.py:1173-1465."""
    ALGO = ALGO_DDPG
    WEIGHT_DECAY = 0.0          # torch.optim.Adam (:1201-1202)
    POLYAK_EVERY = 40           # literal at :1397

    def __init__(self, obs_dim, ac_dim, config, weights, nenvs, gradient_step, **kw):
        super().__init__(obs_dim, ac_dim, config, weights, nenvs, gradient_step, **kw)
        H, L = config.hidden_dim, config.layer_count
        self.actor = _NetView(self, NET_ACTOR, "base_net")
        self.target_actor = _NetView(self, NET_T_ACTOR, "base_net")
        self.critic = _NetView(self, NET_CRITIC, "net")
        self.target_critic = _NetView(self, NET_T_CRITIC, "net")
        # same construction order / RNG consumption as :1187-1198
        self._lin = {}
        for net, (i, o) in ((NET_ACTOR, (obs_dim, ac_dim)), (NET_T_ACTOR, (obs_dim, ac_dim)),
                            (NET_CRITIC, (obs_dim + ac_dim, 1)), (NET_T_CRITIC, (obs_dim + ac_dim, 1))):
            params, self._lin[net] = _torch_init_mlp(i, H, o, L)
            self._set_layers(net, params)
        if weights:
            self.actor.load(os.path.join(weights, "actor.pth"))
            critic_path = os.path.join(weights, "critic.pth")
            if not os.path.exists(critic_path):
                critic_path = os.path.join(weights, "critic_1.pth")
            self.critic.load(critic_path)
        self.update_target_network()

    def update_target_network(self, hard_update: bool = True, tau: float = 0.005):      # :1255-1271
        if hard_update:
            self.hard_update()
        else:
            check(lib.gcrl_agent_soft_update(self._h, 3, float(tau), self._stream()))

    def _flags(self, step):
        return (1 if step % self.ac_update_freq == 0 else 0) | (2 if step % self.POLYAK_EVERY == 0 else 0)

    def select_action(self, obs_tensor, eval_action: bool = False):          # :1345-1366
        if not eval_action:
            if random.random() < 0.2:
                return np.clip(np.random.randn(obs_tensor.shape[0], self.ac_dim), a_min=-1, a_max=1)
            action = np.tanh(self._actor_forward(obs_tensor))   # second tanh, as the reference
            noise = np.random.normal(0, self.noise_std, size=action.shape)
            return np.clip(action + noise, -1, 1)
        return np.clip(np.tanh(self._actor_forward(obs_tensor)), -1, 1)

    def update(self, step: int, batch=None, indices=None):                    # :1378-1404
        m = self._run_update(step, batch=batch, indices=indices)
        self.beta_scheduler(step)
        return self._result(step, m)

    def _result(self, step, m):
        critic_loss, ac_loss, td, q, cg, agn = m[0], m[1], np.float32(m[2]), m[3], m[4], m[5]
        if self._last_td is not None:          # prioritised replay: the per-sample array (:1338-1340)
            td = self._last_td
        if step % self.ac_update_freq == 0:
            return critic_loss, ac_loss, td, q, cg, agn
        return critic_loss, td, q, cg

    def update_async(self, step: int, batch=None, indices=None):
        """update() without the host read-back; metrics via read_metrics()."""
        self._run_update(step, batch=batch, indices=indices, sync=False)

    def save_weights(self, path: str):                                        # :1406-1408
        self.actor.save(os.path.join(path, "actor.pth"))
        self.critic.save(os.path.join(path, "critic.pth"))

    def reset(self):                                                          # :1461-1465
        for net in (NET_ACTOR, NET_T_ACTOR, NET_CRITIC, NET_T_CRITIC):
            params, _ = _torch_xavier(self._lin[net])
            self._set_layers(net, params)


class TD3Agent(_AgentBase):
    """Reference src/agent.py:12-386."""
    ALGO = ALGO_TD3
    WEIGHT_DECAY = 0.01         # torch.optim.AdamW default (:46-48)

    def __init__(self, obs_dim, ac_dim, config, weights, nenvs, gradient_step, **kw):
        super().__init__(obs_dim, ac_dim, config, weights, nenvs, gradient_step, **kw)
        H, L = config.hidden_dim, config.layer_count
        self.actor = _NetView(self, NET_ACTOR, "base_net")
        self.target_actor = _NetView(self, NET_T_ACTOR, "base_net")
        self.critic_1 = _NetView(self, NET_CRITIC, "net")
        self.critic_2 = _NetView(self, NET_CRITIC2, "net")
        self.target_critic_1 = _NetView(self, NET_T_CRITIC, "net")
        self.target_critic_2 = _NetView(self, NET_T_CRITIC2, "net")
        self._lin = {}
        ci = obs_dim + ac_dim
        for net, (i, o) in ((NET_ACTOR, (obs_dim, ac_dim)), (NET_T_ACTOR, (obs_dim, ac_dim)),
                            (NET_CRITIC, (ci, 1)), (NET_CRITIC2, (ci, 1)),
                            (NET_T_CRITIC, (ci, 1)), (NET_T_CRITIC2, (ci, 1))):   # order of :25-44
            params, self._lin[net] = _torch_init_mlp(i, H, o, L)
            self._set_layers(net, params)
        if weights:
            self.actor.load(os.path.join(weights, "actor.pth"))
            self.critic_1.load(os.path.join(weights, "critic_1.pth"))
            self.critic_2.load(os.path.join(weights, "critic_2.pth"))
        self.update_target_network()

    def update_target_network(self):
        self.hard_update()

    def update_actor(self, tau: float = 0.005):                                          # :117-121
        check(lib.gcrl_agent_soft_update(self._h, 1, float(tau), self._stream()))

    def update_critic(self, tau: float = 0.005):                                         # :123-132
        check(lib.gcrl_agent_soft_update(self._h, 2, float(tau), self._stream()))

    def _trainable_critics(self):
        return (NET_CRITIC, NET_CRITIC2)

    def _flags(self, step):
        return 1 if step % self.ac_update_freq == 0 else 0

    def select_action(self, obs_tensor, eval_action: bool = False):          # :253-269
        if not eval_action:
            action = np.tanh(self._actor_forward(obs_tensor))
            noise = np.random.normal(0, self.noise_std, size=action.shape)
            return np.clip(action + noise, -1, 1)
        return self._actor_forward(obs_tensor)

    def update(self, step: int, batch=None, indices=None, noise=None):        # :281-317
        import torch
        B = self.batch_size if batch is None else batch[0].shape[0]
        if noise is None:   # torch.randn_like(action) on the device (:175)
            noise = torch.randn((B, self.ac_dim), dtype=torch.float32, device=self.device)
        m = self._run_update(step, batch=batch, indices=indices, noise=noise)
        self.beta_scheduler(step)
        return self._result(step, m)

    def _many_noise(self, B, flags):
        """n separate draws of update()'s noise, in step order: the CUDA generator advances as under the loop."""
        import torch
        return (torch.stack([torch.randn((B, self.ac_dim), dtype=torch.float32, device=self.device) for _ in flags]),)

    def _result(self, step, m):
        q1l, acl, td, q, c1g, acg, q2l, c2g = m
        td = np.float32(td) if self._last_td is None else self._last_td
        if step % self.ac_update_freq == 0:
            return q1l, q2l, acl, td, q, c1g, c2g, acg
        return q1l, q2l, td, q, c1g, c2g

    def save_weights(self, path: str):                                        # :319-322
        self.actor.save(os.path.join(path, "actor.pth"))
        self.critic_1.save(os.path.join(path, "critic_1.pth"))
        self.critic_2.save(os.path.join(path, "critic_2.pth"))

    def reset(self):                                                          # :379-386
        for net in (NET_ACTOR, NET_T_ACTOR, NET_CRITIC, NET_CRITIC2, NET_T_CRITIC, NET_T_CRITIC2):
            params, _ = _torch_xavier(self._lin[net])
            self._set_layers(net, params)

"""GPU: SAC / TQC ``update_many(steps)`` -- a training cycle's gradient steps as one CUDA graph launch per 64 steps
(csrc/sac.cu: gcrl_sac_update_many) -- against the loop ``[update(s) for s in steps]`` it replaces.

  * bit identity with the loop: every returned tuple (values and types), the actor's Linears and BatchNorm
    parameters / running statistics, every online and target critic, log_alpha, both schedules, beta, the
    BatchNorm batch count and the interpreter / NumPy / torch CUDA random states; then one more plain update()
    on each agent (SAC / TQC export no AdamW moments: a moment or step counter that differs shows there).
    Precision 0 at B = 64, 256, 1024; precision 2 at B = 256 (tcgen05 below the precision-1 switch); precision 1
    at B = 2048 (the ensemble's batched backward) and 4608 (above kEnsembleBatchMax: the per-critic loop);
    host and device index streams; step lists that cross Polyak, actor and alpha_min_steps boundaries, span two
    chunks, or repeat and go backwards;
  * a replayed graph reads this call's buffer totals, positions and scalars, not the captured ones;
  * one cudaGraphLaunch per chunk, no stream synchronisation, one device-to-host copy per chunk (the metric
    rows, after the last update), and the same kernel count as the loop;
  * refused calls leave no trace; sync-BN and phase-wise data-parallel agents run the loop;
  * GCRL_B200_NO_GRAPH=1 equals the graph path.
"""
import ctypes as C

import numpy as np
import pytest

from tests.helpers import bits
from tests.test_ddpg_gpu import synthetic_episodes
from tests.test_sac_gpu import sac_config
from tests.test_update_many_gpu import rng_states, same_results, same_rng_states, seed_all

pytestmark = pytest.mark.gpu

D, A, G = 22, 3, 3
ALPHA_MIN_STEPS = 50
STEP_LISTS = {"range37_82": list(range(37, 82)), "two_chunks": list(range(1, 71)), "unordered": [5, 5, 40, 3]}


def make_agent(algo, B, index_source="host", episodes=None, hidden=64, precision=0):
    """Seeded weights; the buffer holds seeded episodes, enough that the oldest are partly evicted."""
    import torch
    from gcrl_b200 import SACAgent, TQCAgent
    max_len = 2 * B + 100
    cfg = sac_config(hidden_dim=hidden, batch_size=B, max_len=max_len, ac_update_freq=2,
                     alpha_min_steps=ALPHA_MIN_STEPS, alpha_lr=1e-2, actor_lr=1e-3, actor_lr_min=1e-4,
                     ac_scheduler_steps=30, critic_lr=1e-3, critic_lr_min=1e-4, cr_scheduler_steps=25, beta=0.4,
                     beta_end=100)
    torch.manual_seed(5)
    ag = (SACAgent if algo == "sac" else TQCAgent)(D, A, cfg, None, 1, 40, index_source=index_source,
                                                    precision=precision)
    eps = episodes if episodes is not None else synthetic_episodes(B, max_len // 200 + 3, D, A, G)
    for ep in eps:
        ag.buffer.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], ep["fut"])
    assert len(ag.buffer) >= B and ag.buffer.max_mem_len == max_len
    return ag


def episodes_for(B):
    return synthetic_episodes(B, (2 * B + 100) // 200 + 3, D, A, G)


def sac_state(ag):
    L = ag.config.layer_count
    out = []
    for l in range(L + 2):
        out += list(ag.actor.linear(l))
    for l in range(L):
        out += list(ag.actor.bn(l))               # weight, bias, running mean, running var
    for view in ag._critic_views + ag._target_views:
        for w, b in view.layers():
            out += [w, b]
    out.append(np.float32(ag.get_log_alpha()))
    return out


def assert_same_state(a1, a2):
    for i, (x, y) in enumerate(zip(sac_state(a1), sac_state(a2))):
        assert np.array_equal(bits(x), bits(y)), i
    for name in ("critic_scheduler", "actor_scheduler"):
        s1, s2 = getattr(a1, name), getattr(a2, name)
        assert (s1.last_epoch, s1.lr) == (s2.last_epoch, s2.lr), name
    assert a1.beta == a2.beta and a1._bn_batches == a2._bn_batches


def loop_vs_many(a_loop, a_many, steps):
    seed_all()
    r_loop = [a_loop.update(s) for s in steps]
    st_loop = rng_states()
    seed_all()
    r_many = a_many.update_many(steps)
    st_many = rng_states()
    same_results(r_loop, r_many)
    assert same_rng_states(st_loop, st_many)
    return r_loop


def one_more_update(a1, a2, step=83):
    seed_all()
    u1 = a1.update(step)
    seed_all()
    u2 = a2.update(step)
    same_results([u1], [u2])


def last_metrics(ag, step):
    from gcrl_b200._lib import check, lib
    out = (C.c_float * 12)()
    check(lib.gcrl_sac_read_metrics(ag._h, ag._flags(step), C.cast(out, C.c_void_p), ag._stream()))
    return np.array(out, np.float32)


# ---- 1. bit identity against the loop --------------------------------------------------------------------------
CASES = [(64, 64, 0), (256, 64, 0), (1024, 64, 0), (256, 64, 2), (2048, 256, 1), (4608, 256, 1)]


@pytest.mark.parametrize("index_source", ["host", "device"])
@pytest.mark.parametrize("algo", ["sac", "tqc"])
@pytest.mark.parametrize("B,H,precision", CASES, ids=[f"p{p}_B{b}_H{h}" for b, h, p in CASES])
def test_update_many_equals_the_loop_bitwise(B, H, precision, algo, index_source, monkeypatch):
    """The three step lists in turn on the same pair of agents (later lists replay graphs of earlier flag patterns
    where they repeat), everything compared after each, then one more plain update()."""
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    eps = episodes_for(B)
    a_loop, a_many = (make_agent(algo, B, index_source, eps, H, precision) for _ in range(2))
    for name, steps in STEP_LISTS.items():
        loop_vs_many(a_loop, a_many, steps)
        assert_same_state(a_loop, a_many)
        assert np.array_equal(bits(last_metrics(a_loop, steps[-1])), bits(last_metrics(a_many, steps[-1]))), name
    one_more_update(a_loop, a_many)
    assert_same_state(a_loop, a_many)


# ---- 2. the same graph, different contents --------------------------------------------------------------------
@pytest.mark.parametrize("index_source", ["host", "device"])
@pytest.mark.parametrize("algo", ["sac", "tqc"])
def test_replayed_graph_reads_the_new_buffer_state(algo, index_source, monkeypatch):
    """Two calls with one flag pattern (the second replays the first's graph); between them new episodes are
    committed to both buffers, which moves the totals and evicts old entries."""
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    B = 256
    more = synthetic_episodes(B + 1, 3, D, A, G)
    a_loop, a_many = (make_agent(algo, B, index_source, episodes_for(B)) for _ in range(2))
    loop_vs_many(a_loop, a_many, list(range(81, 121)))
    for ag in (a_loop, a_many):
        n0, t0 = len(ag.buffer), ag.buffer.state_dict()["episodes"][0]["s"][0].copy()
        for ep in more:
            ag.buffer.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], ep["fut"])
        assert len(ag.buffer) == n0 and not np.array_equal(ag.buffer.state_dict()["episodes"][0]["s"][0], t0)
    loop_vs_many(a_loop, a_many, list(range(121, 161)))          # 40 steps later: the same flags
    assert_same_state(a_loop, a_many)


# ---- 3. one launch per chunk ---------------------------------------------------------------------------------
@pytest.mark.parametrize("algo,B,H,precision", [("sac", 256, 64, 0), ("tqc", 256, 64, 0), ("tqc", 2048, 256, 1)],
                         ids=["sac_p0_B256", "tqc_p0_B256", "tqc_p1_B2048_tcgen05"])
def test_one_graph_launch_per_chunk(algo, B, H, precision, monkeypatch):
    """Under torch.profiler, a warmed-up call of 70 steps issues two cudaGraphLaunch calls, instantiates no graph,
    synchronises no stream and copies device to host once per chunk; gcrl_kernel_launches() grows as under the
    loop."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from gcrl_b200._lib import lib
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    eps = episodes_for(B)
    a_loop, a_many = (make_agent(algo, B, "device", eps, H, precision) for _ in range(2))
    # both lists lie past alpha_min_steps and 80 apart: same actor / Polyak / alpha pattern, the graphs repeat
    warm, steps = list(range(81, 151)), list(range(161, 231))
    loop_vs_many(a_loop, a_many, warm)
    k0 = lib.gcrl_kernel_launches()
    seed_all()
    r_loop = [a_loop.update(s) for s in steps]
    k_loop = lib.gcrl_kernel_launches() - k0
    seed_all()
    torch.cuda.synchronize()
    k1 = lib.gcrl_kernel_launches()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        r_many = a_many.update_many(steps)
        torch.cuda.synchronize()
    k_many = lib.gcrl_kernel_launches() - k1
    same_results(r_loop, r_many)
    names = [e.name for e in prof.events()]
    launches = sum(n in ("cudaGraphLaunch", "cuGraphLaunch") for n in names)
    assert launches == 2, sorted(set(names))
    assert not any("GraphInstantiate" in n for n in names)
    d2h = [n for n in names if "DtoH" in n or "Device -> Pinned" in n or "Device -> Pageable" in n]
    assert len(d2h) == 2, d2h                     # the metric rows of each chunk, once
    syncs = [n for n in names if "StreamSynchronize" in n]
    assert len(syncs) <= 1, syncs                 # the test's own torch.cuda.synchronize() only
    assert k_many == k_loop > 0
    if precision == 1:
        assert any("tc_dense" in n for n in names), "the tcgen05 engine did not run"


# ---- 4. errors leave no trace; the data-parallel modes loop ---------------------------------------------------
def update_many_c(ag, n, flags=0):
    """gcrl_sac_update_many with n updates of `flags` (host positions 0..B-1 on the host index stream)."""
    import torch
    from gcrl_b200._lib import check, lib, np_ptr
    B = ag.batch_size
    m = max(n, 1)
    cflags = (C.c_int * m)(*([flags] * m))
    lr = (C.c_double * m)(*([1e-3] * m))
    idx = np.tile(np.arange(B, dtype=np.int64), (m, 1))
    noise = torch.zeros((m, B, A), dtype=torch.float32, device="cuda")
    out = np.empty((m, 12), np.float32)
    ptr = C.c_void_p(noise.data_ptr())
    check(lib.gcrl_sac_update_many(ag._h, ag.buffer.handle, B, n, cflags,
                                   np_ptr(idx) if ag.index_source == "host" else None, ptr, ptr, lr, lr,
                                   np_ptr(out), ag._stream()))


def world1(ag, sync_bn):
    ag.enable_data_parallel(allreduce_mean=lambda t: t, sync_bn=sync_bn, world=1, rank=0,
                            allgather=lambda t: t)          # world of one: identity


@pytest.mark.parametrize("error", ["underfilled", "above_max_batch", "n0", "n65", "flags_bit3", "sync_bn"])
@pytest.mark.parametrize("index_source", ["host", "device"])
@pytest.mark.parametrize("algo", ["sac", "tqc"])
def test_refused_calls_leave_no_trace(algo, error, index_source, monkeypatch):
    """After each refusal the random states, weights, schedules, draw epoch and AdamW step counters (seen through
    the next update) are those of an agent that was never called."""
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    B = 256
    eps = synthetic_episodes(B, 5, D, A, G)
    ref, ag = make_agent(algo, B, index_source, eps), make_agent(algo, B, index_source, eps)
    seed_all()
    if error == "underfilled":
        ag.batch_size = ref.batch_size = len(ag.buffer) + 1
        with pytest.raises(AssertionError):
            ag.update_many([1, 2])
    elif error == "above_max_batch":
        ag.batch_size = B + 1
        with pytest.raises(ValueError):
            ag.update_many([1, 2])
        ag.batch_size = B
    elif error == "sync_bn":
        world1(ag, True)        # a world-of-one sync-BN update equals the plain one bit for bit (test_sac_gpu.py)
        with pytest.raises(ValueError):
            update_many_c(ag, 2, 7)
    else:
        with pytest.raises(ValueError):
            update_many_c(ag, {"n0": 0, "n65": 65}.get(error, 2), 8 if error == "flags_bit3" else 7)
    st = rng_states()
    seed_all()
    assert same_rng_states(st, rng_states())
    if error == "underfilled":
        ag.batch_size = ref.batch_size = B
    assert_same_state(ref, ag)
    one_more_update(ref, ag, 52)                 # an actor and alpha step: every counter is read
    assert_same_state(ref, ag)


@pytest.mark.parametrize("sync_bn", [False, True])
@pytest.mark.parametrize("algo", ["sac", "tqc"])
def test_data_parallel_agents_run_the_loop(algo, sync_bn):
    eps = episodes_for(64)
    a_loop, a_many = make_agent(algo, 64, "host", eps), make_agent(algo, 64, "host", eps)
    for ag in (a_loop, a_many):
        world1(ag, sync_bn)
    loop_vs_many(a_loop, a_many, [39, 40, 41, 42, 40, 51, 52])
    one_more_update(a_loop, a_many, 54)
    assert_same_state(a_loop, a_many)


# ---- 5. eager == graph -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo,B,H,precision", [("sac", 256, 64, 0), ("tqc", 256, 64, 0), ("tqc", 2048, 256, 1)],
                         ids=["sac_p0_B256", "tqc_p0_B256", "tqc_p1_B2048"])
def test_eager_equals_graph(algo, B, H, precision, monkeypatch):
    eps = episodes_for(B)
    monkeypatch.setenv("GCRL_B200_NO_GRAPH", "1")
    eager = make_agent(algo, B, "device", eps, H, precision)
    monkeypatch.delenv("GCRL_B200_NO_GRAPH")
    graph = make_agent(algo, B, "device", eps, H, precision)
    steps = list(range(37, 82))
    seed_all()
    r_e = eager.update_many(steps)
    seed_all()
    r_g = graph.update_many(steps)
    same_results(r_e, r_g)
    assert_same_state(eager, graph)

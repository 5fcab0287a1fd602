"""GPU: ``update_many(steps)`` -- a training cycle's gradient steps as one CUDA graph launch per 64 steps
(csrc/agent.cu: gcrl_agent_update_many) -- against the loop ``[update(s) for s in steps]`` it replaces.

  * bit identity with the loop: every returned tuple, all online and target weights, Adam moments and step
    counts, both schedules, beta, and the interpreter / NumPy / torch CUDA random states; then one more plain
    update() on each agent.  DDPG and TD3 at one batch per row-slab variant (64, 301, 517 on the 2-CTA cluster,
    1021), on the fp32 tiles (1500), on tcgen05 (2048, 4096), and with the sampler as a launch of its own
    (GCRL_B200_NO_FUSED_SAMPLER=1); host and device index streams; step lists that cross Polyak steps, span two
    chunks, or repeat and go backwards;
  * a replayed graph reads this call's buffer totals, positions and scalars, not the captured ones;
  * one cudaGraphLaunch per chunk, no device-to-host copy or stream synchronisation between the updates, and
    the same kernel count as the loop;
  * SAC, TQC, REPLAY, PER and data-parallel agents run the loop;
  * refused calls leave no trace; GCRL_B200_NO_GRAPH=1 equals the graph path.
"""
import ctypes as C
import random

import numpy as np
import pytest

from tests.helpers import bits, her_episodes, load
from tests.test_ddpg_gpu import make_config, synthetic_episodes
from tests.test_fused_variants_gpu import all_weights, first_difference
from tests.test_per_gpu import rand_rows

pytestmark = pytest.mark.gpu

D, A, G = 22, 3, 3
STEP_LISTS = {"range37_82": list(range(37, 82)), "two_chunks": list(range(1, 71)), "unordered": [5, 5, 40, 3]}


# ---- agents -----------------------------------------------------------------------------------------------
def make_agent(algo, B, index_source="host", episodes=None, hidden=64, **over):
    """Seeded weights; the buffer holds seeded episodes, enough that the oldest are partly evicted."""
    import torch
    from gcrl_b200 import DDPG, TD3Agent
    max_len = 2 * B + 100
    cfg = make_config(hidden_dim=hidden, batch_size=B, max_len=max_len, ac_update_freq=1 if algo == "ddpg" else 2,
                      actor_lr=1e-3, actor_lr_min=1e-4, ac_scheduler_steps=30, critic_lr=1e-3, critic_lr_min=1e-4,
                      cr_scheduler_steps=25, beta=0.4, beta_end=100, **over)
    torch.manual_seed(5)
    ag = (DDPG if algo == "ddpg" else TD3Agent)(D, A, cfg, None, 1, 40, index_source=index_source)
    eps = episodes if episodes is not None else synthetic_episodes(B, max_len // 200 + 3, D, A, G)
    for ep in eps:
        ag.buffer.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], ep["fut"])
    assert len(ag.buffer) >= B and ag.buffer.max_mem_len == max_len
    return ag


def seed_all():
    import torch
    random.seed(11)
    np.random.seed(12)
    torch.cuda.manual_seed(13)


def rng_states():
    import torch
    return random.getstate(), np.random.get_state(), torch.cuda.get_rng_state()


def same_rng_states(a, b):
    return a[0] == b[0] and all(np.array_equal(x, y) for x, y in zip(a[1], b[1])) and bool((a[2] == b[2]).all())


def same_value(x, y):
    if isinstance(x, np.ndarray) or isinstance(y, np.ndarray):
        return type(x) is type(y) and x.dtype == y.dtype and np.array_equal(bits(x), bits(y))
    return type(x) is type(y) and (bits(np.float32(x)) == bits(np.float32(y))).all() and x == y


def same_results(r1, r2):
    assert len(r1) == len(r2)
    for i, (t1, t2) in enumerate(zip(r1, r2)):
        assert len(t1) == len(t2) and all(same_value(x, y) for x, y in zip(t1, t2)), (i, t1, t2)


def assert_same_state(a1, a2):
    assert first_difference(all_weights(a1), all_weights(a2)) is None, first_difference(all_weights(a1), all_weights(a2))
    s1, s2 = a1.state_dict(), a2.state_dict()
    for net in s1["adam"]:
        assert s1["adam"][net]["step"] == s2["adam"][net]["step"], net
        for l1, l2 in zip(s1["adam"][net]["layers"], s2["adam"][net]["layers"]):
            assert all(np.array_equal(bits(x.numpy()), bits(y.numpy())) for x, y in zip(l1, l2)), net
    for name in ("actor_scheduler", "critic_scheduler"):
        assert s1[name] == s2[name], name
    assert a1.beta == a2.beta


def loop_vs_many(a_loop, a_many, steps):
    """Runs the loop on one agent and update_many on the other from the same random states; checks the results
    and the random states.  -> the loop's results."""
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


# ---- 1. bit identity against the loop --------------------------------------------------------------------------
CASES = [(64, False), (301, False), (517, False), (1021, False), (1500, False), (2048, False), (4096, False),
         (256, True)]


@pytest.mark.parametrize("index_source", ["host", "device"])
@pytest.mark.parametrize("algo", ["ddpg", "td3"])
@pytest.mark.parametrize("B,separate_sampler", CASES,
                         ids=[f"B{b}" + ("_separate_sampler" if s else "") for b, s in CASES])
def test_update_many_equals_the_loop_bitwise(B, separate_sampler, algo, index_source, monkeypatch):
    """The three step lists in turn on the same pair of agents (the later lists replay graphs of earlier flag
    patterns where they repeat), everything compared after each, then one more plain update()."""
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    monkeypatch.delenv("GCRL_FUSED_R", raising=False)
    if separate_sampler:
        monkeypatch.setenv("GCRL_B200_NO_FUSED_SAMPLER", "1")        # read when the handle is created
    else:
        monkeypatch.delenv("GCRL_B200_NO_FUSED_SAMPLER", raising=False)
    eps = synthetic_episodes(B, (2 * B + 100) // 200 + 3, D, A, G)
    a_loop, a_many = (make_agent(algo, B, index_source, eps) for _ in range(2))
    for name, steps in STEP_LISTS.items():
        loop_vs_many(a_loop, a_many, steps)
        assert_same_state(a_loop, a_many)
    one_more_update(a_loop, a_many)
    assert_same_state(a_loop, a_many)


# ---- 2. the same graph, different contents --------------------------------------------------------------------
@pytest.mark.parametrize("algo,B,separate_sampler", [("ddpg", 256, False), ("td3", 256, True), ("ddpg", 2048, False)],
                         ids=["ddpg_B256", "td3_B256_separate_sampler", "ddpg_B2048"])
@pytest.mark.parametrize("index_source", ["host", "device"])
def test_replayed_graph_reads_the_new_buffer_state(algo, B, separate_sampler, index_source, monkeypatch):
    """Two calls with one flag pattern (the second replays the first's graph); between them new episodes are
    committed to both buffers, which moves the totals and evicts old entries."""
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    if separate_sampler:
        monkeypatch.setenv("GCRL_B200_NO_FUSED_SAMPLER", "1")
    else:
        monkeypatch.delenv("GCRL_B200_NO_FUSED_SAMPLER", raising=False)
    eps = synthetic_episodes(B, (2 * B + 100) // 200 + 3, D, A, G)
    more = synthetic_episodes(B + 1, 3, D, A, G)
    a_loop, a_many = (make_agent(algo, B, index_source, eps) for _ in range(2))
    loop_vs_many(a_loop, a_many, list(range(1, 41)))
    for ag in (a_loop, a_many):
        n0, t0 = len(ag.buffer), ag.buffer.state_dict()["episodes"][0]["s"][0].copy()
        for ep in more:
            ag.buffer.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], ep["fut"])
        assert len(ag.buffer) == n0 and not np.array_equal(ag.buffer.state_dict()["episodes"][0]["s"][0], t0)
    loop_vs_many(a_loop, a_many, list(range(41, 81)))
    assert_same_state(a_loop, a_many)


# ---- 3. one launch per chunk ---------------------------------------------------------------------------------
@pytest.mark.parametrize("algo,B,separate_sampler", [("ddpg", 256, False), ("td3", 256, True), ("ddpg", 4096, False)],
                         ids=["ddpg_B256", "td3_B256_separate_sampler", "ddpg_B4096"])
def test_one_graph_launch_per_chunk(algo, B, separate_sampler, monkeypatch):
    """Under torch.profiler, a warmed-up call of 70 steps issues two cudaGraphLaunch calls, instantiates no graph,
    and neither copies device to host nor synchronises a stream; gcrl_kernel_launches() grows as under the loop."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from gcrl_b200._lib import lib
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    if separate_sampler:
        monkeypatch.setenv("GCRL_B200_NO_FUSED_SAMPLER", "1")
    else:
        monkeypatch.delenv("GCRL_B200_NO_FUSED_SAMPLER", raising=False)
    eps = synthetic_episodes(B, (2 * B + 100) // 200 + 3, D, A, G)
    a_loop, a_many = (make_agent(algo, B, "device", eps) for _ in range(2))
    warm, steps = list(range(1, 71)), list(range(81, 151))     # 80 % 40 == 0: the chunks' flag patterns repeat
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
    assert not any("DtoH" in n or "Device -> Pinned" in n or "Device -> Pageable" in n for n in names)
    syncs = [n for n in names if "StreamSynchronize" in n]
    assert len(syncs) <= 1, syncs                 # the test's own torch.cuda.synchronize() only
    assert k_many == k_loop > 0


# ---- 4. agents that run the loop ---------------------------------------------------------------------------
def sac_agent(cls_name, B):
    import torch
    import gcrl_b200
    from tests.test_sac_gpu import sac_config
    torch.manual_seed(5)
    cfg = sac_config(hidden_dim=64, batch_size=B, max_len=2 * B + 100, ac_update_freq=2)
    ag = getattr(gcrl_b200, cls_name)(D, A, cfg, None, 1, 40)
    for ep in synthetic_episodes(B, (2 * B + 100) // 200 + 3, D, A, G):
        ag.buffer.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], ep["fut"])
    return ag


def replay_agent(buffer_type, B):
    import torch
    from gcrl_b200 import DDPG
    torch.manual_seed(5)
    ag = DDPG(D, A, make_config(hidden_dim=64, batch_size=B, buffer_type=buffer_type, max_len=300, beta=0.4,
                                beta_end=100), None, 1, 40)
    rows = rand_rows(np.random.default_rng(4), 400, D, A)
    for i in range(400):
        ag.push(*(x[i] for x in rows))
    return ag


def dp_agent(B):
    ag = make_agent("ddpg", B, "host", her_episodes(load("her_push_evict")))
    ag.enable_data_parallel(allreduce_mean=lambda t: t)          # one emulated rank: identity
    return ag


@pytest.mark.parametrize("kind", ["sac", "tqc", "replay", "per", "data_parallel"])
def test_other_agents_run_the_loop(kind):
    B = 64
    make = {"sac": lambda: sac_agent("SACAgent", B), "tqc": lambda: sac_agent("TQCAgent", B),
            "replay": lambda: replay_agent("REPLAY", B), "per": lambda: replay_agent("PER", B),
            "data_parallel": lambda: dp_agent(B)}[kind]
    a_loop, a_many = make(), make()
    steps = [39, 40, 41, 42, 40]
    r = loop_vs_many(a_loop, a_many, steps)
    if kind == "per":                  # the per-sample TD arrays of prioritised replay
        assert all(isinstance(t[1 if len(t) == 4 else 2], np.ndarray) for t in r)
    one_more_update(a_loop, a_many, 43)
    if kind in ("replay", "per", "data_parallel"):
        assert first_difference(all_weights(a_loop), all_weights(a_many)) is None


# ---- 5. errors leave no trace; eager == graph ----------------------------------------------------------------
def update_many_c(ag, n):
    """gcrl_agent_update_many with n updates of flags 0 (host positions 0..B-1)."""
    from gcrl_b200._lib import check, lib, np_ptr
    B = ag.batch_size
    m = max(n, 1)
    flags = (C.c_int * m)()
    lr = (C.c_double * m)(*([1e-3] * m))
    idx = np.tile(np.arange(B, dtype=np.int64), (m, 1))
    out = np.empty((m, 8), np.float32)
    check(lib.gcrl_agent_update_many(ag._h, ag.buffer.handle, B, n, flags, np_ptr(idx), None, lr, lr, np_ptr(out),
                                     ag._stream()))


@pytest.mark.parametrize("error", ["underfilled", "above_max_batch", "n0", "n65"])
@pytest.mark.parametrize("index_source", ["host", "device"])
def test_refused_calls_leave_no_trace(error, index_source, monkeypatch):
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    B = 256
    eps = synthetic_episodes(B, 5, D, A, G)
    ref, ag = make_agent("ddpg", B, index_source, eps), make_agent("ddpg", B, index_source, eps)
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
    else:
        with pytest.raises(ValueError):
            update_many_c(ag, 0 if error == "n0" else 65)
    st = rng_states()
    seed_all()
    assert same_rng_states(st, rng_states())
    if error == "underfilled":
        ag.batch_size = ref.batch_size = B
    one_more_update(ref, ag, 40)
    assert_same_state(ref, ag)


@pytest.mark.parametrize("algo", ["ddpg", "td3"])
@pytest.mark.parametrize("B,separate_sampler", [(256, False), (256, True), (2048, False)],
                         ids=["B256", "B256_separate_sampler", "B2048"])
def test_eager_equals_graph(algo, B, separate_sampler, monkeypatch):
    if separate_sampler:
        monkeypatch.setenv("GCRL_B200_NO_FUSED_SAMPLER", "1")
    else:
        monkeypatch.delenv("GCRL_B200_NO_FUSED_SAMPLER", raising=False)
    eps = synthetic_episodes(B, (2 * B + 100) // 200 + 3, D, A, G)
    monkeypatch.setenv("GCRL_B200_NO_GRAPH", "1")
    eager = make_agent(algo, B, "device", eps)
    monkeypatch.delenv("GCRL_B200_NO_GRAPH")
    graph = make_agent(algo, B, "device", eps)
    steps = list(range(37, 82))
    seed_all()
    r_e = eager.update_many(steps)
    seed_all()
    r_g = graph.update_many(steps)
    same_results(r_e, r_g)
    assert_same_state(eager, graph)

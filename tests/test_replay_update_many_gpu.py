"""GPU: ``update_many(steps)`` of agents that sample from a uniform (REPLAY) or prioritised (PER) buffer -- up to 64
updates with their draws and priority write-backs as one CUDA graph launch (csrc/agent.cu:
gcrl_agent_update_many_replay, csrc/sac.cu: gcrl_sac_update_many_replay, csrc/per.cu: the staged draws) -- against
the loop ``[update(s) for s in steps]`` it replaces.

  * bit identity with the loop: every returned tuple (with PER's per-sample TD arrays), all online and target
    weights, optimiser moments and step counts, BatchNorm statistics and log_alpha, both schedules, beta, the ring,
    the priorities, ``last_positions(B)`` and the interpreter / NumPy / torch CUDA random states; then one more
    plain update().  DDPG and TD3 at one batch per row-slab variant (64, 301, 517, 1021), on the fp32 tiles (1500)
    and on tcgen05 (2048); SAC and TQC at 64 and 256 (precision 0) and 2048 (precision 1); step lists that cross
    Polyak steps, span two chunks, or repeat and go backwards;
  * the ring: full and wrapping, pushes between two calls that move its start and evict rows under a replayed
    graph, a filling ring whose length changes between calls, duplicate positions in one draw;
  * the exact fixed-point cumsum and the rounding-tracking one both inside one call;
  * one cudaGraphLaunch per chunk, no device-to-host copy but the final read-back of each chunk, no stream
    synchronisation, and the kernel count of the loop;
  * GCRL_B200_NO_GRAPH=1 equals the graph path; refused calls leave no trace.
"""
import ctypes as C

import numpy as np
import pytest

from tests.helpers import bits
from tests.test_ddpg_gpu import make_config
from tests.test_fused_variants_gpu import all_weights, first_difference
from tests.test_per_gpu import rand_rows
from tests.test_sac_gpu import sac_config
from tests.test_update_many_gpu import rng_states, same_results, same_rng_states, seed_all

pytestmark = pytest.mark.gpu

D, A = 22, 3
STEP_LISTS = {"range37_82": list(range(37, 82)), "two_chunks": list(range(1, 71)), "unordered": [5, 5, 40, 3]}
SAC_ALGOS = ("sac", "tqc")


# ---- agents -----------------------------------------------------------------------------------------------
def make_agent(algo, kind, B, *, max_len=None, rows=None, hidden=64, precision=None, alpha=0.6, seed=4):
    """Seeded weights; the buffer (REPLAY or PER) holds seeded rows -- by default more than it keeps, so the ring is
    full and has wrapped."""
    import torch
    import gcrl_b200
    max_len = 2 * B + 100 if max_len is None else max_len
    rows = max_len + B // 2 + 37 if rows is None else rows
    common = dict(hidden_dim=hidden, batch_size=B, buffer_type=kind, max_len=max_len, alpha=alpha, ac_update_freq=2,
                  actor_lr=1e-3, actor_lr_min=1e-4, ac_scheduler_steps=30, critic_lr=1e-3, critic_lr_min=1e-4,
                  cr_scheduler_steps=25, beta=0.4, beta_end=100)
    torch.manual_seed(5)
    if algo in SAC_ALGOS:
        cfg = sac_config(alpha_min_steps=50, alpha_lr=1e-2, **common)
        cls = gcrl_b200.SACAgent if algo == "sac" else gcrl_b200.TQCAgent
        ag = cls(D, A, cfg, None, 1, 40, precision=0 if precision is None else precision)
    else:
        if algo == "ddpg":
            common["ac_update_freq"] = 1
        cfg = make_config(**common)
        cls = gcrl_b200.DDPG if algo == "ddpg" else gcrl_b200.TD3Agent
        ag = cls(D, A, cfg, None, 1, 40, **({} if precision is None else {"precision": precision}))
    push(ag, rows, seed)
    assert len(ag.buffer) == min(rows, max_len)
    return ag


def push(ag, n, seed):
    ag.buffer.push_rows(*rand_rows(np.random.default_rng(seed), n, D, A))


def is_per(ag):
    from gcrl_b200 import PERBuffer
    return isinstance(ag.buffer, PERBuffer)


def buffer_state(ag):
    out = [ag.buffer.rows()]
    if is_per(ag):
        out += [ag.buffer.priorities, ag.buffer.last_positions(ag.batch_size)]
    return out


def agent_state(ag):
    """Everything update() moves, as a list of arrays / scalars."""
    out = []
    if ag.ALGO >= 2:                                   # SAC / TQC
        L = ag.config.layer_count
        for l in range(L + 2):
            out += list(ag.actor.linear(l))
        for l in range(L):
            out += list(ag.actor.bn(l))               # weight, bias, running mean, running var
        for view in ag._critic_views + ag._target_views:
            for w, b in view.layers():
                out += [w, b]
        out += [np.float32(ag.get_log_alpha()), ag._bn_batches]
    else:
        sd = ag.state_dict()
        out += [x.numpy() for net in sorted(sd["nets"]) for layer in sd["nets"][net] for x in layer]
        for net in sorted(sd["adam"]):
            out.append(sd["adam"][net]["step"])
            out += [x.numpy() for layer in sd["adam"][net]["layers"] for x in layer]
    for sch in (ag.critic_scheduler, ag.actor_scheduler):
        out += [sch.last_epoch, sch.lr]
    out.append(ag.beta)
    return out + buffer_state(ag)


def assert_same_state(a1, a2):
    if a1.ALGO < 2:
        assert first_difference(all_weights(a1), all_weights(a2)) is None, first_difference(all_weights(a1), all_weights(a2))
    s1, s2 = agent_state(a1), agent_state(a2)
    assert len(s1) == len(s2)
    for i, (x, y) in enumerate(zip(s1, s2)):
        if isinstance(x, np.ndarray):
            assert x.dtype == y.dtype and np.array_equal(bits(x), bits(y)), i
        else:
            assert x == y, (i, x, y)


def loop_vs_many(a_loop, a_many, steps):
    """The loop on one agent, update_many on the other, from the same random states -> the loop's results."""
    seed_all()
    r_loop = [a_loop.update(s) for s in steps]
    st_loop = rng_states()
    seed_all()
    r_many = a_many.update_many(steps)
    st_many = rng_states()
    same_results(r_loop, r_many)
    assert same_rng_states(st_loop, st_many)
    if is_per(a_loop):                 # the per-sample TD arrays of prioritised replay
        shape = (a_loop.batch_size, 1)
        assert all(sum(isinstance(x, np.ndarray) and x.shape == shape for x in t) == 1 for t in r_many)
    return r_loop


def one_more_update(a1, a2, step=83):
    seed_all()
    u1 = a1.update(step)
    seed_all()
    u2 = a2.update(step)
    same_results([u1], [u2])


# ---- 1. bit identity against the loop --------------------------------------------------------------------------
def run_lists(a_loop, a_many):
    for steps in STEP_LISTS.values():
        loop_vs_many(a_loop, a_many, steps)
        assert_same_state(a_loop, a_many)
    one_more_update(a_loop, a_many)
    assert_same_state(a_loop, a_many)


@pytest.mark.parametrize("kind", ["REPLAY", "PER"])
@pytest.mark.parametrize("algo", ["ddpg", "td3"])
@pytest.mark.parametrize("B", [64, 301, 517, 1021, 1500, 2048])
def test_ddpg_td3_equal_the_loop_bitwise(B, algo, kind, monkeypatch):
    """Row-slab variants (64 .. 1021), fp32 tiles (1500), tcgen05 (2048); the three step lists in turn on one pair."""
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    a_loop, a_many = (make_agent(algo, kind, B) for _ in range(2))
    run_lists(a_loop, a_many)


SAC_CASES = [(64, 64, 0), (256, 64, 0), (2048, 256, 1)]


@pytest.mark.parametrize("kind", ["REPLAY", "PER"])
@pytest.mark.parametrize("algo", SAC_ALGOS)
@pytest.mark.parametrize("B,H,precision", SAC_CASES, ids=[f"p{p}_B{b}_H{h}" for b, h, p in SAC_CASES])
def test_sac_tqc_equal_the_loop_bitwise(B, H, precision, algo, kind, monkeypatch):
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    a_loop, a_many = (make_agent(algo, kind, B, hidden=H, precision=precision) for _ in range(2))
    run_lists(a_loop, a_many)


# ---- 2. the ring -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["REPLAY", "PER"])
@pytest.mark.parametrize("algo", ["ddpg", "td3", "tqc"])
def test_replayed_graph_follows_pushes(algo, kind, monkeypatch):
    """Three calls with one flag pattern on a full, wrapping ring (the later ones replay a graph: PER captures when
    the key repeats); between calls new rows move the ring's start and evict the oldest."""
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    B = 256
    a_loop, a_many = (make_agent(algo, kind, B) for _ in range(2))
    for c in range(3):
        if c:
            for ag in (a_loop, a_many):
                first = ag.buffer.rows(0, 1)
                push(ag, 150 + c, seed=20 + c)
                assert len(ag.buffer) == ag.buffer.max_len and not np.array_equal(ag.buffer.rows(0, 1), first)
        loop_vs_many(a_loop, a_many, list(range(80 * c + 81, 80 * c + 121)))
        assert_same_state(a_loop, a_many)


@pytest.mark.parametrize("kind", ["REPLAY", "PER"])
@pytest.mark.parametrize("algo", ["ddpg", "sac"])
def test_filling_ring_changes_length_between_calls(algo, kind, monkeypatch):
    """The ring is not full: every call draws from a new length (PER issues such calls without a graph)."""
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    B = 128
    a_loop, a_many = (make_agent(algo, kind, B, max_len=5000, rows=600) for _ in range(2))
    for c in range(3):
        if c:
            for ag in (a_loop, a_many):
                push(ag, 97 * c, seed=30 + c)
        assert len(a_many.buffer) == 600 + 97 * (c * (c + 1) // 2)
        loop_vs_many(a_loop, a_many, list(range(40 * c + 1, 40 * c + 21)))
        assert_same_state(a_loop, a_many)


@pytest.mark.parametrize("algo", ["ddpg", "tqc"])
def test_duplicate_positions_last_occurrence_wins(algo, monkeypatch):
    """A few rows hold almost all the priority mass, so every draw repeats positions; the write-back of each update
    keeps the LAST occurrence's TD error (update_priorities applies the list in order)."""
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    B = 64
    a_loop, a_many = (make_agent(algo, "PER", B, max_len=300, alpha=1.0) for _ in range(2))
    prio = np.full(300, 1e-3, np.float32)
    prio[[3, 77, 150, 299]] = 50.0
    for ag in (a_loop, a_many):
        ag.buffer.set_priorities(prio)
    steps = list(range(1, 11))
    loop_vs_many(a_loop, a_many, steps)
    assert_same_state(a_loop, a_many)
    pos = a_many.buffer.last_positions(B)
    assert len(np.unique(pos)) < B // 2
    td = a_many._last_td.reshape(-1)
    last = {p: j for j, p in enumerate(pos)}
    expect = np.abs(td[list(last.values())]) + np.float32(1e-6)
    assert np.array_equal(bits(a_many.buffer.priorities[list(last.keys())]), bits(expect.astype(np.float32)))


@pytest.mark.parametrize("algo", ["ddpg", "sac"])
def test_both_cumsum_branches_inside_one_call(algo, monkeypatch):
    """Fresh priorities (all 1.0) make the first draw's cumsum exact in fixed point; alpha = 16 spreads the written
    priorities over so many binades that later draws take the rounding-tracking branch."""
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    B = 64
    a_loop, a_many = (make_agent(algo, "PER", B, max_len=300, alpha=16.0) for _ in range(2))
    steps = list(range(1, 13))
    seed_all()
    branches, r_loop = [], []
    for s in steps:
        r_loop.append(a_loop.update(s))
        branches.append(a_loop.buffer.last_sample_info()[1])
    st_loop = rng_states()
    seed_all()
    r_many = a_many.update_many(steps)
    same_results(r_loop, r_many)
    assert same_rng_states(st_loop, rng_states())
    assert not branches[0] and any(branches), branches
    info_loop, info_many = a_loop.buffer.last_sample_info(), a_many.buffer.last_sample_info()
    assert bits(info_loop[0]) == bits(info_many[0]) and info_loop[1] == info_many[1]
    assert_same_state(a_loop, a_many)


# ---- 3. one launch per chunk ---------------------------------------------------------------------------------
@pytest.mark.parametrize("algo,kind", [("ddpg", "REPLAY"), ("ddpg", "PER"), ("td3", "PER"), ("tqc", "PER")])
def test_one_graph_launch_per_chunk(algo, kind, monkeypatch):
    """Under torch.profiler, a warmed-up call of 70 steps issues two cudaGraphLaunch calls, instantiates no graph,
    synchronises no stream and copies device to host only the final read-back of each chunk (the TD rows of PER, with
    the metric rows for SAC / TQC); gcrl_kernel_launches() grows as under the loop."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from gcrl_b200._lib import lib
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    B = 256
    a_loop, a_many = (make_agent(algo, kind, B) for _ in range(2))
    # 40 apart (alpha steps: past alpha_min_steps): the chunks' flag patterns repeat; PER captures on the second
    for warm in (list(range(81, 151)), list(range(121, 191))):
        loop_vs_many(a_loop, a_many, warm)
    steps = list(range(161, 231))
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
    assert len(d2h) == (2 if kind == "PER" or algo in SAC_ALGOS else 0), d2h
    syncs = [n for n in names if "StreamSynchronize" in n]
    assert len(syncs) <= 1, syncs                 # the test's own torch.cuda.synchronize() only
    assert k_many == k_loop > 0
    assert_same_state(a_loop, a_many)


# ---- 4. eager == graph; refused calls leave no trace ---------------------------------------------------------
@pytest.mark.parametrize("algo,kind", [("ddpg", "REPLAY"), ("td3", "PER"), ("tqc", "PER")])
def test_eager_equals_graph(algo, kind, monkeypatch):
    monkeypatch.setenv("GCRL_B200_NO_GRAPH", "1")            # read when the agent and the buffer are created
    eager = make_agent(algo, kind, 256)
    monkeypatch.delenv("GCRL_B200_NO_GRAPH")
    graph = make_agent(algo, kind, 256)
    for steps in (list(range(37, 82)), list(range(77, 122)), list(range(117, 162))):
        seed_all()
        r_e = eager.update_many(steps)
        seed_all()
        r_g = graph.update_many(steps)
        same_results(r_e, r_g)
        assert_same_state(eager, graph)


def update_many_c(ag, n, flags, buf=None):
    """The n-update C call of the agent's family with positions 0..B-1 (REPLAY) or uniforms 0.5 and beta 0.4 (PER)."""
    import torch
    from gcrl_b200._lib import check, lib, np_ptr
    B, m = ag.batch_size, max(n, 1)
    buf = ag.buffer if buf is None else buf
    cflags = (C.c_int * m)(*([flags] * m))
    lr = (C.c_double * m)(*([1e-3] * m))
    pos = np.tile(np.arange(B, dtype=np.int64), (m, 1))
    u, beta = np.full((m, B), 0.5), np.full(m, 0.4)
    noise = torch.zeros((m, B, A), dtype=torch.float32, device="cuda")
    td = np.empty((m, B), np.float32)
    nptr = C.c_void_p(noise.data_ptr())
    args = (np_ptr(pos), np_ptr(u), np_ptr(beta))
    if ag.ALGO >= 2:
        check(lib.gcrl_sac_update_many_replay(ag._h, buf.handle, B, n, cflags, *args, nptr, nptr, lr, lr,
                                              np_ptr(np.empty((m, 12), np.float32)), np_ptr(td), ag._stream()))
    else:
        check(lib.gcrl_agent_update_many_replay(ag._h, buf.handle, B, n, cflags, *args, nptr, lr, lr,
                                                np_ptr(np.empty((m, 8), np.float32)), np_ptr(td), ag._stream()))


ERRORS = ["underfilled", "above_max_batch", "n0", "n65", "bit3_mismatch", "shape_mismatch"]


@pytest.mark.parametrize("error", ERRORS)
@pytest.mark.parametrize("algo,kind", [("ddpg", "REPLAY"), ("td3", "PER"), ("tqc", "PER")])
def test_refused_calls_leave_no_trace(algo, kind, error, monkeypatch):
    """The call raises; the ring, priorities, optimiser state, schedules and random states are those of an agent
    that never made it, and the next update() agrees with that agent's."""
    from gcrl_b200 import PERBuffer, ReplayBuffer
    monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    B = 256
    ref, ag = make_agent(algo, kind, B), make_agent(algo, kind, B)
    for a in (ref, ag):                  # a first call: the slots and the graph cache exist
        seed_all()
        a.update_many(list(range(1, 5)))
    per = 8 if kind == "PER" else 0
    seed_all()
    before = rng_states()
    if error == "underfilled":
        ag.batch_size = len(ag.buffer) + 1
        with pytest.raises(AssertionError):
            ag.update_many([5, 6])
        ag.batch_size = B
    elif error == "above_max_batch":
        ag.batch_size = B + 1
        with pytest.raises(ValueError):
            ag.update_many([5, 6])
        ag.batch_size = B
    elif error in ("n0", "n65"):
        with pytest.raises(ValueError):
            update_many_c(ag, 0 if error == "n0" else 65, per)
    elif error == "bit3_mismatch":
        with pytest.raises(ValueError):
            update_many_c(ag, 3, per ^ 8)
    else:
        other = (PERBuffer(1000, 0.6) if per else ReplayBuffer(1000))
        other.push_rows(*rand_rows(np.random.default_rng(9), 600, D + 1, A))
        rows0 = other.rows()
        with pytest.raises(ValueError):
            update_many_c(ag, 3, per, other)
        assert np.array_equal(other.rows(), rows0)
    assert same_rng_states(before, rng_states())
    assert_same_state(ref, ag)
    one_more_update(ref, ag, 7)
    assert_same_state(ref, ag)

"""GPU: the row-slab update kernels (csrc/fused.cu) at every rows-per-CTA variant.

The launcher picks R rows per CTA from the batch size and the SM count (fused.cu::fused_rows_per_cta,
launch_fused_critic): on 148 SMs R = 2 up to B = 296, 4 up to 512, 8 up to 1024, and the critic phase runs as
2-CTA clusters (target path | critic path, q' handed over through distributed shared memory) when both CTAs of
every slab fit in one wave -- by default only at R = 8 for B in 513..592.  GCRL_FUSED_R forces R.

  * which kernel ran: every case names the template instantiations it expects (computed with the launcher's
    rule from this GPU's SM count) and fails unless exactly those ran, under torch.profiler;
  * eager launches == graph replay, bit for bit;
  * variant equivalence: slab_matmul's K split depends only on the layer width and slab_head reduces one
    (output, row) pair per warp, so a row's arithmetic does not depend on R, and the weight-gradient kernel
    depends only on B.  Every supported R must therefore leave bit-identical weights in all networks; only the
    loss / td / q metrics, summed per slab first, may differ in the last bits;
  * the arithmetic's branches against the NumPy oracle at one batch per R: DDPG's y clamp at both ends, TD3's
    smooth-L1 linear branch, smoothing-noise clamp and action clamp, and prioritised weights (flags bit 3);
  * GCRL_FUSED_R values other than 2, 4 and 8 are ignored.
"""
import ctypes as C
import re

import numpy as np
import pytest

from oracle import ddpg as OD
from oracle import td3 as OT
from tests.helpers import bits, weights_close
from tests.test_ddpg_gpu import make_config

pytestmark = pytest.mark.gpu

PUSH = dict(D=21, A=3, H=256, L=3)              # the headline network shape
STEPS = (39, 40, 41)                            # DDPG: Polyak at 40; TD3 (actor every 2nd step): actor at 40
SLAB_KERNEL = re.compile(r"(fused_critic_kernel|fused_actor_kernel|wgrad_tile_kernel)<([^>]*)>")


# ---- the launcher's rule, restated ------------------------------------------------------------------
def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def rows_per_cta(B, forced=None):
    """fused.cu::fused_rows_per_cta."""
    if forced in (2, 4, 8):
        return forced
    if B <= 2 * sm_count():
        return 2
    return 4 if B <= 512 else 8


def fused_smem_bytes(R, D, A, H, L, two_keeps):
    kinp = (D + A + 3) & ~3
    return 4 * (2 * kinp * R + 2 * H * R + L * H * R * (2 if two_keeps else 1) + 2048 * R + 24 * R)


def expected_kernels(algo, B, forced, D, A, H, L, actor_step):
    """The row-slab instantiations one or more updates must launch, or None where the row-slab path does not
    take the batch (fused_supported) and the update runs on the fp32 GEMM tiles."""
    R = rows_per_cta(B, forced)
    grid = -(-B // R)
    if grid > 256 or fused_smem_bytes(R, D, A, H, L, True) > 200 * 1024:
        return None
    split = R != 2 and 2 * grid <= sm_count()
    td3 = algo == "td3"
    out = {f"fused_critic_kernel<{R},{str(td3).lower()},{str(split).lower()}>",
           f"wgrad_tile_kernel<{8 if B > 256 else 4}>"}
    if td3:
        out.add(f"fused_critic_kernel<{R},true,false>")          # critic 2 reuses y: no target path to split
    if actor_step:
        out.add(f"fused_actor_kernel<{R}>")
    return out


# ---- what ran ---------------------------------------------------------------------------------------
def launched_kernels(fn):
    """Run fn() under torch.profiler (CUDA activities) -> the names of every kernel it launched.  The agent
    must have been created with GCRL_B200_NO_GRAPH=1 so that each kernel is a launch of its own."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events()}


def check_kernels(names, expect, label, capsys):
    got = {m.group(1) + "<" + re.sub(r"\s+", "", m.group(2)) + ">" for n in names for m in SLAB_KERNEL.finditer(n)}
    tiles = sorted({n for n in names if "gemm_kernel" in n})
    with capsys.disabled():
        print(f"\n[coverage] {label}: " + (", ".join(sorted(got)) if got else "no row-slab kernel") +
              (f"; fp32 tiles: {len(tiles)} kernel names" if tiles else ""))
    if expect is None:
        assert not any(k.startswith("fused_") for k in got) and tiles, (label, sorted(got))
    else:
        assert got == expect, (label, sorted(got), sorted(expect))
        assert not tiles, (label, tiles)


# ---- agents, batches, weights ---------------------------------------------------------------------------
def init_nets(rng, algo, D, A, H, L):
    return [OD.init_mlp(rng, D, H, A, L)] + [OD.init_mlp(rng, D + A, H, 1, L) for _ in range(1 if algo == "ddpg" else 2)]


def make_agent(algo, B, nets, monkeypatch, D, A, H, L, graphs=False, precision=1, **over):
    from gcrl_b200 import DDPG, TD3Agent
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC, NET_CRITIC2
    if graphs:
        monkeypatch.delenv("GCRL_B200_NO_GRAPH", raising=False)
    else:
        monkeypatch.setenv("GCRL_B200_NO_GRAPH", "1")             # read at creation
    cfg = make_config(hidden_dim=H, layer_count=L, batch_size=B, grad_clip=0.5, tau=0.05,
                      ac_update_freq=1 if algo == "ddpg" else 2, **over)
    ag = (DDPG if algo == "ddpg" else TD3Agent)(D, A, cfg, None, 1, 40, precision=precision)
    for net, params in zip((NET_ACTOR, NET_CRITIC, NET_CRITIC2), nets):
        ag._set_layers(net, params)
    ag.update_target_network()
    return ag


def set_rows_per_cta(monkeypatch, R):
    if R is None:
        monkeypatch.delenv("GCRL_FUSED_R", raising=False)
    else:
        monkeypatch.setenv("GCRL_FUSED_R", str(R))


def make_batch(rng, B, D, A):
    s = rng.standard_normal((B, D)).astype(np.float32)
    ns = (s + 0.1 * rng.standard_normal((B, D))).astype(np.float32)
    a = rng.uniform(-1, 1, (B, A)).astype(np.float32)
    r = -(rng.random((B, 1)) > 0.3).astype(np.float32)
    d = (rng.random((B, 1)) < 0.1).astype(np.float32)
    return s, a, r, ns, d


def run_updates(ag, algo, batches, noises, steps=STEPS):
    import torch
    out = []
    for step, b, nz in zip(steps, batches, noises):
        kw = {"noise": torch.from_numpy(nz).cuda()} if algo == "td3" else {}
        out.append([float(x) for x in ag.update(step, batch=tuple(torch.from_numpy(x).cuda() for x in b), **kw)])
    return out


def all_weights(ag):
    """{(net, layer, "W" | "b"): float32 array} over every network, targets included."""
    return {(net, li, k): x for net in ag._all_nets() for li, wb in enumerate(ag._get_layers(net))
            for k, x in zip("Wb", wb)}


def first_difference(w0, w1):
    """-> None, or (net, layer, W | b, first differing row) of the first tensor whose bits differ."""
    for key in w0:
        diff = bits(w0[key]) != bits(w1[key])
        if diff.any():
            return key + (int(np.argwhere(diff)[0][0]),)
    return None


# ---- a. which kernel ran; eager == graph replay -----------------------------------------------------------
@pytest.mark.parametrize("algo", ["ddpg", "td3"])
@pytest.mark.parametrize("B", [256, 301, 517, 1000])
def test_eager_update_equals_graph_replay(B, algo, monkeypatch, capsys):
    """The captured graph (production path) and plain launches of the same update: bit-identical metrics and
    weights over three updates (the second replays the first one's graph where the flags repeat)."""
    monkeypatch.delenv("GCRL_FUSED_R", raising=False)
    rng = np.random.default_rng(B + 5)
    nets = init_nets(rng, algo, **PUSH)
    batches = [make_batch(rng, B, PUSH["D"], PUSH["A"]) for _ in STEPS]
    noises = [rng.standard_normal((B, PUSH["A"])).astype(np.float32) for _ in STEPS]
    eager = make_agent(algo, B, nets, monkeypatch, **PUSH)
    info_e = []
    names = launched_kernels(lambda: info_e.extend(run_updates(eager, algo, batches, noises)))
    check_kernels(names, expected_kernels(algo, B, None, **PUSH, actor_step=True), f"{algo} B={B} default R", capsys)
    graph = make_agent(algo, B, nets, monkeypatch, graphs=True, **PUSH)
    info_g = run_updates(graph, algo, batches, noises)
    assert info_e == info_g
    assert first_difference(all_weights(eager), all_weights(graph)) is None


# ---- b. every supported R leaves the same weights -----------------------------------------------------------
@pytest.mark.parametrize("algo", ["ddpg", "td3"])
@pytest.mark.parametrize("B,variants", [(256, (None, 4, 8)), (301, (None, 8)), (517, (None, 4, 2)), (1000, (None, 4))],
                         ids=["B256", "B301", "B517", "B1000"])
def test_rows_per_cta_variants_leave_identical_weights(B, variants, algo, monkeypatch, capsys):
    """For a fixed batch and weights, every supported R (None: the launcher's own choice) leaves bit-identical
    weights in all 4 (DDPG) / 6 (TD3) networks after steps 39-41; loss / td / q, summed per slab first, agree
    to rel 1e-6.  A variant the row-slab path does not take (B = 517 at R = 2: 259 slabs > 256) must fall back
    to the fp32 tiles; it is compared at the engines' fp32 tolerance only."""
    rng = np.random.default_rng(B)
    nets = init_nets(rng, algo, **PUSH)
    batches = [make_batch(rng, B, PUSH["D"], PUSH["A"]) for _ in STEPS]
    noises = [rng.standard_normal((B, PUSH["A"])).astype(np.float32) for _ in STEPS]
    ref = None
    for R in variants:
        set_rows_per_cta(monkeypatch, R)
        ag = make_agent(algo, B, nets, monkeypatch, **PUSH)
        info = []
        names = launched_kernels(lambda: info.extend(run_updates(ag, algo, batches, noises)))
        expect = expected_kernels(algo, B, R, **PUSH, actor_step=True)
        check_kernels(names, expect, f"{algo} B={B} GCRL_FUSED_R={R}", capsys)
        got = (np.concatenate([np.array(x) for x in info]), all_weights(ag))     # TD3: 6 or 8 metrics per step
        if ref is None:
            assert expect is not None
            ref = got
        elif expect is not None:
            np.testing.assert_allclose(got[0], ref[0], rtol=1e-6, atol=1e-7, err_msg=f"R={R} metrics")
            assert first_difference(ref[1], got[1]) is None, (f"R={R}: (net, layer, tensor, row)",
                                                               first_difference(ref[1], got[1]))
        else:
            np.testing.assert_allclose(got[0], ref[0], rtol=1e-4, atol=2e-6, err_msg=f"R={R} (fp32 tiles) metrics")


# ---- c / d. branch edges and prioritised weights against the oracle -------------------------------------------
EDGE = dict(D=21, A=3, H=128, L=2)
EDGE_STEPS = (39, 40, 41, 42)


def edge_batch(rng, algo, B, D, A):
    """DDPG: rewards -60 / +2 push y below -1 / (1 - gamma) and above 0 (both ends of the clamp), d = 1 on a
    quarter of the rows.  TD3: rewards -4 / +3 put |q - y| >= 1 (smooth-L1's linear branch) on part of the batch;
    the noise is scaled by 4 on half of the rows so that some hit noise_clamp and some push a' out of [-1, 1]."""
    s, a, _, ns, _ = make_batch(rng, B, D, A)
    far = (-60.0, 2.0) if algo == "ddpg" else (-4.0, 3.0)
    r = rng.choice([-1.0, 0.0, *far], size=(B, 1), p=[0.6, 0.2, 0.1, 0.1]).astype(np.float32)
    d = (rng.random((B, 1)) < 0.25).astype(np.float32)
    noise = (rng.standard_normal((B, A)) * np.where(rng.random((B, 1)) < 0.5, 4.0, 1.0)).astype(np.float32)
    return (s, a, r, ns, d), noise


def priority_weights(rng, B):
    w = (1.0 - rng.random(B)).astype(np.float32)        # (0, 1]
    w[rng.choice(B, 5, replace=False)] = 0.0
    w[rng.integers(B)] = 1.0
    return w


def branches_hit(orc, algo, batch, randn, gamma, policy_noise, noise_clamp):
    """The branches the oracle takes on this batch: {name: (some rows take it, some do not)}."""
    s, a, r, ns, d = batch
    if algo == "ddpg":
        na, _ = OD.mlp_forward(orc.target_actor, ns, True)
        q_next, _ = OD.mlp_forward(orc.target_critic, np.concatenate([ns, na], -1), False)
        y = r + gamma * (1 - d) * q_next
        return {"y below -1/(1-gamma)": y < -1.0 / (1.0 - gamma), "y above 0": y > 0}
    raw = randn * np.float32(policy_noise)
    na, _ = OD.mlp_forward(orc.target_actor, ns, True)
    na = na + np.clip(raw, -noise_clamp, noise_clamp)
    tin = np.concatenate([ns, np.clip(na, -1, 1)], -1)
    q_next = np.minimum(OD.mlp_forward(orc.target_critic_1, tin, False)[0], OD.mlp_forward(orc.target_critic_2, tin, False)[0])
    y = r + gamma * (1 - d) * q_next
    q1, _ = OD.mlp_forward(orc.critic_1, np.concatenate([s, a], -1), False)
    return {"noise clamp": np.abs(raw) > noise_clamp, "action clamp": np.abs(na) > 1, "smooth-L1 linear": np.abs(q1 - y) >= 1}


def update_direct(ag, step, batch, noise, w):
    """One update through gcrl_agent_update_batch, as _run_update issues it; with ``w`` the importance weights are
    written into the agent's weight array first and flags bit 3 is set.  -> (metric vector, per-sample TD or None)."""
    import torch
    from gcrl_b200._lib import check, lib, vp
    from gcrl_b200.parallel import device_tensor
    B = batch[0].shape[0]
    dev = [torch.from_numpy(x).cuda() for x in batch]
    nz = torch.from_numpy(noise).cuda() if noise is not None else None
    flags = ag._flags(step)
    if w is not None:
        wptr, td_ptr = ag._per_ptrs()
        device_tensor(wptr.value, B, ag.device_index).copy_(torch.from_numpy(w))
        flags |= 8
    torch.cuda.synchronize()
    check(lib.gcrl_agent_update_batch(ag._h, B, *(vp(t.data_ptr()) for t in dev), vp(nz.data_ptr()) if nz is not None else None,
                                      ag.critic_scheduler.lr, ag.actor_scheduler.lr, flags, C.cast(ag._metrics, vp),
                                      ag._stream()))
    torch.cuda.synchronize()
    td = device_tensor(td_ptr.value, B, ag.device_index).cpu().numpy().copy() if w is not None else None
    return [float(x) for x in ag._metrics], td


def as_oracle_tuple(algo, m, actor_step):
    """The agent's metric vector in the order of DDPGOracle / TD3Oracle.update_on_batch."""
    if algo == "ddpg":
        return m[:6] if actor_step else [m[0], m[2], m[3], m[4]]
    q1l, acl, td, q, c1g, acg, q2l, c2g = m
    return [q1l, q2l, acl, td, q, c1g, c2g, acg] if actor_step else [q1l, q2l, td, q, c1g, c2g]


@pytest.mark.parametrize("weighted", [False, True], ids=["uniform", "prioritised"])
@pytest.mark.parametrize("algo", ["ddpg", "td3"])
@pytest.mark.parametrize("B", [301, 517, 1021])
def test_branch_edges_match_oracle(B, algo, weighted, monkeypatch, capsys):
    """Four updates at one batch per R (148 SMs: 4; 8 as 2-CTA clusters; 8) on batches that drive every branch
    of the loss and the target (edge_batch), uniform or with prioritised weights (flags bit 3: weighted loss, the
    per-sample TD written back -- for TD3 the larger of both critics'), versus the NumPy oracle: metrics at
    5e-5 * sqrt(B / 256) (plus the oracle's LeakyReLU flip slack on DDPG's gradient norms), per-sample TD at
    rel 5e-5, all networks' weights at weights_close."""
    monkeypatch.delenv("GCRL_FUSED_R", raising=False)
    D, A, H, L = EDGE["D"], EDGE["A"], EDGE["H"], EDGE["L"]
    rng = np.random.default_rng(3 * B + 2 * (algo == "td3") + weighted)
    nets = init_nets(rng, algo, D, A, H, L)
    pn, nc, gamma, lr = 0.5, 1.5, 0.98, 1e-3
    ag = make_agent(algo, B, nets, monkeypatch, D, A, H, L, policy_noise=pn, noise_clamp=nc, gamma=gamma)
    kw = dict(gamma=gamma, tau=0.05, grad_clip=0.5, actor_lr=lr, critic_lr=lr, ac_update_freq=ag.ac_update_freq)
    if algo == "ddpg":
        orc = OD.DDPGOracle(*nets, **kw)
        orc.flip_delta = 5e-6
    else:
        orc = OT.TD3Oracle(*nets, policy_noise=pn, noise_clamp=nc, **kw)
    hit = {}
    critic_flips = False
    base = 5e-5 * max(1.0, (B / 256.0) ** 0.5)
    for si, step in enumerate(EDGE_STEPS):
        batch, randn = edge_batch(rng, algo, B, D, A)
        w = priority_weights(rng, B) if weighted else None
        for name, rows in branches_hit(orc, algo, batch, randn, gamma, pn, nc).items():
            hit[name] = hit.get(name, False) or bool(rows.any() and not rows.all())
        noise = randn if algo == "td3" else None
        if si == 0:
            out = []
            names = launched_kernels(lambda: out.append(update_direct(ag, step, batch, noise, w)))
            check_kernels(names, expected_kernels(algo, B, None, D, A, H, L, actor_step=bool(ag._flags(step) & 1)),
                          f"{algo} B={B} {'prioritised' if weighted else 'uniform'} vs oracle", capsys)
            m, td = out[0]
        else:
            m, td = update_direct(ag, step, batch, noise, w)
        wcol = None if w is None else w.reshape(B, 1)
        want = (orc.update_on_batch(step, *batch, weights=wcol) if algo == "ddpg"
                else orc.update_on_batch(step, *batch, randn, weights=wcol))
        actor_step = step % ag.ac_update_freq == 0
        got = as_oracle_tuple(algo, m, actor_step)
        assert len(got) == len(want)
        td_pos = (2 if actor_step else 1) if algo == "ddpg" else (3 if actor_step else 2)
        rtol = np.full(len(want), base)
        if algo == "ddpg":
            rtol[-2 if actor_step else -1] += orc.last_critic_flip_slack
            if actor_step:
                rtol[-1] += orc.last_actor_flip_slack
            critic_flips = critic_flips or orc.last_critic_flip_slack > 0
        keep = [i for i in range(len(want)) if not (weighted and i == td_pos)]
        g_, w_ = np.array(got)[keep], np.array([float(want[i]) for i in keep])
        assert np.all(np.abs(g_ - w_) <= rtol[keep] * np.abs(w_) + 2e-6), (step, g_, w_, rtol[keep])
        if weighted:
            np.testing.assert_allclose(td, np.asarray(want[td_pos]).ravel(), rtol=5e-5, atol=5e-6, err_msg=f"step {step} td")
    assert all(hit.values()), hit
    n = len(EDGE_STEPS)
    if algo == "ddpg":
        pairs = (("actor", ag.actor, orc.actor), ("critic", ag.critic, orc.critic),
                 ("target_actor", ag.target_actor, orc.target_actor), ("target_critic", ag.target_critic, orc.target_critic))
    else:
        pairs = (("actor", ag.actor, orc.actor), ("critic_1", ag.critic_1, orc.critic_1),
                 ("critic_2", ag.critic_2, orc.critic_2), ("target_actor", ag.target_actor, orc.target_actor),
                 ("target_critic_1", ag.target_critic_1, orc.target_critic_1),
                 ("target_critic_2", ag.target_critic_2, orc.target_critic_2))
    for name, net, ref in pairs:
        for li, ((w, b), (rw, rb)) in enumerate(zip(net.layers(), ref)):
            if algo == "ddpg":       # per-element LeakyReLU flip allowance, as in test_update_matches_oracle_odd_shapes
                allow = orc.flip_allowance if "actor" in name else orc.flip_allowance_critic
                scale = 0.05 * n if name.startswith("target") else 1.0
                frac = 5e-3 if ("actor" in name and critic_flips) else 2e-4
                ok = (weights_close(w, rw, lr, n, extra=allow[li][0] * scale, outlier_frac=frac) and
                      weights_close(b, rb, lr, n, extra=allow[li][1] * scale, outlier_frac=frac))
            else:
                ok = weights_close(w, rw, lr, n) and weights_close(b, rb, lr, n)
            assert ok, (name, li)


# ---- e. GCRL_FUSED_R accepts 2, 4 or 8 only --------------------------------------------------------------------
@pytest.mark.parametrize("value", ["16", "0"])
def test_invalid_rows_per_cta_setting_is_ignored(value, monkeypatch):
    """GCRL_FUSED_R outside {2, 4, 8} falls back to the default rule: the same weights, bit for bit, as without
    it.  (16 used to launch the R = 8 kernels on ceil(B / 16) CTAs, i.e. on half the batch; 0 divided by zero.)"""
    B, D, A, H, L = 128, 22, 3, 64, 3
    rng = np.random.default_rng(16)
    nets = init_nets(rng, "ddpg", D, A, H, L)
    batches = [make_batch(rng, B, D, A) for _ in STEPS]
    runs = []
    for v in (None, value):
        if v is None:
            monkeypatch.delenv("GCRL_FUSED_R", raising=False)
        else:
            monkeypatch.setenv("GCRL_FUSED_R", v)
        ag = make_agent("ddpg", B, nets, monkeypatch, D, A, H, L, graphs=True)
        runs.append((run_updates(ag, "ddpg", batches, [None] * len(STEPS)), all_weights(ag)))
    assert runs[0][0] == runs[1][0]
    assert first_difference(runs[0][1], runs[1][1]) is None

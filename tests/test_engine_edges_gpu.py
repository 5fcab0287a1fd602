"""GPU: DDPG and TD3 updates on the two large-batch engines -- the fp32 FFMA tiles (mlp.cu) and tcgen05
(tc_gemm.cu) -- against the NumPy oracle at every branch of the loss and the target, uniform and with prioritised
weights (flags bit 3).

Neither engine shares the row-slab kernels' loss code: head_bwd_kernel (mlp.cu) forms the Bellman target, DDPG's y
clamp, TD3's smooth-L1 branch, the importance weights, the per-sample TD write-back and TD3's max(td1, td2);
td3_smooth_kernel applies the noise and action clamps; action_grad_kernel and the dgrad GEMMs carry the actor
gradient.  Every case

  * proves its engine under torch.profiler: no row-slab kernel; fp32 tiles: gemm_kernel runs and no tc_dense*
    kernel does; tcgen05: tc_dense_kernel runs, or tc_dense_pair_kernel where the batch fills the CTA pairs;
  * asserts that every branch of test_fused_variants_gpu.branches_hit is taken by some rows and not by others;
  * runs four updates (steps 39-42: DDPG's Polyak step at 40, TD3's actor steps at 40 and 42) and compares the
    metrics, the per-sample TD (prioritised) and the weights of all 4 / 6 networks with the oracle, at the
    tolerances the project uses for each engine (test_branch_edges_match_oracle for the fp32 tiles,
    test_tensor_core_update_matches_fp32_update for tcgen05), and prints the worst errors it saw.
"""
import re

import numpy as np
import pytest

from oracle import ddpg as OD
from oracle import td3 as OT
from tests.helpers import weight_error_report, weights_close
from tests.test_fused_variants_gpu import (EDGE, EDGE_STEPS, PUSH, as_oracle_tuple, branches_hit, edge_batch, init_nets,
                                           launched_kernels, make_agent, priority_weights, update_direct)

pytestmark = pytest.mark.gpu

# id -> (engine, B, network shape, precision, GCRL_B200_NO_FUSED).  The row-slab kernels take B <= 1024 unless
# GCRL_B200_NO_FUSED=1; tcgen05 takes B >= 2048 at precision 1 and B >= 128 at precision 2 (agent.cu::use_tc).
CASES = {
    "tiles-B1500": ("tiles", 1500, EDGE, 1, False),
    "tiles-B2047": ("tiles", 2047, EDGE, 1, False),
    "tiles-nofused-B301": ("tiles", 301, EDGE, 0, True),      # head_bwd: 19 slabs of 16 rows, the last one 13
    "tc-B2048": ("tc", 2048, EDGE, 1, False),
    "tc-B4096": ("tc", 4096, EDGE, 1, False),
    "tc-nofused-B517": ("tc", 517, EDGE, 2, True),
    # CTA pairs need N % 256 == 0 and 4 * ceil(B / 256) >= 3 * (pairs resident): 65 tiles of 256 rows, the last
    # holding one row
    "pairs-B16385": ("pairs", 16385, PUSH, 1, False),
}
ENGINE_KERNEL = re.compile(r"\b(gemm_kernel|tc_dense_kernel|tc_dense_pair_kernel)<")


def check_engine(names, engine, label, capsys):
    ran = {m.group(1) for n in names for m in ENGINE_KERNEL.finditer(n)}
    slab = sorted(n for n in names if "fused_" in n)
    with capsys.disabled():
        print(f"\n[engine] {label}: " + ", ".join(sorted(ran)) + (f"; row-slab: {slab}" if slab else ""))
    assert not slab, (label, slab)
    if engine == "tiles":
        assert "gemm_kernel" in ran and not any("tc_dense" in n for n in names), (label, sorted(ran))
    else:
        assert ("tc_dense_pair_kernel" if engine == "pairs" else "tc_dense_kernel") in ran, (label, sorted(ran))


@pytest.mark.parametrize("weighted", [False, True], ids=["uniform", "prioritised"])
@pytest.mark.parametrize("algo", ["ddpg", "td3"])
@pytest.mark.parametrize("case", list(CASES))
def test_engine_branch_edges_match_oracle(case, algo, weighted, monkeypatch, capsys):
    """test_branch_edges_match_oracle on the fp32 tiles and on tcgen05.  Tolerances: metrics at 5e-5 * sqrt(B / 256)
    (tcgen05: times the step number, the implementations drift apart step by step) plus the oracle's LeakyReLU flip
    slack on DDPG's gradient norms; per-sample TD at rel 5e-5 + 5e-6 (tcgen05: 4x); weights at weights_close
    (tcgen05: rtol 4e-5 and 4x the Adam allowance, the 3xTF32 engine's ~2e-6 per layer against the tiles' ~5e-7)."""
    engine, B, shape, precision, no_fused = CASES[case]
    D, A, H, L = shape["D"], shape["A"], shape["H"], shape["L"]
    tc = engine != "tiles"
    monkeypatch.delenv("GCRL_FUSED_R", raising=False)
    if no_fused:
        monkeypatch.setenv("GCRL_B200_NO_FUSED", "1")             # read at creation
    else:
        monkeypatch.delenv("GCRL_B200_NO_FUSED", raising=False)
    rng = np.random.default_rng(3 * B + 2 * (algo == "td3") + weighted)
    nets = init_nets(rng, algo, D, A, H, L)
    pn, nc, gamma, lr = 0.5, 1.5, 0.98, 1e-3
    ag = make_agent(algo, B, nets, monkeypatch, D, A, H, L, precision=precision, policy_noise=pn, noise_clamp=nc,
                    gamma=gamma)
    kw = dict(gamma=gamma, tau=0.05, grad_clip=0.5, actor_lr=lr, critic_lr=lr, ac_update_freq=ag.ac_update_freq)
    if algo == "ddpg":
        orc = OD.DDPGOracle(*nets, **kw)
        orc.flip_delta = 2e-5 if tc else 5e-6
    else:
        orc = OT.TD3Oracle(*nets, policy_noise=pn, noise_clamp=nc, **kw)
    label = f"{case} {algo} {'prioritised' if weighted else 'uniform'}"
    hit = {}
    critic_flips = False
    base = 5e-5 * max(1.0, (B / 256.0) ** 0.5)
    td_rtol, td_atol = (2e-4, 2e-5) if tc else (5e-5, 5e-6)
    # TD3Oracle does not track LeakyReLU flips (DDPGOracle._flip_track does).  On tcgen05, with 4x the tiles' rounding,
    # the few weight elements whose gradient is at that rounding level take the other Adam sign (a 2 lr step, the
    # sign regime of weights_close) -- on the PUSH shape at B = 16 385 in more than weights_close's 2e-4 of a tensor --
    # and the rows whose Q such a critic weight moves carry it into their TD.  Those are held to Adam's hard bound /
    # 10x the TD tolerance, on at most 5e-3 of the elements / rows: the allowance the DDPG tests give the actor
    # elements the stepped critic moves.
    sign_regime_frac = 5e-3 if (tc and algo == "td3") else 0.0
    failures = []
    worst_metric = worst_td = 0.0               # largest |error| / allowance seen
    for si, step in enumerate(EDGE_STEPS):
        batch, randn = edge_batch(rng, algo, B, D, A)
        w = priority_weights(rng, B) if weighted else None
        for name, rows in branches_hit(orc, algo, batch, randn, gamma, pn, nc).items():
            taken, total, split = hit.get(name, (0, 0, False))          # split: some rows take it and some do not
            hit[name] = taken + int(rows.sum()), total + rows.size, split or bool(rows.any() and not rows.all())
        noise = randn if algo == "td3" else None
        if si == 0:
            out = []
            check_engine(launched_kernels(lambda: out.append(update_direct(ag, step, batch, noise, w))), engine, label,
                         capsys)
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
        rtol = np.full(len(want), base * (si + 1 if tc else 1))
        if algo == "ddpg":
            rtol[-2 if actor_step else -1] += orc.last_critic_flip_slack
            if actor_step:
                rtol[-1] += orc.last_actor_flip_slack
            critic_flips = critic_flips or orc.last_critic_flip_slack > 0
        keep = [i for i in range(len(want)) if not (weighted and i == td_pos)]
        g_, w_ = np.array(got)[keep], np.array([float(want[i]) for i in keep])
        allowed = rtol[keep] * np.abs(w_) + 2e-6
        worst_metric = max(worst_metric, float(np.max(np.abs(g_ - w_) / allowed)))
        for i in np.flatnonzero(np.abs(g_ - w_) > allowed):
            failures.append(("metric", step, keep[i], float(g_[i]), float(w_[i]), float(rtol[keep][i])))
        if weighted:
            want_td = np.asarray(want[td_pos], np.float64).ravel()
            err = np.abs(td.astype(np.float64) - want_td)
            ratio = err / (td_rtol * np.abs(want_td) + td_atol)
            worst_td = max(worst_td, float(ratio.max()))
            if ratio.max() > (10.0 if sign_regime_frac else 1.0) or np.mean(ratio > 1.0) > sign_regime_frac:
                failures.append(("td", step, int(np.argmax(err)), float(err.max()), float(np.mean(ratio > 1.0))))
    n = len(EDGE_STEPS)
    if algo == "ddpg":
        pairs = (("actor", ag.actor, orc.actor), ("critic", ag.critic, orc.critic),
                 ("target_actor", ag.target_actor, orc.target_actor), ("target_critic", ag.target_critic, orc.target_critic))
    else:
        pairs = (("actor", ag.actor, orc.actor), ("critic_1", ag.critic_1, orc.critic_1),
                 ("critic_2", ag.critic_2, orc.critic_2), ("target_actor", ag.target_actor, orc.target_actor),
                 ("target_critic_1", ag.target_critic_1, orc.target_critic_1),
                 ("target_critic_2", ag.target_critic_2, orc.target_critic_2))
    w_lr, w_rtol = (4 * lr, 4e-5) if tc else (lr, 1e-5)
    worst_w = (0.0, 0.0, "")                     # (max |error|, share of the bulk allowance used by its 99.99 %)
    worst_over = 0.0                             # largest fraction of a tensor beyond the bulk allowance
    for name, net, ref in pairs:
        for li, ((wt, b), (rw, rb)) in enumerate(zip(net.layers(), ref)):
            ew = eb = None
            frac = max(2e-4, sign_regime_frac)
            if algo == "ddpg":       # per-element LeakyReLU flip allowance, as in test_update_matches_oracle_odd_shapes
                allow = orc.flip_allowance if "actor" in name else orc.flip_allowance_critic
                scale = 0.05 * n if name.startswith("target") else 1.0
                ew, eb = allow[li][0] * scale, allow[li][1] * scale
                frac = 5e-3 if ("actor" in name and critic_flips) else 2e-4
            mx, _, tol, used = weight_error_report(wt, rw, w_lr, n, rtol=w_rtol)
            if not worst_w[2] or used > worst_w[1]:
                worst_w = (mx, used, f"{name}.{li}")
            over = float(np.mean(np.abs(np.asarray(wt, np.float64) - rw) > tol))    # before the flip allowance
            worst_over = max(worst_over, over)
            if not (weights_close(wt, rw, w_lr, n, rtol=w_rtol, extra=ew, outlier_frac=frac) and
                    weights_close(b, rb, w_lr, n, rtol=w_rtol, extra=eb, outlier_frac=frac)):
                failures.append(("weights", name, li, mx, used, over))
    with capsys.disabled():
        print(f"[branches] {label}: " + ", ".join(f"{k}: {v[0]} of {v[1]}" for k, v in hit.items()))
        print(f"[errors] {label}: metrics {100 * worst_metric:.1f} % of allowance, " +
              (f"per-sample TD {100 * worst_td:.1f} %, " if weighted else "") +
              f"weights max |err| {worst_w[0]:.2e} in {worst_w[2]} (99.99 % at {100 * worst_w[1]:.1f} % of the bulk allowance; "
              f"at most {100 * worst_over:.3f} % of a tensor beyond it)")
    assert all(split for _, _, split in hit.values()), hit
    assert not failures, failures

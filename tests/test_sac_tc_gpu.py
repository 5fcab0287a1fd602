"""GPU: the SAC / TQC tensor-core engine (precision 1 / 2: hidden-layer GEMMs of the critics and the actor on tcgen05
with the 3xTF32 split, the critic ensemble batched into one launch per layer).

Stated tolerance (DESIGN.md 5): 4x the fp32 engines' -- metrics rel 8e-5 + abs 4e-6 (times sqrt(B / 256) above 256
rows), weights tests.helpers.weights_close with rtol 4e-5 and 4x its Adam allowance, BatchNorm running variance
rel 4e-5.  The ensemble kernel itself is held to bit-identity with the single-problem launch."""
import ctypes as C

import numpy as np
import pytest

from tests import test_sac_gpu as T
from tests.helpers import SAC_CASES, load, sac_initial_nets, sac_params_from_golden, weights_close

pytestmark = pytest.mark.gpu

ENG = 4.0                     # the tensor-core engine's tolerance factor over the fp32 engines'


def _tc_kernels_ran(fn):
    """Run fn() under torch.profiler; number of tcgen05 dense / weight-gradient kernel launches seen."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(1 for e in prof.events() if "tc_dense_kernel" in e.name or "tc_dense_pair_kernel" in e.name)


# ---- 1. the ensemble kernel ------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [128, 200, 512, 4096])
@pytest.mark.parametrize("n", [1, 2, 5])
def test_ensemble_launch_equals_single_launches_bitwise(n, M):
    """Members with distinct weights, every mode (3 = bare product): each member's output equals
    gcrl_dense_layer_presplit of that member alone bit for bit, matches float64 to 1e-5 (the bound of
    test_tc_gemm_gpu.py), and the guard cells around every output (padding columns and rows past M) are untouched."""
    import torch
    from gcrl_b200._lib import check, lib, vp
    st = vp(torch.cuda.current_stream().cuda_stream)
    guard = 12345.0
    for N in (64, 256, 512):
        for K in (28, 256):
            torch.manual_seed(n * 1000 + M + N + K)
            ldx, ldw, ldy = K + 4, K + 8, N + 8
            xs = [torch.randn(M, ldx, device="cuda") for _ in range(n)]
            ws = [torch.randn(N, ldw, device="cuda") / K ** 0.5 for _ in range(n)]
            bs = [torch.randn(N, device="cuda") for _ in range(n)]
            acts = [torch.randn(M, N, device="cuda") for _ in range(n)]
            his, los = [torch.empty_like(w) for w in ws], [torch.empty_like(w) for w in ws]
            for w, hi, lo in zip(ws, his, los):
                check(lib.gcrl_split_tf32(0, vp(w.data_ptr()), vp(hi.data_ptr()), vp(lo.data_ptr()), w.numel(), st))
            arr = lambda ts: (C.c_void_p * n)(*[t.data_ptr() for t in ts])  # noqa: E731
            for mode in (0, 1, 2, 3):
                ys = [torch.full((M + 3, ldy), guard, device="cuda") for _ in range(n)]
                check(lib.gcrl_dense_layer_ensemble(0, n, mode, M, N, K, arr(xs), ldx, arr(his), arr(los), ldw,
                                                    arr(bs) if mode in (0, 2) else None,
                                                    arr(acts) if mode == 1 else None, N, arr(ys), ldy, st))
                for i in range(n):
                    one = torch.full((M + 3, ldy), guard, device="cuda")
                    check(lib.gcrl_dense_layer_presplit(0, mode, M, N, K, vp(xs[i].data_ptr()), ldx,
                                                        vp(his[i].data_ptr()), vp(los[i].data_ptr()), ldw,
                                                        vp(bs[i].data_ptr()) if mode in (0, 2) else None,
                                                        vp(acts[i].data_ptr()) if mode == 1 else None, N,
                                                        vp(one.data_ptr()), ldy, st))
                    torch.cuda.synchronize()
                    tag = (n, M, N, K, mode, i)
                    assert torch.equal(ys[i], one), tag
                    assert bool((ys[i][:M, N:] == guard).all()) and bool((ys[i][M:] == guard).all()), tag
                    ref = xs[i][:, :K].double() @ ws[i][:, :K].double().T
                    want = {0: torch.nn.functional.leaky_relu(ref + bs[i].double(), 0.01),
                            1: ref * torch.where(acts[i] > 0, 1.0, 0.01).double(),
                            2: ref + bs[i].double(), 3: ref}[mode]
                    err = ((ys[i][:M, :N].double() - want).abs().max() / want.abs().max()).item()
                    assert err <= 1e-5, (tag, err)


# ---- 2. reference fixtures at precision 2 -------------------------------------------------------------------
def _make_fixture_agent(algo, g, precision):
    from gcrl_b200 import SACAgent, TQCAgent
    D, A, H, L, B, seed, freq, gstep, amin = (int(x) for x in g["meta"])
    gamma, tau, clip, lr, alpha_lr = (float(x) for x in g["hp"])
    cfg = T.sac_config(hidden_dim=H, layer_count=L, batch_size=B, gamma=gamma, tau=tau, grad_clip=clip, actor_lr=lr,
                       critic_lr=lr, actor_lr_min=lr, critic_lr_min=lr, ac_update_freq=freq, alpha_lr=alpha_lr,
                       alpha_min_steps=amin)
    ag = (SACAgent if algo == "sac" else TQCAgent)(D, A, cfg, None, 1, gstep, precision=precision)
    T.load_initial(ag, *sac_initial_nets(algo, g))
    return ag


def _assert_actor_close(params, ref, lr, n, eng):
    L = (len(params) - 2) // 2
    for i, ((w, b), (rw, rb)) in enumerate(zip(params, ref)):
        assert weights_close(w, rw, lr * eng, n, rtol=1e-5 * eng), ("actor", i)
        if i < 2 * L and i % 2 == 0:       # pre-BatchNorm bias: zero true gradient, Adam's hard bound only
            assert float(np.max(np.abs(np.asarray(b, np.float64) - rb))) <= 2.0 * lr * n + 1e-6, ("actor bias", i)
        else:
            assert weights_close(b, rb, lr * eng, n, rtol=1e-5 * eng), ("actor", i)


@pytest.mark.parametrize("algo,case", SAC_CASES)
def test_precision2_matches_reference_fixture(algo, case):
    """The four SAC / TQC fixtures (B = 128..256, H = 64 / 256) at precision 2, where every hidden-layer GEMM runs on
    tcgen05: metrics every step and all weights, BatchNorm statistics and log_alpha after the last, against the
    unmodified reference at the stated tolerance; the tcgen05 kernels must actually have run."""
    import torch
    g = load(f"{algo}_{case}")
    ag = _make_fixture_agent(algo, g, 2)
    lr = float(g["hp"][3])
    B = int(g["meta"][4])
    steps = [int(x) for x in g["steps"]]
    rtol = ENG * 2e-5 * max(1.0, (B / 256.0) ** 0.5)
    ran = 0
    for si, step in enumerate(steps):
        def one():
            return ag.update(step, batch=T.batch_to_device(g, si), eps_next=torch.from_numpy(g[f"s{si}_eps_next"]).cuda(),
                             eps_cur=torch.from_numpy(g[f"s{si}_eps_cur"]).cuda())
        if si == 0:
            info = one()
        else:
            box = []
            ran += _tc_kernels_ran(lambda: box.append(one()))
            info = box[0]
        np.testing.assert_allclose(np.array([float(x) for x in info]), g[f"s{si}_info"], rtol=rtol, atol=ENG * 1e-6)
        np.testing.assert_allclose(ag.get_log_alpha(), float(g[f"s{si}_log_alpha"][0]), rtol=ENG * 1e-5, atol=1e-7)
    assert ran > 0, "precision 2 must run the tcgen05 kernels"
    si, n = len(steps) - 1, len(steps)
    params, stats = T.actor_params(ag)
    ref = sac_params_from_golden(g, si, "actor")
    _assert_actor_close(params, ref["params"], lr, n, ENG)
    for (m, v), (rm, rv) in zip(stats, ref["stats"]):
        np.testing.assert_allclose(m, rm, rtol=ENG * 1e-5, atol=2.0 * lr * n)
        np.testing.assert_allclose(v, rv, rtol=ENG * 1e-5, atol=1e-6)
    for i in (0, ag.N_CRITICS - 1):                 # the critics the fixtures record
        tag = f"critic_{i + 1}" if algo == "sac" else f"critic_{i}"
        for view, t in ((ag._critic_views[i], tag), (ag._target_views[i], "target_" + tag)):
            for (w, b), (rw, rb) in zip(view.layers(), sac_params_from_golden(g, si, t)):
                assert weights_close(w, rw, lr * ENG, n, rtol=1e-5 * ENG), (case, t)
                assert weights_close(b, rb, lr * ENG, n, rtol=1e-5 * ENG), (case, t)


def _make(algo, D, A, H, L, B, seed=5, precision=0, default=False):
    from gcrl_b200 import SACAgent, TQCAgent
    from oracle import ddpg as OD
    from oracle import sac as OS
    rng = np.random.default_rng(seed)
    cfg = T.sac_config(hidden_dim=H, layer_count=L, batch_size=B, grad_clip=0.5, tau=0.05, alpha_min_steps=0,
                       alpha_lr=1e-2)
    actor0, stats0 = OS.init_sac_actor(rng, D, H, A, L, head_scale=0.1, log_std_bias=-1.0)
    critics0 = [OD.init_mlp(rng, D + A, H, 1, L) for _ in range(2 if algo == "sac" else 5)]
    cls = SACAgent if algo == "sac" else TQCAgent
    ag = cls(D, A, cfg, None, 1, 2) if default else cls(D, A, cfg, None, 1, 2, precision=precision)
    T.load_initial(ag, actor0, stats0, critics0)
    return ag, (actor0, stats0, critics0)


def _assert_close_to(ag, actor, stats, critics, targets, lr, n):
    """ag's weights, BatchNorm statistics, critics and target critics against another run's, at the stated
    tolerance (pre-BatchNorm Linear biases, whose true gradient is zero, to Adam's hard bound only)."""
    params, st = T.actor_params(ag)
    _assert_actor_close(params, actor, lr, n, ENG)
    for (m, v), (rm, rv) in zip(st, stats):
        np.testing.assert_allclose(m, rm, rtol=ENG * 1e-5, atol=2.0 * lr * n)
        np.testing.assert_allclose(v, rv, rtol=ENG * 1e-5, atol=1e-6)
    for views, refs in ((ag._critic_views, critics), (ag._target_views, targets)):
        for i, (view, ref) in enumerate(zip(views, refs)):
            for k, ((w, b), (rw, rb)) in enumerate(zip(view.layers(), ref)):
                assert weights_close(w, rw, lr * ENG, n, rtol=1e-5 * ENG), (i, k)
                assert weights_close(b, rb, lr * ENG, n, rtol=1e-5 * ENG), (i, k)


def _state(ag):
    p, s = T.actor_params(ag)
    return p, s, [v.layers() for v in ag._critic_views], [v.layers() for v in ag._target_views]


def _all_params(ag):
    p, s = T.actor_params(ag)
    out = [x for pair in p + s for x in pair]
    for v in ag._critic_views + ag._target_views:
        out += [x for pair in v.layers() for x in pair]
    return out + [np.float32(ag.get_log_alpha())]


def test_precision0_runs_no_tensor_core_kernel_and_equals_the_default():
    import torch
    D, A, H, L, B = 22, 3, 64, 3, 256
    rng = np.random.default_rng(0)
    data = [T._rand_batch(rng, B, D, A) for _ in range(3)]
    agents = [_make("tqc", D, A, H, L, B, default=True)[0], _make("tqc", D, A, H, L, B, precision=0)[0]]
    for ag in agents:
        for step, (*batch, e1, e2) in enumerate(data, 1):
            assert _tc_kernels_ran(lambda: ag.update(step, batch=tuple(batch), eps_next=e1, eps_cur=e2)) == 0
    for x, y in zip(_all_params(agents[0]), _all_params(agents[1])):
        assert np.array_equal(x, y)
    torch.cuda.synchronize()


@pytest.mark.parametrize("algo", ["sac", "tqc"])
def test_precision1_below_its_threshold_equals_precision0_bitwise(algo):
    D, A, H, L, B = 22, 3, 256, 3, 512
    rng = np.random.default_rng(1)
    data = [T._rand_batch(rng, B, D, A) for _ in range(3)]
    infos, agents = [], []
    for p in (0, 1):
        ag = _make(algo, D, A, H, L, B, precision=p)[0]
        infos.append([[float(x) for x in ag.update(s, batch=tuple(b[:5]), eps_next=b[5], eps_cur=b[6])]
                      for s, b in enumerate(data, 1)])
        agents.append(ag)
    assert infos[0] == infos[1]
    for x, y in zip(_all_params(agents[0]), _all_params(agents[1])):
        assert np.array_equal(x, y)


# ---- 3. large batches at precision 1 against the oracle and precision 0 -------------------------------------
@pytest.mark.parametrize("algo,B", [("sac", 2048), ("sac", 4096), ("tqc", 2048), ("tqc", 4096), ("tqc", 8192)])
def test_precision1_large_batch_metrics_match_oracle(algo, B):
    """Three updates with gradient_step 2 (critic steps, actor + alpha steps, Polyak steps) at precision 1, where the
    tensor cores run: every metric and log_alpha against the NumPy oracle at the stated tolerance.  B = 8192 takes the
    per-critic backward loop above kEnsembleBatchMax, the others the batched ensemble path.  The weights are compared
    with precision 0 below: at these batches the fp32 engine itself drifts from the oracle's weights (DESIGN.md 5)."""
    from oracle import sac as OS
    D, A, H, L = 22, 3, 256, 3
    rng = np.random.default_rng(B + len(algo))
    data = [T._rand_batch(rng, B, D, A) for _ in range(3)]
    ag, (actor0, stats0, critics0) = _make(algo, D, A, H, L, B, seed=7, precision=1)
    cfg = ag.config
    orc = OS.SACOracle(algo, actor0, stats0, critics0, act_dim=A, gamma=cfg.gamma, tau=cfg.tau,
                       grad_clip=cfg.grad_clip, actor_lr=cfg.actor_lr, critic_lr=cfg.critic_lr, alpha_lr=1e-2,
                       alpha_min_steps=0, gradient_step=2)
    rtol = ENG * 5e-5 * (B / 256.0) ** 0.5          # test_sac_gpu.py's oracle bound, times the engine factor
    for s, b in enumerate(data, 1):
        want = np.array(orc.update_on_batch(s, *(t.cpu().numpy() for t in b)), np.float64)
        got = ag.update(s, batch=tuple(b[:5]), eps_next=b[5], eps_cur=b[6])
        np.testing.assert_allclose(np.array([float(x) for x in got]), want, rtol=rtol, atol=ENG * 2e-6)
        np.testing.assert_allclose(ag.get_log_alpha(), float(orc.log_alpha), rtol=ENG * 1e-5, atol=1e-7)


class _AdamTrack:
    """Per-element bound on how far one flat parameter buffer of the tensor-core run may sit from the same buffer of
    the precision-0 run, given the two runs' clipped gradients of every step (Adam's sign regime, DESIGN.md 5).
    The difference d = |g1 - g0| of a step enters both moments, dm <- b1 dm + (1 - b1) d, dv <- b2 dv +
    (1 - b2)(2 |g0| d + d^2); the step lr/bc1 * m / (sqrt(v)/sqrt(bc2) + eps) is monotone in m and in v separately,
    so its largest deviation over the box [m +- dm] x [v +- dv] is at a corner (as oracle/ddpg.py::_flip_track).
    The allowance accumulates that deviation, capped at Adam's hard bound 2 lr per step.  An element whose gradient
    is far above the engines' difference gets almost nothing; one whose gradient sits at that difference gets up to
    2 lr -- which is what Adam does to it in either engine."""

    def __init__(self, n):
        self.m, self.v, self.dm, self.dv = (np.zeros(n) for _ in range(4))
        self.allow, self.t = np.zeros(n), 0

    def step(self, g0, g1, lr, b1=0.9, b2=0.999, eps=1e-8):
        self.t += 1
        bc1, bc2s = 1.0 - b1 ** self.t, (1.0 - b2 ** self.t) ** 0.5
        d = np.abs(g1 - g0)
        self.dm = b1 * self.dm + (1.0 - b1) * d
        self.dv = b2 * self.dv + (1.0 - b2) * (2.0 * np.abs(g0) * d + d * d)
        self.m = b1 * self.m + (1.0 - b1) * g0
        self.v = b2 * self.v + (1.0 - b2) * g0 * g0
        nom = self.m / (np.sqrt(self.v) / bc2s + eps)
        dev = np.zeros_like(nom)
        for mm in (self.m - self.dm, self.m + self.dm):
            for vv in (np.maximum(self.v - self.dv, 0.0), self.v + self.dv):
                dev = np.maximum(dev, np.abs(mm / (np.sqrt(vv) / bc2s + eps) - nom))
        self.allow += np.minimum(2.0 * lr, (lr / bc1) * dev)


def _clipped(g, clip):
    g = np.asarray(g, np.float64)
    return g * min(1.0, clip / (float(np.sqrt(np.sum(g * g))) + 1e-6))


def _actor_slices(D, A, H, L):
    """(param index in T.actor_params order, weight / bias / BN slot, offset, rows, cols, ld) of the actor's flat buffer
    (csrc/sac.cu ActorNet)."""
    pad = lambda x: (x + 3) // 4 * 4  # noqa: E731
    out, off = [], 0
    for l in range(L):
        ld = pad(D if l == 0 else H)
        out += [(2 * l, 0, off, H, D if l == 0 else H, ld)]; off += H * ld
        out += [(2 * l, 1, off, 1, H, H)]; off += pad(H)
        out += [(2 * l + 1, 0, off, 1, H, H)]; off += pad(H)
        out += [(2 * l + 1, 1, off, 1, H, H)]; off += pad(H)
    for k in (2 * L, 2 * L + 1):
        out += [(k, 0, off, A, H, pad(H))]; off += A * pad(H)
        out += [(k, 1, off, 1, A, A)]; off += 4
    return out, off


def _critic_slices(D, A, H, L):
    pad = lambda x: (x + 3) // 4 * 4  # noqa: E731
    out, off = [], 0
    for l in range(L + 1):
        i, o = (D + A if l == 0 else H), (1 if l == L else H)
        out += [(l, 0, off, o, i, pad(i))]; off += o * pad(i)
        out += [(l, 1, off, 1, o, o)]; off += pad(o)
    return out, off


def _unflat(flat, sl):
    return {(k, j): flat[off:off + r * ld].reshape(r, ld)[:, :c].reshape(-1) for k, j, off, r, c, ld in sl}


@pytest.mark.parametrize("algo,B", [("sac", 2048), ("sac", 4096), ("tqc", 2048), ("tqc", 4096), ("tqc", 8192)])
def test_precision1_large_batch_matches_precision0(algo, B):
    """Precision 1 (tensor cores) against precision 0 on the same weights and inputs, three updates (critic, actor,
    alpha every step; Polyak at step 2 for SAC, every step for TQC): every metric and log_alpha at the stated
    tolerance; the first step's flat gradients of every network within 1e-3 of their max-norm (both runs start from the same weights, so this is the
    engine alone: measured up to 5.1e-4); and every weight -- actor
    Linears, BatchNorm parameters and running statistics, heads, critics, target critics -- within the stated
    tolerance plus the element-wise Adam allowance that the two runs' gradient differences carry (_AdamTrack).
    Comparing with precision 0 rather than the oracle isolates the engine: at these batches the fp32 engine itself
    drifts from the NumPy oracle by up to 9e-4 (TQC, B = 4096)."""
    D, A, H, L, n = 22, 3, 256, 3, 3
    rng = np.random.default_rng(B + len(algo))
    data = [T._rand_batch(rng, B, D, A) for _ in range(n)]
    ags = {p: _make(algo, D, A, H, L, B, seed=7, precision=p)[0] for p in (0, 1)}
    cfg = ags[0].config
    lr, clip, nc = cfg.critic_lr, cfg.grad_clip, ags[0].N_CRITICS
    asl, atot = _actor_slices(D, A, H, L)
    csl, ctot = _critic_slices(D, A, H, L)
    track_a, track_c = _AdamTrack(atot), [_AdamTrack(ctot) for _ in range(nc)]
    rtol = ENG * 2e-5 * (B / 256.0) ** 0.5
    tau_allow = [np.zeros(ctot) for _ in range(nc)]
    worst = 0.0
    for s, b in enumerate(data, 1):
        info, ga, gc = {}, {}, {}
        for p, ag in ags.items():
            info[p] = [float(x) for x in ag.update(s, batch=tuple(b[:5]), eps_next=b[5], eps_cur=b[6])]
            ga[p] = ag.grad_tensor(0).double().cpu().numpy()[:atot]
            gc[p] = ag.grad_tensor(1).double().cpu().numpy().reshape(nc, ctot)
        np.testing.assert_allclose(info[1], info[0], rtol=rtol, atol=ENG * 1e-6, err_msg=f"step {s}")
        np.testing.assert_allclose(ags[1].get_log_alpha(), ags[0].get_log_alpha(), rtol=ENG * 1e-5, atol=1e-7)
        for g0, g1 in [(ga[0], ga[1])] + [(gc[0][i], gc[1][i]) for i in range(nc)]:
            if s == 1:          # same weights in both runs: the difference is the engine's alone
                err = float(np.max(np.abs(g1 - g0)) / np.max(np.abs(g0)))
                worst = max(worst, err)
                assert err <= 1e-3, err
        track_a.step(_clipped(ga[0], clip), _clipped(ga[1], clip), lr)
        for i in range(nc):
            track_c[i].step(_clipped(gc[0][i], clip), _clipped(gc[1][i], clip), lr)
            if ags[0]._polyak_now(s):                        # Polyak: the target moves by tau of the difference
                tau_allow[i] = tau_allow[i] * (1 - cfg.tau) + cfg.tau * track_c[i].allow
    print(f"{algo} B={B}: first-step gradient difference {worst:.1e} of the max-norm")
    allow_a = _unflat(track_a.allow, asl)
    (p0, s0), (p1, s1) = T.actor_params(ags[0]), T.actor_params(ags[1])
    for k in range(len(p0)):
        for j in range(2):
            w, ref = p1[k][j], p0[k][j]
            if k < 2 * L and k % 2 == 0 and j == 1:          # pre-BatchNorm bias: zero true gradient
                assert float(np.max(np.abs(np.asarray(w, np.float64) - ref))) <= 2.0 * lr * n + 1e-6, ("actor bias", k)
                continue
            assert weights_close(w, ref, lr * ENG, n, rtol=1e-5 * ENG, extra=allow_a[(k, j)]), ("actor", k, j)
    # running statistics: 4x the fp32 tolerance plus what the differences of the unit's incoming weights dw and bias
    # db can move the batch moments of z = w.x + b:  |dmean| <= |db| + |dw|_1 rms,  |dvar| <= 2 sd(z) |dw|_1 rms +
    # (|dw|_1 rms)^2  with rms >= the rms of every input column (layer 0: the batch; later layers: relu(gamma xhat +
    # beta) <= |gamma| + |beta|), summed over the 2 n running updates (momentum 0.1: weights < 0.5 in all) with the
    # final differences, and var(z) <= 10 running_var
    rms_in = max(float(np.sqrt(np.mean(np.concatenate([b[0].cpu().numpy(), b[3].cpu().numpy()]) ** 2, 0)).max())
                 for b in data)
    for k, ((rm, rv), (rm0, rv0)) in enumerate(zip(s1, s0)):
        rms = rms_in if k == 0 else float(np.max(np.abs(p0[2 * k - 1][0]) + np.abs(p0[2 * k - 1][1])))
        dl = np.sum(np.abs(np.asarray(p1[2 * k][0], np.float64) - p0[2 * k][0]), axis=1) * rms
        db = np.abs(np.asarray(p1[2 * k][1], np.float64) - p0[2 * k][1])
        mean_allow = 0.5 * (db + dl)
        var_allow = 0.5 * (2.0 * np.sqrt(10.0 * np.asarray(rv0, np.float64)) * dl + dl * dl)
        err_m = np.abs(np.asarray(rm, np.float64) - rm0)
        err_v = np.abs(np.asarray(rv, np.float64) - rv0)
        assert np.all(err_m <= ENG * 1e-5 * np.abs(rm0) + 2e-6 + mean_allow), f"running_mean {k}"
        assert np.all(err_v <= ENG * 2e-5 * np.abs(rv0) + 1e-7 + var_allow), f"running_var {k}"
    for i in range(nc):
        ac, at = _unflat(track_c[i].allow, csl), _unflat(tau_allow[i], csl)
        for views, al in ((lambda a: a._critic_views, ac), (lambda a: a._target_views, at)):
            for k, ((w, bb), (rw, rb)) in enumerate(zip(views(ags[1])[i].layers(), views(ags[0])[i].layers())):
                assert weights_close(w, rw, lr * ENG, n, rtol=1e-5 * ENG, extra=al[(k, 0)]), (i, k)
                assert weights_close(bb, rb, lr * ENG, n, rtol=1e-5 * ENG, extra=al[(k, 1)]), (i, k)


# ---- 4. bit-identity properties at precision 2 ---------------------------------------------------------------
def _make_p2(algo, D, A, H, L, B, seed=5):
    return _make(algo, D, A, H, L, B, seed=seed, precision=2)[0]


@pytest.mark.parametrize("sync_bn", [False, True])
@pytest.mark.parametrize("algo", ["sac", "tqc"])
def test_precision2_world1_phases_and_segments_equal_whole_update_bitwise(algo, sync_bn, monkeypatch):
    """test_sac_gpu.py's world-of-one check with every agent at precision 2 (B = 128: the tensor cores run)."""
    monkeypatch.setattr(T, "_make", _make_p2)
    T.test_world1_phases_equal_whole_update_bitwise(algo, sync_bn)


@pytest.mark.parametrize("algo,world", [("sac", 2), ("tqc", 2)])
def test_precision2_sync_bn_ranks_equal_one_rank_on_the_concatenated_batch(algo, world, monkeypatch):
    monkeypatch.setattr(T, "_make", _make_p2)
    T.test_sync_bn_ranks_equal_one_rank_on_the_concatenated_batch(algo, world)


@pytest.mark.parametrize("algo", ["sac", "tqc"])
def test_precision2_graph_replay_equals_eager_launches(algo, monkeypatch):
    D, A, H, L, B = 22, 3, 64, 3, 256
    rng = np.random.default_rng(3)
    data = [T._rand_batch(rng, B, D, A) for _ in range(3)]
    graph = _make_p2(algo, D, A, H, L, B)
    monkeypatch.setenv("GCRL_B200_NO_GRAPH", "1")          # read when the agent is created
    eager = _make_p2(algo, D, A, H, L, B)
    monkeypatch.delenv("GCRL_B200_NO_GRAPH")
    for ag in (graph, eager):
        ag._infos = [[float(x) for x in ag.update(s, batch=tuple(b[:5]), eps_next=b[5], eps_cur=b[6])]
                     for s, b in enumerate(data, 1)]
    assert graph._infos == eager._infos
    for x, y in zip(_all_params(graph), _all_params(eager)):
        assert np.array_equal(x, y)


def test_precision2_update_from_buffer_equals_sample_then_update():
    import torch
    from gcrl_b200 import TQCAgent
    from tests.helpers import her_episodes
    g = load("her_reach_small")
    B = 128
    agents = []
    for _ in range(2):
        torch.manual_seed(0)
        ag = TQCAgent(10, 3, T.sac_config(batch_size=B, max_len=100000), None, 2, 2, precision=2)
        for ep in her_episodes(g):
            ag.buffer.push_episode(ep["s"], ep["a"], ep["ns"], ep["r"], ep["d"], ep["ag"], ep["fut"])
        agents.append(ag)
    src = agents[1]._critic_views + agents[1]._target_views
    for v_dst, v_src in zip(agents[0]._critic_views + agents[0]._target_views, src):
        v_dst.set_layers(v_src.layers())
    for l in range(agents[0].config.layer_count + 2):
        agents[0].actor.set_linear(l, *agents[1].actor.linear(l))
    assert len(agents[0].buffer) >= B
    rng = np.random.default_rng(4)
    for step in (1, 2, 3):
        idx = rng.permutation(len(agents[0].buffer))[:B]
        e1, e2 = torch.randn(B, 3, device="cuda"), torch.randn(B, 3, device="cuda")
        i0 = agents[0].update(step, indices=idx, eps_next=e1, eps_cur=e2)
        batch = tuple(torch.as_tensor(x).reshape(B, -1).cuda() for x in agents[1].buffer.sample_host(B, indices=idx))
        i1 = agents[1].update(step, batch=batch, eps_next=e1, eps_cur=e2)
        assert [float(x) for x in i0] == [float(x) for x in i1]
    for x, y in zip(_all_params(agents[0]), _all_params(agents[1])):
        assert np.array_equal(x, y)


# ---- 6. prioritised weights at precision 2 --------------------------------------------------------------------
@pytest.mark.parametrize("algo", ["sac", "tqc"])
def test_precision2_prioritised_weights_agree_with_precision0(algo):
    """flags bit 3: importance-weighted critic loss and the per-sample TD array, precision 2 against precision 0."""
    import torch
    from gcrl_b200._lib import check, lib, vp
    from gcrl_b200.parallel import device_tensor
    D, A, H, L, B = 22, 3, 256, 3, 256
    rng = np.random.default_rng(6)
    data = [T._rand_batch(rng, B, D, A) for _ in range(2)]
    isw = [torch.from_numpy(rng.uniform(0.2, 1.0, B).astype(np.float32)).cuda() for _ in data]
    st = vp(torch.cuda.current_stream().cuda_stream)
    out = {}
    for p in (0, 2):
        ag = _make(algo, D, A, H, L, B, precision=p)[0]
        w, td = vp(), vp()
        check(lib.gcrl_sac_per_buffers(ag._h, C.byref(w), C.byref(td)))
        wt, tdt = device_tensor(w.value, B, 0), device_tensor(td.value, B, 0)
        rows = []
        for k, (b, iw) in enumerate(zip(data, isw)):
            wt.copy_(iw)
            flags = 8 | 2 | ((1 | 4) if k == 1 else 0)
            buf = (C.c_float * 12)()
            check(lib.gcrl_sac_update_batch(ag._h, B, *(vp(t.data_ptr()) for t in b[:5]), vp(b[5].data_ptr()),
                                            vp(b[6].data_ptr()), 1e-3, 1e-3, flags, C.cast(buf, vp), st))
            torch.cuda.synchronize()
            rows.append((np.array(list(buf)), tdt.cpu().numpy().copy()))
        out[p] = (rows, ag)
    for (m0, td0), (m2, td2) in zip(out[0][0], out[2][0]):
        np.testing.assert_allclose(m2, m0, rtol=ENG * 2e-5, atol=ENG * 1e-6)
        np.testing.assert_allclose(td2, td0, rtol=ENG * 2e-5, atol=ENG * 1e-6)
    _assert_close_to(out[2][1], *_state(out[0][1]), 1e-3, 2)


# ---- 7. invalid precision -------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", [-1, 3])
def test_invalid_precision_is_rejected(precision):
    from gcrl_b200 import SACAgent
    with pytest.raises(ValueError, match="precision must be"):
        SACAgent(22, 3, T.sac_config(batch_size=64), None, 1, 2, precision=precision)

"""GPU: the loss kernels of TQC's quantile critics (csrc/sac.cu quantile_target_kernel<KPL>, quantile_huber_kernel,
quantile_metrics_kernel) against a float64 restatement of the loss, through gcrl_quantile_critic_loss: the launch
sequence a TQC update issues, on buffers the test fills.

The cases sit where the kernels branch: every sort width (KPL 1, 2, 4, 8 for n M up to 32, 64, 128, 256) at both
ends of its band, the truncation (d = 0, 2, M - 1), tied, widely spread and grid-valued keys (u = 0 and |u| = 1
exactly), the Huber kernel's last partial block (B = rows - 1, rows, rows + 1 with M not dividing 256), the target
kernel's second grid-stride pass (B = 64 x SMs + 1), importance weights with zeros and a coefficient read from a
device scalar.  Every output buffer starts as NaN; a guard row past B, the padding of y and dZ and the gaps between
critics must stay NaN.  The padding and gaps of the inputs, and the element past B of every row vector, hold -1e30:
read, it would sort first into y or swamp a sum.

Bounds, u = 2^-24 the unit roundoff of fp32; each is the worst case of the kernel's own rounding steps, taken per
element so that one wrong term shows:
  * sort: y equals the sorted, truncated pool bit for bit when gamma = 1, r = d = 0 and coef = 0;
  * y: |y - y64| <= 4 u S, S = |r| + g (|z| + |coef logp|), g = gamma (1 - d) (d in {0, 1}): the rounding of
    coef logp, of the subtraction, of the product and of the sum, each at most u S;
  * dZ: u |w| ((K + 6) sum_j wt_j |c_j| + sum_j |c_j|) / (B M K), c = clamp(u, -1, 1), wt = |tau - 1{u < 0}|: u - z
    and the K fused multiply-adds (K + 1), the weight, the two products of the denominator and the division (4),
    one spare; the second sum is tau's rounding, at most u in absolute terms in either weight (1 - tau near the top
    atom has a relative error of up to M u, so a relative bound there would be wrong);
  * loss of critic i: u ((K + 26 + ceil(nblk / 1024)) sum |w| wt h + sum |w| h) / (B M K): h (3), the K fused
    multiply-adds, the weight (1), the block's 8-level tree, the serial pass and 10-level tree of the metrics kernel,
    the count and the division (3), one spare; the second sum is tau's again;
  * TD of critic i and row b: u ((M + 1) mean |z| + (K + 1) mean |y| + td), the two serial means and the difference;
    the row's max over critics moves by at most the largest of those; the batch mean adds
    (ceil(B / 1024) + 11) u mean td for its serial pass, tree and division.
The largest error of each output, as a fraction of its bound, is printed."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -24
PAD = np.float32(-1e30)

# (n, M): n M = 1, 32 | 33, 64 | 65, 128 | 129, 255, 256, 256 -- both ends of every sort width's band
WIDTHS = [(1, 1), (1, 32), (1, 33), (8, 8), (5, 13), (1, 128), (3, 43), (5, 51), (8, 32), (1, 256)]
KEYS = ["normal", "ties", "spread", "grid"]


def pad4(x):
    return (x + 3) // 4 * 4


def drops(M):
    return sorted({0, min(2, M - 1), M - 1})


def kpl(n, M):
    t = n * M
    return 1 if t <= 32 else 2 if t <= 64 else 4 if t <= 128 else 8


# ---- the call --------------------------------------------------------------------------------------------------
def run_loss(zt, z, logp, r, d, w, gamma, coef, drop, alpha=None, ldm=None, gap=0, ldy=None, td_rows=True):
    """gcrl_quantile_critic_loss on zt, z [n, B, M] laid out [n][B][ldm] with gap floats between critics ->
    (y [B, K], dz [n, B, M], out [n + 1], td_rows [B] or None), after checking that nothing outside them was
    written."""
    import torch
    from gcrl_b200._lib import check, lib, vp
    n, B, M = z.shape
    K = n * (M - drop)
    ldm = ldm or pad4(M)
    ldy = ldy or pad4(K)
    zstride = B * ldm + gap
    nblk = -(-B // max(1, 256 // M))

    def atoms(a):
        buf = np.full((n, zstride), PAD, np.float32)
        for i in range(n):
            buf[i, :B * ldm].reshape(B, ldm)[:, :M] = a[i]
        return torch.from_numpy(buf).cuda()

    def rowvec(v):
        return None if v is None else torch.from_numpy(np.append(np.asarray(v, np.float32), PAD)).cuda()

    nan = float("nan")
    zt_d, z_d = atoms(zt), atoms(z)
    logp_d, r_d, d_d, w_d = rowvec(logp), rowvec(r), rowvec(d), rowvec(w)
    alpha_d = None if alpha is None else torch.tensor([alpha], dtype=torch.float32, device="cuda")
    y = torch.full((B + 1, ldy), nan, device="cuda")
    dz = torch.full((n * zstride + ldm,), nan, device="cuda")
    out = torch.full((n + 2,), nan, device="cuda")
    td = torch.full((B + 1,), nan, device="cuda")
    scratch = torch.full((n * (B + nblk),), nan, device="cuda")

    def p(t):
        return None if t is None else vp(t.data_ptr())
    check(lib.gcrl_quantile_critic_loss(0, n, M, drop, B, p(zt_d), p(z_d), ldm, zstride, p(logp_d), p(r_d), p(d_d),
                                        p(w_d), float(gamma), float(coef), p(alpha_d), p(y), ldy, p(dz), p(out),
                                        p(td) if td_rows else None, p(scratch),
                                        vp(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    y, dz, out, td = (t.cpu().numpy() for t in (y, dz, out, td))
    assert np.isnan(y[:B, K:]).all() and np.isnan(y[B]).all(), "y written outside [B, K]"
    dzc = dz[:n * zstride].reshape(n, zstride)
    assert np.isnan(dzc[:, B * ldm:]).all() and np.isnan(dz[n * zstride:]).all(), "dZ written past a critic's rows"
    dzm = dzc[:, :B * ldm].reshape(n, B, ldm)
    assert np.isnan(dzm[:, :, M:]).all(), "dZ written into row padding"
    assert np.isnan(out[n + 1]) and np.isnan(td[B]), "out / td_rows written past their ends"
    if not td_rows:
        assert np.isnan(td).all()
    return y[:B, :K], dzm[:, :, :M], out[:n + 1], td[:B] if td_rows else None


# ---- the float64 restatement -----------------------------------------------------------------------------------
def ref_targets(zt, logp, r, d, gamma, coef, drop):
    """(sorted, truncated pool [B, K] in fp32, y [B, K] in float64, its bound)"""
    n, B, M = zt.shape
    pool = np.sort(zt.transpose(1, 0, 2).reshape(B, n * M), axis=1)[:, :n * (M - drop)]
    p64 = pool.astype(np.float64)
    ent = (float(np.float32(coef)) * np.asarray(logp, np.float64))[:, None]
    disc = (float(np.float32(gamma)) * (1.0 - np.asarray(d, np.float64)))[:, None]
    r64 = np.asarray(r, np.float64)[:, None]
    y = r64 + disc * (p64 - ent)
    bound = 4.0 * EPS * (np.abs(r64) + np.abs(disc) * (np.abs(p64) + np.abs(ent)))
    return pool, y, bound


def ref_loss(z, y, w, drop):
    """Loss, dZ and TD of the critics' atoms z [n, B, M] against the kernel's own targets y [B, K] (fp32), in
    float64, with the bounds of the module docstring."""
    n, B, M = z.shape
    K = n * (M - drop)
    count = float(B) * M * K
    nblk = -(-B // max(1, 256 // M))
    tau = ((np.arange(M) + 0.5) / M)[None, :, None]
    yy = np.asarray(y, np.float64)
    ww = np.ones(B) if w is None else np.asarray(w, np.float64)
    dz, dzb = np.zeros((n, B, M)), np.zeros((n, B, M))
    loss, lossa, lossh = np.zeros(n), np.zeros(n), np.zeros(n)
    td, tdb = np.zeros((n, B)), np.zeros((n, B))
    chunk = max(1, int(4e6 // (M * K)))
    for i in range(n):
        zi = np.asarray(z[i], np.float64)
        for b0 in range(0, B, chunk):
            b1 = min(B, b0 + chunk)
            u = yy[b0:b1, None, :] - zi[b0:b1, :, None]              # [b, M, K], exact
            wt = np.where(u < 0, 1.0 - tau, tau)
            c = np.clip(u, -1.0, 1.0)
            au = np.abs(u)
            h = np.where(au > 1.0, au - 0.5, 0.5 * u * u)
            wb = ww[b0:b1, None]
            dz[i, b0:b1] = -wb * (wt * c).sum(-1) / count
            dzb[i, b0:b1] = EPS * np.abs(wb) * ((K + 6) * (wt * np.abs(c)).sum(-1) + np.abs(c).sum(-1)) / count
            lw = (wt * h).sum(-1) * wb
            loss[i] += lw.sum()
            lossa[i] += np.abs(lw).sum()
            lossh[i] += (h.sum(-1) * np.abs(wb)).sum()
        td[i] = np.abs(zi.mean(1) - yy.mean(1))
        tdb[i] = EPS * ((M + 1) * np.abs(zi).mean(1) + (K + 1) * np.abs(yy).mean(1) + td[i])
    lossb = EPS * ((K + 26 + math.ceil(nblk / 1024)) * lossa + lossh) / count
    rows, rowsb = td.max(0), tdb.max(0)
    mean = rows.mean()
    meanb = rowsb.mean() + EPS * (math.ceil(B / 1024) + 11) * mean
    return dict(dz=(dz, dzb), loss=(loss / count, lossb), td_rows=(rows, rowsb), td=(np.array([mean]),
                                                                                    np.array([meanb])))


def within(name, got, want, bound, errs):
    got = np.asarray(got, np.float64)
    assert np.isfinite(got).all(), f"{name}: non-finite output"
    err = np.abs(got - want)
    frac = np.where(bound > 0, err / np.where(bound > 0, bound, 1.0), np.where(err > 0, np.inf, 0.0))
    errs[name] = (float(err.max()), float(frac.max()))
    bad = np.argwhere(frac > 1.0)
    assert bad.size == 0, (f"{name}: {bad.shape[0]} elements outside the bound, first at {tuple(bad[0])}: "
                           f"got {got[tuple(bad[0])]!r}, want {want[tuple(bad[0])]!r} +- {bound[tuple(bad[0])]!r}")


def check_loss(z, y, w, drop, out, dz, td_rows, errs):
    n = z.shape[0]
    ref = ref_loss(z, y, w, drop)
    within("dz", dz, *ref["dz"], errs)
    within("loss", out[:n], *ref["loss"], errs)
    within("td", out[n:], *ref["td"], errs)
    if td_rows is not None:
        within("td_rows", td_rows, *ref["td_rows"], errs)


def report(tag, errs, capsys):
    with capsys.disabled():
        print(f"\n[quantile loss] {tag}: largest error (fraction of bound) " +
              ", ".join(f"{k} {e:.2e} ({f:.3f})" for k, (e, f) in errs.items()))


# ---- inputs ----------------------------------------------------------------------------------------------------
def keys(rng, kind, n, B, M):
    """(zt, z) [n, B, M] fp32"""
    shape = (n, B, M)
    if kind == "normal":
        zt, z = rng.standard_normal(shape), rng.standard_normal(shape)
    elif kind == "ties":        # rounded to 0.5 and the same in every critic: long runs of equal keys, u = 0
        zt = np.broadcast_to(np.round(2.0 * rng.standard_normal((1, B, M))) / 2.0, shape).copy()
        z = np.round(2.0 * rng.standard_normal(shape)) / 2.0
    elif kind == "spread":      # magnitudes 1e-6 .. 1e6, both signs, some -0 and +0
        zt = rng.choice([-1.0, 1.0], shape) * 10.0 ** rng.uniform(-6, 6, shape)
        z = rng.choice([-1.0, 1.0], shape) * 10.0 ** rng.uniform(-6, 6, shape)
        zt.flat[::7] = 0.0
        zt.flat[3::11] = -0.0
    else:                       # "grid": the atoms are the target keys, some moved by exactly +-1 or +-0.5
        zt = rng.integers(-4, 5, shape) * 0.5
        z = zt + rng.choice([-1.0, -0.5, 0.0, 0.0, 1.0], shape)
    return zt.astype(np.float32), z.astype(np.float32)


def rows(rng, B, weights):
    logp = rng.standard_normal(B).astype(np.float32)
    r = -(rng.random(B) > 0.3).astype(np.float32) + 0.1 * rng.standard_normal(B).astype(np.float32)
    d = (rng.random(B) < 0.1).astype(np.float32)
    w = None
    if weights:
        w = rng.uniform(0.0, 2.0, B).astype(np.float32)
        w[rng.random(B) < 0.15] = 0.0
    return logp, r.astype(np.float32), d, w


# ---- 1. the sort, bit for bit, and the loss on its targets --------------------------------------------------------
SORT_CASES = [(n, M, dr, k) for n, M in WIDTHS for dr in drops(M) for k in KEYS]


@pytest.mark.parametrize("n,M,drop,kind", SORT_CASES,
                         ids=[f"n{n}_M{M}_d{dr}_{k}_kpl{kpl(n, M)}" for n, M, dr, k in SORT_CASES])
def test_sort_is_exact_and_loss_matches_float64(n, M, drop, kind, capsys):
    """gamma = 1, r = d = 0, coef = 0: y is the pooled atoms sorted ascending and truncated to K = n (M - drop), bit
    for bit (+0 and -0 compare equal); dZ, the per-critic losses, the TD rows and their mean on those targets within
    their bounds.  Grid keys make u = 0 and |u| = 1 occur exactly (the branch points of the weight and of Huber)."""
    B = 77
    rng = np.random.default_rng(1000 * n + 10 * M + drop + KEYS.index(kind))
    zt, z = keys(rng, kind, n, B, M)
    zero = np.zeros(B, np.float32)
    logp = rng.standard_normal(B).astype(np.float32)
    y, dz, out, td_rows = run_loss(zt, z, logp, zero, zero, None, 1.0, 0.0, drop)
    pool, _, _ = ref_targets(zt, logp, zero, zero, 1.0, 0.0, drop)
    assert np.array_equal(y, pool), np.argwhere(y != pool)[:5]
    errs = {}
    check_loss(z, y, None, drop, out, dz, td_rows, errs)
    report(f"sort n={n} M={M} d={drop} {kind}", errs, capsys)


# ---- 2. general targets: rewards, done rows, entropy term, importance weights ---------------------------------------
GEN_CASES = [(n, M, dr, mode) for n, M in WIDTHS for dr in sorted({min(2, M - 1), M - 1}) for mode in (0, 1)]


@pytest.mark.parametrize("n,M,drop,mode", GEN_CASES,
                         ids=[f"n{n}_M{M}_d{dr}_{'coef-w' if mode else 'const'}" for n, M, dr, mode in GEN_CASES])
def test_targets_and_loss_match_float64(n, M, drop, mode, capsys):
    """gamma 0.98, rewards, 10 % done rows.  mode 0: constant coefficient, no weights, no TD rows, the agent's layout;
    mode 1:
    coefficient from a device scalar, importance weights with zeros, the TD rows, wider ldm and ldy and a gap between
    critics."""
    B = 123
    rng = np.random.default_rng(7 + 1000 * n + 10 * M + drop + mode)
    zt, z = keys(rng, "normal", n, B, M)
    logp, r, d, w = rows(rng, B, weights=mode == 1)
    coef, alpha = (0.2, None) if mode == 0 else (-1.0, 0.37)
    lay = {} if mode == 0 else dict(ldm=pad4(M) + 4, gap=13, ldy=pad4(n * (M - drop)) + 8)
    y, dz, out, td_rows = run_loss(zt, z, logp, r, d, w, 0.98, coef, drop, alpha=alpha, td_rows=mode == 1, **lay)
    _, want, bound = ref_targets(zt, logp, r, d, 0.98, alpha if coef < 0 else coef, drop)
    errs = {}
    within("y", y, want, bound, errs)
    check_loss(z, y, w, drop, out, dz, td_rows, errs)
    report(f"general n={n} M={M} d={drop} mode {mode}", errs, capsys)


# ---- 3. batch edges ----------------------------------------------------------------------------------------------
def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# (n, M, drop, B): B = 1; around the Huber kernel's rows = 256 // M when M does not divide 256 (M = 51: 5 rows,
# M = 7: 36 rows); 64 x SMs + 1 rows, one more than the warps of the capped grid of the target kernel, at every sort
# width ("wrap"); 32768 rows, the agent's largest batch, at small n M
EDGE_CASES = ([(5, 51, 2, 1), (1, 1, 0, 1), (8, 32, 0, 1)] +
              [(5, 51, 2, b) for b in (4, 5, 6, 11)] + [(4, 7, 2, b) for b in (35, 36, 37)] +
              [(2, 16, 0, "wrap"), (4, 12, 2, "wrap"), (5, 13, 2, "wrap"), (8, 32, 31, "wrap"), (1, 256, 255, "wrap")] +
              [(1, 1, 0, 32768), (2, 8, 1, 32768)])


@pytest.mark.parametrize("n,M,drop,B", EDGE_CASES,
                         ids=[f"n{n}_M{M}_d{dr}_B{b}_kpl{kpl(n, M)}" for n, M, dr, b in EDGE_CASES])
def test_batch_edges_match_float64(n, M, drop, B, capsys):
    """Every row of y, dZ and the TD rows present and right at the batch sizes where the grids end; odd cases with
    the coefficient from a device scalar and importance weights."""
    if B == "wrap":
        B = 64 * _sms() + 1
    mode = (n + M + B) % 2
    rng = np.random.default_rng(n * 7919 + M * 104729 + B)
    zt, z = keys(rng, "normal", n, B, M)
    logp, r, d, w = rows(rng, B, weights=mode == 1)
    coef, alpha = (0.2, None) if mode == 0 else (-1.0, 0.37)
    y, dz, out, td_rows = run_loss(zt, z, logp, r, d, w, 0.98, coef, drop, alpha=alpha)
    _, want, bound = ref_targets(zt, logp, r, d, 0.98, alpha if coef < 0 else coef, drop)
    errs = {}
    within("y", y, want, bound, errs)
    check_loss(z, y, w, drop, out, dz, td_rows, errs)
    report(f"edge n={n} M={M} d={drop} B={B}", errs, capsys)


# ---- 4. which kernels run ----------------------------------------------------------------------------------------
def test_every_sort_width_runs():
    """n M = 32, 64, 128, 256 launch quantile_target_kernel<1>, <2>, <4>, <8>, each with the Huber and metrics
    kernels behind it."""
    import re

    import torch
    from torch.profiler import ProfilerActivity, profile
    seen = set()
    for n, M in ((1, 32), (8, 8), (1, 128), (8, 32)):
        rng = np.random.default_rng(M)
        zt, z = keys(rng, "normal", n, 64, M)
        logp, r, d, _ = rows(rng, 64, False)
        run_loss(zt, z, logp, r, d, None, 0.98, 0.2, 1)      # warm
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run_loss(zt, z, logp, r, d, None, 0.98, 0.2, 1)
            torch.cuda.synchronize()
        names = [e.name for e in prof.events()]
        got = {int(m.group(1)) for nm in names for m in [re.search(r"quantile_target_kernel<(\d+)>", nm)] if m}
        assert got == {kpl(n, M)}, (n, M, sorted(set(names)))
        for k in ("quantile_huber_kernel", "quantile_metrics_kernel"):
            assert any(k in nm for nm in names), (k, sorted(set(names)))
        seen |= got
    assert seen == {1, 2, 4, 8}

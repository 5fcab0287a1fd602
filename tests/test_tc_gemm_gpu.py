"""GPU numerics: the two dense-layer engines -- the tcgen05 kernel (csrc/tc_gemm.cu, 3xTF32 split) and the fp32
FFMA tiles (csrc/mlp.cu) -- against a float64 reference of nn.Linear + LeakyReLU (src/model.py:17-30), of its input
gradient and of its weight gradient.  Tolerance: max-norm relative error <= 1e-5 on tcgen05 (observed 2e-6) and
<= 2e-6 on the fp32 tiles (observed ~5e-7); the observed errors are printed."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOL = {0: 2e-6, 1: 1e-5}          # engine 0: fp32 FFMA tiles; engine 1: tcgen05


def _run(engine, mode, x, w, b, act):
    """y = gcrl_dense_layer(x, w); y is written into rows padded to a multiple of 4 floats, whose padding must stay
    untouched (NaN)."""
    import torch
    from gcrl_b200._lib import check, lib, vp
    M, K = x.shape
    N = w.shape[0]
    y = torch.full((M, (N + 3) // 4 * 4), float("nan"), device="cuda")
    check(lib.gcrl_dense_layer(0, engine, mode, M, N, K, vp(x.data_ptr()), x.stride(0), vp(w.data_ptr()), w.stride(0),
                               None if b is None else vp(b.data_ptr()), None if act is None else vp(act.data_ptr()),
                               0 if act is None else act.stride(0), vp(y.data_ptr()), y.stride(0),
                               vp(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    assert bool(torch.isnan(y[:, N:]).all())
    return y[:, :N]


# launch_gemm (mlp.cu) picks its tile from the tile count on 148 SMs: 128 x 128 when those tiles alone reach the SM
# count, 64 x 64 above half of it, 32 x 32 below.  Its K loop runs in steps of BK = 16.
DENSE_SHAPES = [(128, 256, 256), (1, 64, 64), (1000, 256, 256), (65536, 256, 256), (300, 64, 64), (4096, 512, 512),
                (777, 96, 100), (5000, 256, 24), (129, 16, 4)]
# the tiles alone take N % 16 != 0 and K % 4 != 0 (rows padded to a multiple of 4 floats)
TILE_SHAPES = [(70000, 30, 27),          # 128 x 128, ragged M and N, K tail 11 in a padded row
               (4097, 130, 64),          # 64 x 64, N % 4 == 2
               (1, 7, 5),                # 32 x 32, M = 1
               (333, 61, 19)]            # 32 x 32, K tail 3


@pytest.mark.parametrize("engine,M,N,K", [pytest.param(1, *s, id="-".join(map(str, s))) for s in DENSE_SHAPES] +
                         [pytest.param(0, *s, id="tiles-" + "-".join(map(str, s))) for s in DENSE_SHAPES + TILE_SHAPES])
def test_tc_dense_matches_float64(engine, M, N, K, capsys):
    """Modes 0 (bias + LeakyReLU) and 2 (bias) on both engines, mode 1 (times LeakyReLU'(act)) on tcgen05, which alone
    implements it.  Operand rows are padded to a multiple of 4 floats with random values the kernels must not read."""
    import torch
    torch.manual_seed(M + N + K)
    ldk = (K + 3) // 4 * 4
    x = torch.randn(M, ldk, device="cuda")[:, :K]
    w = (torch.randn(N, ldk, device="cuda") / K ** 0.5)[:, :K]
    b = torch.randn(N, device="cuda")
    act = torch.randn(M, N, device="cuda")
    ref = x.double() @ w.double().T
    wants = {0: torch.nn.functional.leaky_relu(ref + b.double(), 0.01),
             1: ref * torch.where(act > 0, 1.0, 0.01).double(),
             2: ref + b.double()}
    errs = {}
    for mode, want in wants.items():
        if engine == 0 and mode == 1:
            continue
        got = _run(engine, mode, x, w, b if mode != 1 else None, act if mode == 1 else None)
        assert torch.isfinite(got).all()
        errs[mode] = ((got.double() - want).abs().max() / want.abs().max()).item()
    with capsys.disabled():
        print(f"\n[dense] engine {engine} M={M} N={N} K={K}: max-norm rel err " +
              ", ".join(f"mode {m} {e:.1e}" for m, e in errs.items()) + f" (allowed {TOL[engine]:.0e})")
    assert all(e <= TOL[engine] for e in errs.values()), errs


def test_tc_dense_strided_operands_and_zero_padding():
    """Leading dimensions larger than the logical widths (the agent's padded rows)."""
    import torch
    torch.manual_seed(3)
    M, N, K = 2048, 64, 24
    xs = torch.randn(M, 28, device="cuda")
    ws = torch.randn(N, 28, device="cuda")
    b = torch.randn(N, device="cuda")
    ys = torch.zeros(M, 80, device="cuda")
    from gcrl_b200._lib import check, lib, vp
    check(lib.gcrl_dense_layer(0, 1, 2, M, N, K, vp(xs.data_ptr()), 28, vp(ws.data_ptr()), 28, vp(b.data_ptr()), None, 0,
                               vp(ys.data_ptr()), 80, vp(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    want = xs[:, :K].double() @ ws[:, :K].double().T + b.double()
    assert ((ys[:, :N].double() - want).abs().max() / want.abs().max()).item() <= 1e-5
    assert float(ys[:, N:].abs().max()) == 0.0          # columns beyond N untouched


WGRAD_SHAPES = [(1024, 128, 32), (4096, 256, 256), (5000, 64, 64), (3000, 256, 24), (8192, 512, 512), (777, 96, 100),
                (2048, 4, 64), (16, 256, 256), (65536, 256, 256)]
# launch_linear_wgrad splits the batch into at most max_splits slabs of >= 64 rows and picks its tile like launch_gemm
# (tiles x slabs against 148 SMs).  Every slab is one sequential fp32 sum, whose error grows with its rows: these keep
# a slab at <= 2048 rows even at max_splits = 1.
TILE_WGRAD_SHAPES = [(1024, 128, 32), (777, 96, 100), (2048, 4, 64), (16, 256, 256),   # 32 x 32 (except below)
                     (1000, 30, 27), (300, 7, 5),           # N % 4 != 0, K % 4 != 0
                     (1500, 512, 512),                      # 64 x 64 at max_splits 3 and 128
                     (1200, 1030, 1030)]                    # 64 x 64 at max_splits 1, else 128 x 128


@pytest.mark.parametrize("engine,M,N,K,max_splits",
                         [pytest.param(1, *s, 128, id="-".join(map(str, s))) for s in WGRAD_SHAPES] +
                         [pytest.param(0, *s, ms, id="tiles-" + "-".join(map(str, s)) + f"-splits{ms}")
                          for s in TILE_WGRAD_SHAPES for ms in (1, 3, 128)])
def test_tc_wgrad_matches_float64(engine, M, N, K, max_splits, capsys):
    """Weight gradient as split-batch partial slabs: tcgen05 (MN-major operands, 32-byte-atom swizzle) and the fp32
    tiles (launch_linear_wgrad).  The summed slabs against dZ^T X in float64, and the row padding of every slab
    (columns K to ldw, which reaches 4 floats past K padded to a multiple of 4) exactly zero.  Tolerance: max-norm
    relative 1e-5 on tcgen05 (observed 1e-7 .. 7e-6, growing with the rows accumulated per TMEM tile), 2e-6 on the
    tiles."""
    import ctypes as C
    import torch
    from gcrl_b200._lib import check, lib, vp
    torch.manual_seed(M + N + K)
    lddz, ldx = (N + 3) // 4 * 4, (K + 3) // 4 * 4
    dz = (torch.randn(M, lddz, device="cuda") / M ** 0.5)[:, :N]
    x = torch.randn(M, ldx, device="cuda")[:, :K]
    ldw = ldx + 4
    stride = N * ldw + 8
    pw = torch.full((max_splits, stride), float("nan"), device="cuda")
    pb = torch.full((max_splits, N + 4), float("nan"), device="cuda")
    sp = C.c_int()
    check(lib.gcrl_dense_wgrad(0, engine, M, N, K, vp(dz.data_ptr()), lddz, vp(x.data_ptr()), ldx, vp(pw.data_ptr()), ldw,
                               stride, vp(pb.data_ptr()), N + 4, max_splits, C.byref(sp),
                               vp(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    S = sp.value
    assert 1 <= S <= max_splits
    slabs = pw[:S, :N * ldw].double().reshape(S, N, ldw)
    assert float(slabs[:, :, K:].abs().max()) == 0.0
    W = slabs.sum(0)
    want = dz.double().T @ x.double()
    err_w = ((W[:, :K] - want).abs().max() / want.abs().max()).item()
    wb = dz.double().sum(0)
    err_b = ((pb[:S, :N].double().sum(0) - wb).abs().max() / wb.abs().max()).item()
    with capsys.disabled():
        print(f"\n[wgrad] engine {engine} M={M} N={N} K={K} max_splits={max_splits}: {S} slabs, max-norm rel err "
              f"weights {err_w:.1e}, bias {err_b:.1e} (allowed {TOL[engine]:.0e})")
    assert err_w <= TOL[engine] and err_b <= TOL[engine], (err_w, err_b)


@pytest.mark.parametrize("call,operand", [("dense", "x"), ("dense", "w"), ("dense", "y"),
                                          ("wgrad", "dz"), ("wgrad", "x"), ("wgrad", "w")])
def test_tiles_refuse_leading_dimensions_not_multiple_of_4(call, operand):
    """The fp32 tiles load and store float4 at base + row * ld + column, so a leading dimension that is not a
    multiple of 4 floats would make misaligned accesses: engine 0 refuses it with GCRL_ERR_INVALID, as tcgen05 does,
    and writes nothing."""
    import ctypes as C
    import torch
    from gcrl_b200._lib import ERR_INVALID, lib, vp
    M, N, K = 16, 6, 6
    ld = {name: 6 if name == operand else 8 for name in ("x", "w", "y", "dz")}
    st = vp(torch.cuda.current_stream().cuda_stream)
    x = torch.randn(M, ld["x"], device="cuda")
    if call == "dense":
        w = torch.randn(N, ld["w"], device="cuda")
        b = torch.randn(N, device="cuda")
        out = torch.full((M, ld["y"]), float("nan"), device="cuda")
        rc = lib.gcrl_dense_layer(0, 0, 0, M, N, K, vp(x.data_ptr()), ld["x"], vp(w.data_ptr()), ld["w"], vp(b.data_ptr()),
                                  None, 0, vp(out.data_ptr()), ld["y"], st)
    else:
        dz = torch.randn(M, ld["dz"], device="cuda")
        out = torch.full((2, N * ld["w"] + 8), float("nan"), device="cuda")
        pb = torch.full((2, 8), float("nan"), device="cuda")
        sp = C.c_int()
        rc = lib.gcrl_dense_wgrad(0, 0, M, N, K, vp(dz.data_ptr()), ld["dz"], vp(x.data_ptr()), ld["x"], vp(out.data_ptr()),
                                  ld["w"], N * ld["w"] + 8, vp(pb.data_ptr()), 8, 2, C.byref(sp), st)
    torch.cuda.synchronize()
    assert rc == ERR_INVALID, (rc, lib.gcrl_last_error())
    assert bool(torch.isnan(out).all())


@pytest.mark.parametrize("M,N,K", [(65536, 256, 256), (16384, 256, 256), (20000, 256, 256), (16385, 256, 256),
                                   (30000, 512, 512), (14500, 256, 24), (1000, 256, 256), (4096, 512, 512),
                                   (8192, 256, 256), (8000, 256, 32)])
def test_tc_dense_presplit_weights_match_float64(M, N, K):
    """The agent's large-batch path: weights pre-split into TF32 hi / lo halves (gcrl_split_tf32), activations split
    in the kernel.  Large M with N % 256 == 0 runs on CTA pairs (cta_group::2: 256 x 256 tiles, every SM stages half
    of the weight tile; a partly filled last round as two 256 x 128 halves per tile),
    the rest on the single-CTA kernel; same tolerance as the un-split entry point (1e-5 max-norm
    relative), ragged row tails and both N tiles covered."""
    import torch
    from gcrl_b200._lib import check, lib, vp
    torch.manual_seed(M + N + K)
    x = torch.randn(M, K, device="cuda")
    w = torch.randn(N, K, device="cuda") / K ** 0.5
    b = torch.randn(N, device="cuda")
    act = torch.randn(M, N, device="cuda")
    hi, lo = torch.empty_like(w), torch.empty_like(w)
    st = vp(torch.cuda.current_stream().cuda_stream)
    check(lib.gcrl_split_tf32(0, vp(w.data_ptr()), vp(hi.data_ptr()), vp(lo.data_ptr()), w.numel(), st))
    assert torch.equal((hi.double() + lo.double()).float(), w) or float((hi + lo - w).abs().max()) <= 2e-7 * float(w.abs().max())
    ref = x.double() @ w.double().T
    wants = {0: torch.nn.functional.leaky_relu(ref + b.double(), 0.01),
             1: ref * torch.where(act > 0, 1.0, 0.01).double(),
             2: ref + b.double()}
    for mode, want in wants.items():
        y = torch.full((M, N), float("nan"), device="cuda")
        check(lib.gcrl_dense_layer_presplit(0, mode, M, N, K, vp(x.data_ptr()), K, vp(hi.data_ptr()), vp(lo.data_ptr()), K,
                                            vp(b.data_ptr()) if mode != 1 else None,
                                            vp(act.data_ptr()) if mode == 1 else None, N if mode == 1 else 0,
                                            vp(y.data_ptr()), N, st))
        torch.cuda.synchronize()
        assert torch.isfinite(y).all(), mode
        err = ((y.double() - want).abs().max() / want.abs().max()).item()
        assert err <= 1e-5, (mode, err)


def test_tc_kernels_ignore_removed_timing_variables(monkeypatch):
    """The tcgen05 dense and weight-gradient launches have no environment switches: variables that once forced kernel
    variants or skipped work for timing experiments change no output bit.  A CTA-pair shape with a partly filled last
    round (half tiles) and a weight gradient with bias sums and in-place slab accumulation (M = 65 536)."""
    import ctypes as C
    import torch
    from gcrl_b200._lib import check, lib, vp
    removed = {"GCRL_TC_DBG": "7", "GCRL_TC_BN": "64", "GCRL_TC_PAIR_RT": "0", "GCRL_TC_NO_HALVES": "1",
               "GCRL_TC_NO_FUSED_COLSUM": "1", "GCRL_TC_NO_SLAB_ACC": "1"}
    torch.manual_seed(11)
    st = vp(torch.cuda.current_stream().cuda_stream)
    M, N, K = 20000, 256, 256
    x = torch.randn(M, K, device="cuda")
    w = torch.randn(N, K, device="cuda") / K ** 0.5
    b = torch.randn(N, device="cuda")
    hi, lo = torch.empty_like(w), torch.empty_like(w)
    check(lib.gcrl_split_tf32(0, vp(w.data_ptr()), vp(hi.data_ptr()), vp(lo.data_ptr()), w.numel(), st))
    Mw = 65536
    dz = torch.randn(Mw, N, device="cuda") / Mw ** 0.5
    xw = torch.randn(Mw, K, device="cuda")
    stride, max_splits = N * K + 8, 128

    def run():
        y = torch.full((M, N), float("nan"), device="cuda")           # fresh outputs: a skipped store stays NaN
        check(lib.gcrl_dense_layer_presplit(0, 0, M, N, K, vp(x.data_ptr()), K, vp(hi.data_ptr()), vp(lo.data_ptr()), K,
                                            vp(b.data_ptr()), None, 0, vp(y.data_ptr()), N, st))
        pw = torch.full((max_splits, stride), float("nan"), device="cuda")
        pb = torch.full((max_splits, N), float("nan"), device="cuda")
        sp = C.c_int()
        check(lib.gcrl_dense_wgrad(0, 1, Mw, N, K, vp(dz.data_ptr()), N, vp(xw.data_ptr()), K, vp(pw.data_ptr()), K,
                                   stride, vp(pb.data_ptr()), N, max_splits, C.byref(sp), st))
        torch.cuda.synchronize()
        S = sp.value
        return y, S, pw[:S, :N * K], pb[:S]

    for name in removed:
        monkeypatch.delenv(name, raising=False)
    y0, s0, pw0, pb0 = run()
    assert torch.isfinite(y0).all() and torch.isfinite(pw0).all() and torch.isfinite(pb0).all()
    for name, value in removed.items():
        monkeypatch.setenv(name, value)
    y1, s1, pw1, pb1 = run()
    assert torch.equal(y1, y0)
    assert s1 == s0 and torch.equal(pw1, pw0) and torch.equal(pb1, pb0)

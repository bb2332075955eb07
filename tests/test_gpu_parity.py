"""Parity tests proper: the CUDA path (through the C-ABI) against the CPU oracle, the golden vectors
produced by the unmodified reference, and size-independent properties at BASELINE sizes.

Tolerances (stated once):
  * CUDA-core Gram (fp64 accumulation of exact products): S within 1e-12 relative of the fp64 oracle.
  * tcgen05 Gram (bf16 hi/lo operands, fp32 TMEM accumulation drained every 8192 rows, fp64 beyond):
    coefficient l_inf error < 1e-4 against the fit of the same rows (BASELINE.json north_star); measured
    values are ~1e-6, asserted at 2e-5 to catch regressions.  intercept_ within 3e-2 (ill-conditioned:
    leverage x_bar * sqrt(D), SURVEY.md H1).
  * metrics: relative 1e-5 (y is staged as fp32).
"""
import io
import os

import numpy as np
import pytest

import bodywork_mlops_demo_b200 as b2
from bodywork_mlops_demo_b200 import stage_1_train_model as s1
from oracle import ols_oracle as orc

pytestmark = pytest.mark.gpu

COEF_TOL = 2e-5      # asserted; the contract is 1e-4
INTERCEPT_TOL = 3e-2   # |d b0| <= sum_j |xbar_j| |d beta_j| ~ D * 50 * coef error (SURVEY.md H1)


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-300))


def _gram(ctx, X, y, kernel, mask=None, keep=1, kind=None):
    ctx.set_kernel(kernel)
    ctx.gram_reset(X.shape[1])
    Xd = ctx.to_device(X, kind) if kind else ctx.to_device(X)
    yd = ctx.to_device(y)
    md = ctx.to_device(mask) if mask is not None else None
    ctx.gram_accumulate(Xd, yd, md, keep)
    S = ctx.gram_export()
    for a in (Xd, yd, md):
        if a is not None:
            a.free()
    ctx.set_kernel(b2.KERNEL_AUTO)
    return S


# ------------------------------------------------------------------------------------------------
# Gram kernels vs the oracle
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d", [(1, 1), (7, 3), (1000, 1), (1440, 1), (5000, 8), (4096, 128), (3001, 37), (333, 128)])
def test_simt_gram_matches_oracle(ctx, n, d):
    X, y = orc.generate_dataset(n, d, seed=n + d, dtype=np.float32)
    S = _gram(ctx, X, y, b2.KERNEL_SIMT)
    assert _rel(S, orc.gram_stats(X, y)) < 1e-12
    assert S[d, d] == n


@pytest.mark.parametrize("n,d", [(64, 128), (4096, 128), (100_003, 128), (50_000, 32), (20_001, 8), (65_536, 64),
                                 (9_999, 4), (40_000, 100),
                                 # packed super-rows with a zero-filled tail: pack = 5, 5, 4, 3, 3, 2, 2
                                 (30_011, 20), (25_000, 24), (40_003, 28), (20_000, 36), (33_333, 40), (45_001, 48),
                                 (10_000, 60)])
def test_tcgen05_gram_matches_oracle(ctx, n, d):
    X, y = orc.generate_dataset(n, d, seed=n + d, dtype=np.float32)
    S = _gram(ctx, X, y, b2.KERNEL_TCGEN05)
    So = orc.gram_stats(X, y)
    assert S[d, d] == n                                    # row count is exact
    assert _rel(S[:d, d], So[:d, d]) < 1e-6                # sum x (CUDA-core side sums, fp32 -> fp64)
    assert _rel(S, So) < 2e-6
    assert np.array_equal(S, S.T)                          # symmetric by construction
    if n > 4 * d:
        ctx.gram_import(S)
        coef, b0 = ctx.solve()
        fo = orc.fit_from_stats(So)
        assert np.max(np.abs(coef - fo["coef"])) < COEF_TOL
        assert abs(b0 - fo["intercept"]) < INTERCEPT_TOL


def test_tcgen05_equals_simt_on_device(ctx):
    X, y = orc.generate_dataset(70_000, 128, seed=77, dtype=np.float32)
    a = _gram(ctx, X, y, b2.KERNEL_TCGEN05)
    b = _gram(ctx, X, y, b2.KERNEL_SIMT)
    assert _rel(a, b) < 2e-6


# ------------------------------------------------------------------------------------------------
# narrow rows (D <= 16): the CUDA-core streaming kernel behind the TMA bulk-copy pipeline
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["f32", "bf16"])
@pytest.mark.parametrize("n,d", [(4096, 1), (50_001, 1), (33_333, 2), (20_000, 3), (70_007, 4), (30_000, 5),
                                 (100_003, 8), (9_000, 9), (25_000, 12), (60_001, 16)])
def test_narrow_gram_matches_oracle(ctx, n, d, kind):
    X, y = orc.generate_dataset(n, d, seed=n + d, dtype=np.float32)
    if kind == "bf16":
        bits = b2.native.to_bf16_bits(X)
        X = b2.native.from_bf16_bits(bits)
        S = _gram(ctx, bits, y, b2.KERNEL_NARROW, kind="bf16")
    else:
        S = _gram(ctx, X, y, b2.KERNEL_NARROW)
    So = orc.gram_stats(X, y)
    assert S[d, d] == n                                    # row count is exact
    assert _rel(S, So) < 1e-6                              # fp32 FMA chains folded into fp64
    assert np.array_equal(S, S.T)
    ctx.gram_import(S)
    coef, b0 = ctx.solve()
    fo = orc.fit_from_stats(So)
    assert np.max(np.abs(coef - fo["coef"])) < COEF_TOL
    assert abs(b0 - fo["intercept"]) < INTERCEPT_TOL


@pytest.mark.parametrize("d,keep", [(1, 1), (8, 1), (8, 0), (16, 1), (11, 0)])
def test_narrow_row_mask_equals_gather(ctx, d, keep):
    X, y = orc.generate_dataset(41_017, d, seed=31 + d, dtype=np.float32)
    mask = s1.split_mask(X.shape[0])
    S = _gram(ctx, X, y, b2.KERNEL_NARROW, mask=mask, keep=keep)
    So = orc.gram_stats(X[mask == keep], y[mask == keep])
    assert S[d, d] == int((mask == keep).sum())
    assert _rel(S, So) < 1e-6


def test_narrow_is_deterministic_additive_and_the_auto_choice(ctx):
    X, y = orc.generate_dataset(120_000, 8, seed=12, dtype=np.float32)
    a = _gram(ctx, X, y, b2.KERNEL_NARROW)
    assert np.array_equal(a, _gram(ctx, X, y, b2.KERNEL_NARROW))
    assert np.array_equal(a, _gram(ctx, X, y, b2.KERNEL_AUTO))       # AUTO takes the narrow kernel for D <= 16
    ctx.set_kernel(b2.KERNEL_NARROW)
    ctx.gram_reset(8)
    for lo, hi in ((0, 50_000), (50_000, 120_000)):
        Xd, yd = ctx.to_device(X[lo:hi]), ctx.to_device(y[lo:hi])
        ctx.gram_accumulate(Xd, yd)
        Xd.free(); yd.free()
    parts = ctx.gram_export()
    ctx.set_kernel(b2.KERNEL_AUTO)
    assert parts[8, 8] == 120_000 and _rel(parts, a) < 1e-7
    assert _rel(a, _gram(ctx, X, y, b2.KERNEL_SIMT)) < 1e-6


def test_narrow_badly_offset_columns_keep_their_digits(ctx):
    """Column means 1e4 times the spread: the per-column shift is what keeps fp32 products usable."""
    rng = np.random.RandomState(4)
    n, d = 200_000, 4
    X = (10_000.0 + rng.normal(0.0, 1.0, size=(n, d))).astype(np.float32)
    y = (3.0 + X.astype(np.float64) @ np.array([0.5, -1.0, 2.0, 0.25]) + rng.normal(0, 0.1, n)).astype(np.float32)
    S = _gram(ctx, X, y, b2.KERNEL_NARROW)
    fo = orc.fit_from_stats(orc.gram_stats(X, y))
    ctx.gram_import(S)
    coef, _ = ctx.solve()
    assert np.max(np.abs(coef - fo["coef"])) < 1e-4


@pytest.mark.parametrize("d", [1, 8, 16])
def test_narrow_large_n_agrees_with_the_other_kernels(ctx, d):
    n = 20_000_000 + 77
    X, y = ctx.synth(n, d, seed=99)
    res = {}
    for kernel in [b2.KERNEL_NARROW] + ([b2.KERNEL_TCGEN05] if d >= 4 else []):   # tcgen05 zero-pads D to 128
        ctx.set_kernel(kernel)
        ctx.gram_reset(d)
        ctx.gram_accumulate(X, y)
        res[kernel] = (ctx.gram_export(), ctx.solve())
    ctx.set_kernel(b2.KERNEL_AUTO)
    S, (coef, b0) = res[b2.KERNEL_NARROW]
    assert S[d, d] == n
    assert np.max(np.abs(coef - 0.5)) < 5e-4 and abs(b0 - 1.0) < 0.05      # the generator's truth (stage_3...:36-41)
    if b2.KERNEL_TCGEN05 in res:
        S2, (coef2, _) = res[b2.KERNEL_TCGEN05]
        assert _rel(S, S2) < 2e-6 and np.max(np.abs(coef - coef2)) < COEF_TOL
    X.free(); y.free()


def _random_case(i):
    rng = np.random.RandomState(1000 + i)
    d = int(rng.choice([1, 2, 3, 4, 5, 7, 8, 12, 16, 20, 32, 33, 48, 64, 96, 100, 128]))
    n = int(rng.choice([1, 2, 63, 64, 65, 1000, 2047, 2048, 4095, 4096, 5000, 9999, 30_000, 70_001]))
    kind = "bf16" if (rng.rand() < 0.3 and d % 8 == 0) else "f32"
    masked = rng.rand() < 0.4
    return n, d, kind, masked


@pytest.mark.parametrize("i", range(48))
def test_randomized_shapes_through_the_auto_dispatch(ctx, i):
    """Whatever kernel AUTO picks (exact fp64 / narrow / tcgen05 / packed), the statistic is the oracle's."""
    n, d, kind, masked = _random_case(i)
    X, y = orc.generate_dataset(n, d, seed=i, dtype=np.float32)
    mask = (np.random.RandomState(i).rand(n) < 0.8).astype(np.uint8) if masked else None
    if kind == "bf16":
        bits = b2.native.to_bf16_bits(X)
        X = b2.native.from_bf16_bits(bits)
        S = _gram(ctx, bits, y, b2.KERNEL_AUTO, mask=mask, keep=1, kind="bf16")
    else:
        S = _gram(ctx, X, y, b2.KERNEL_AUTO, mask=mask, keep=1)
    sel = slice(None) if mask is None else (mask == 1)
    So = orc.gram_stats(X[sel], y[sel])
    assert S[d, d] == So[d, d]
    assert _rel(S, So) < 2e-6
    assert np.array_equal(S, S.T)
    if So[d, d] > 6 * d + 10:
        ctx.gram_import(S)
        coef, b0 = ctx.solve()
        fo = orc.fit_from_stats(So)
        tol = COEF_TOL * max(1.0, 3000.0 / So[d, d]) ** 0.5 * (4 if d > 64 else 1)   # short, wide problems are ill-conditioned
        assert np.max(np.abs(coef - fo["coef"])) < tol


@pytest.mark.parametrize("drain", [64, 1024, 8192, 65536])
def test_drain_interval_does_not_change_the_fit(ctx, drain):
    X, y = orc.generate_dataset(150_000, 128, seed=5, dtype=np.float32)
    ctx.set_drain_rows(drain)
    try:
        S = _gram(ctx, X, y, b2.KERNEL_TCGEN05)
    finally:
        ctx.set_drain_rows(8192)
    ctx.gram_import(S)
    coef, _ = ctx.solve()
    fo = orc.fit_from_stats(orc.gram_stats(X, y))
    assert np.max(np.abs(coef - fo["coef"])) < (COEF_TOL if drain <= 8192 else 1e-4)


@pytest.mark.parametrize("kernel", [b2.KERNEL_SIMT, b2.KERNEL_TCGEN05])
def test_row_mask_equals_gather(ctx, kernel):
    X, y = orc.generate_dataset(30_011, 64, seed=3, dtype=np.float32)
    mask = s1.split_mask(X.shape[0])
    S = _gram(ctx, X, y, kernel, mask=mask, keep=1)
    So = orc.gram_stats(X[mask == 1], y[mask == 1])
    assert S[64, 64] == int((mask == 1).sum())
    assert _rel(S, So) < (1e-12 if kernel == b2.KERNEL_SIMT else 2e-6)


@pytest.mark.parametrize("d,kind", [(20, "f32"), (24, "f32"), (40, "f32"), (48, "f32"), (24, "bf16"), (40, "bf16"),
                                    (56, "bf16")])
def test_packed_rows_with_mask_and_bf16(ctx, d, kind):
    """pack * d < 128: the tile tail is TMA zero fill; the row mask is per original row (2-D mask view at pack = 5)."""
    X, y = orc.generate_dataset(52_345, d, seed=d, dtype=np.float32)
    mask = s1.split_mask(X.shape[0])
    if kind == "bf16":
        bits = b2.native.to_bf16_bits(X)
        X = b2.native.from_bf16_bits(bits)
        src = bits
    else:
        src = X
    for keep in (1, 0):
        S = _gram(ctx, src, y, b2.KERNEL_TCGEN05, mask=mask, keep=keep, kind=kind if kind == "bf16" else None)
        So = orc.gram_stats(X[mask == keep], y[mask == keep])
        assert S[d, d] == int((mask == keep).sum())
        assert _rel(S, So) < 2e-6
    S = _gram(ctx, src, y, b2.KERNEL_AUTO, kind=kind if kind == "bf16" else None)     # AUTO takes the same path
    assert _rel(S, orc.gram_stats(X, y)) < 2e-6
    ctx.gram_import(S)
    coef, _ = ctx.solve()
    assert np.max(np.abs(coef - orc.fit_from_stats(orc.gram_stats(X, y))["coef"])) < COEF_TOL


def test_bf16_storage_fits_the_bf16_rows(ctx):
    X, y = orc.generate_dataset(120_000, 128, seed=19, dtype=np.float32)
    bits = b2.native.to_bf16_bits(X)
    Xr = b2.native.from_bf16_bits(bits)
    S = _gram(ctx, bits, y, b2.KERNEL_TCGEN05, kind="bf16")
    ctx.gram_import(S)
    coef, b0 = ctx.solve()
    fo = orc.fit_from_stats(orc.gram_stats(Xr, y))
    assert np.max(np.abs(coef - fo["coef"])) < COEF_TOL
    S2 = _gram(ctx, bits, y, b2.KERNEL_SIMT, kind="bf16")
    assert _rel(S2, orc.gram_stats(Xr, y)) < 1e-12


def test_accumulate_is_additive_and_deterministic(ctx):
    """Linearity: S(A u B) = S(A) + S(B); same input twice -> bit-identical statistic."""
    X, y = orc.generate_dataset(96_000, 128, seed=8, dtype=np.float32)
    whole = _gram(ctx, X, y, b2.KERNEL_TCGEN05)
    again = _gram(ctx, X, y, b2.KERNEL_TCGEN05)
    assert np.array_equal(whole, again)
    ctx.set_kernel(b2.KERNEL_TCGEN05)
    ctx.gram_reset(128)
    for lo, hi in ((0, 40_000), (40_000, 96_000)):
        Xd, yd = ctx.to_device(X[lo:hi]), ctx.to_device(y[lo:hi])
        ctx.gram_accumulate(Xd, yd)
        Xd.free(); yd.free()
    parts = ctx.gram_export()
    ctx.set_kernel(b2.KERNEL_AUTO)
    assert parts[128, 128] == 96_000
    assert _rel(parts, whole) < 1e-6


def test_host_streamed_equals_device_resident(ctx):
    X, y = orc.generate_dataset(600_000, 32, seed=2, dtype=np.float32)   # > 2 staging blocks of 262 144 rows
    dev = _gram(ctx, X, y, b2.KERNEL_AUTO)
    ctx.gram_reset(32)
    ctx.gram_accumulate(X, y)            # host ndarray -> B2_MEM_HOST
    host = ctx.gram_export()
    assert host[32, 32] == 600_000
    assert _rel(host, dev) < 1e-6
    ctx.gram_import(host)
    coef, _ = ctx.solve()
    assert np.max(np.abs(coef - orc.fit_from_stats(orc.gram_stats(X, y))["coef"])) < COEF_TOL


def test_export_import_round_trip(ctx):
    X, y = orc.generate_dataset(3000, 9, seed=4)
    S = orc.gram_stats(X, y)
    ctx.gram_import(S)
    assert np.array_equal(ctx.gram_export(), S)


# ------------------------------------------------------------------------------------------------
# solve
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d", [(2000, 1), (5000, 8), (20_000, 128), (3000, 33)])
@pytest.mark.parametrize("alpha", [0.0, 10.0])
def test_cholesky_solve_matches_oracle(ctx, n, d, alpha):
    X, y = orc.generate_dataset(n, d, seed=5 * n + d)
    S = orc.gram_stats(X, y)
    ctx.gram_import(S)
    coef, b0 = ctx.solve(alpha=alpha)
    fo = orc.fit_from_stats(S, alpha=alpha)
    assert np.max(np.abs(coef - fo["coef"])) < 1e-10
    assert abs(b0 - fo["intercept"]) < 1e-7
    c0, _ = ctx.solve(alpha=alpha, fit_intercept=False)
    fo0 = orc.fit_from_stats(S, alpha=alpha, fit_intercept=False)
    assert np.max(np.abs(c0 - fo0["coef"])) < 1e-9


@pytest.mark.parametrize("n,d", [(2000, 1), (5000, 8), (20_000, 128), (3000, 33)])
def test_spectral_solve_matches_gelsd_attributes(ctx, n, d):
    from sklearn.linear_model import LinearRegression
    X, y = orc.generate_dataset(n, d, seed=n + 3 * d)
    reg = LinearRegression().fit(X, y)
    ctx.gram_import(orc.gram_stats(X, y))
    coef, b0, sing, rank = ctx.solve_spectral()
    assert rank == reg.rank_
    np.testing.assert_allclose(sing, reg.singular_, rtol=1e-8)
    assert np.max(np.abs(coef - reg.coef_)) < 1e-9
    assert abs(b0 - reg.intercept_) < 1e-6


def test_rank_deficient_gives_minimum_norm_solution(ctx, golden_dir):
    g = np.load(os.path.join(golden_dir, "sk_rank_deficient.npz"))
    ctx.gram_import(orc.gram_stats(g["X"], g["y"]))
    with pytest.raises(np.linalg.LinAlgError):
        ctx.solve()
    coef, b0, sing, rank = ctx.solve_spectral()
    assert rank == int(g["rank"])
    assert np.max(np.abs(coef - g["coef"])) < 1e-7
    est = b2.B200LinearRegression(ctx=ctx).fit(g["X"], g["y"])       # falls through to the spectral solution
    assert np.max(np.abs(est.coef_ - g["coef"])) < 1e-3               # fp32 staging of a singular problem
    assert est.rank_ == int(g["rank"])


def test_docstring_known_answer(ctx, golden_dir):
    g = np.load(os.path.join(golden_dir, "sk_docstring.npz"))
    est = b2.B200LinearRegression(ctx=ctx).fit(g["X"], g["y"])
    np.testing.assert_allclose(est.coef_, [1.0, 2.0], atol=1e-9)
    assert float(est.intercept_) == pytest.approx(3.0, abs=1e-8)
    np.testing.assert_allclose(est.predict(np.array([[3, 5]])), [16.0], atol=1e-5)


# ------------------------------------------------------------------------------------------------
# scoring + metrics
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d", [(10_000, 128), (777, 5), (100_000, 32), (1, 1)])
def test_score_matches_oracle(ctx, n, d):
    X, y = orc.generate_dataset(n, d, seed=n, dtype=np.float32)
    coef = np.linspace(0.3, 0.7, d)
    p = orc.predict(X, coef, 1.5)
    mask = (np.arange(n) % 5 == 0).astype(np.uint8)
    yhat, stats = ctx.score(ctx.to_device(X), coef, 1.5, y=ctx.to_device(y), row_mask=ctx.to_device(mask))
    yh = yhat.to_host()
    assert np.max(np.abs(yh[mask == 1] - p[mask == 1])) <= np.max(np.abs(p)) * 1e-6
    so = orc.score_stats(y[mask == 1], p[mask == 1])
    assert np.max(np.abs(stats - so) / np.maximum(np.abs(so), 1e-300)) < 1e-12
    yh2, _ = ctx.score(X, coef, 1.5)                                     # host path, predict only
    assert np.max(np.abs(yh2 - p)) <= np.max(np.abs(p)) * 1e-6


@pytest.mark.parametrize("kind", ["f32", "bf16"])
@pytest.mark.parametrize("n,d", [(64, 128), (20_000, 128), (70_003, 64), (33_000, 96), (12_345, 100), (50_000, 72),
                                 (40_000, 32), (25_003, 20), (30_000, 48), (9_000, 24), (15_000, 40)])
def test_streaming_score_path_matches_oracle(ctx, n, d, kind):
    """Wide contiguous rows go through the TMA ring (full tiles) + the register-fed kernel (tail): same numbers."""
    if kind == "bf16" and d % 8:
        pytest.skip("bf16 rows need d % 8 == 0 for the 16-byte pitch")
    X, y = orc.generate_dataset(n, d, seed=n + 1, dtype=np.float32)
    if kind == "bf16":
        bits = b2.native.to_bf16_bits(X)
        X = b2.native.from_bf16_bits(bits)
        Xd = ctx.to_device(bits, "bf16")
    else:
        Xd = ctx.to_device(X)
    coef = np.linspace(-0.4, 0.9, d)
    p = orc.predict(X, coef, -2.5)
    yd = ctx.to_device(y)
    for mask in (None, (np.arange(n) % 3 != 0).astype(np.uint8)):
        md = ctx.to_device(mask) if mask is not None else None
        yhat, stats = ctx.score(Xd, coef, -2.5, y=yd, row_mask=md)
        yh = yhat.to_host()
        sel = slice(None) if mask is None else (mask == 1)
        assert np.max(np.abs(yh[sel] - p[sel])) <= np.max(np.abs(p)) * 1e-6
        if mask is not None:
            assert np.all(yh[mask == 0] == 0.0)
        so = orc.score_stats(y[sel], p[sel])
        assert np.max(np.abs(stats - so) / np.maximum(np.abs(so), 1e-300)) < 1e-12
        yhat.free()
        _, stats2 = ctx.score(Xd, coef, -2.5, y=yd, row_mask=md, want_yhat=False)      # metrics only
        assert np.array_equal(stats, stats2)
        yh3, none_stats = ctx.score(Xd, coef, -2.5, row_mask=md)                          # predict only
        assert none_stats is None and np.array_equal(yh3.to_host(), yh)
        yh3.free()
        if md is not None:
            md.free()
    Xd.free(); yd.free()


@pytest.mark.parametrize("kind", ["f32", "bf16"])
@pytest.mark.parametrize("n,d", [(5000, 1), (33_333, 1), (20_000, 2), (9_001, 3), (12_000, 4), (7_000, 5), (30_001, 8),
                                 (5_000, 12), (11_111, 16)])
def test_narrow_score_path_matches_oracle(ctx, n, d, kind):
    """D <= 16: one lane per row behind the bulk-copy ring (full tiles) + the register-fed kernel (tail)."""
    X, y = orc.generate_dataset(n, d, seed=n + 7, dtype=np.float32)
    if kind == "bf16":
        bits = b2.native.to_bf16_bits(X)
        X = b2.native.from_bf16_bits(bits)
        Xd = ctx.to_device(bits, "bf16")
    else:
        Xd = ctx.to_device(X)
    coef = np.linspace(0.45, 0.6, d)
    p = orc.predict(X, coef, 0.75)
    yd = ctx.to_device(y)
    for mask in (None, s1.split_mask(n)):
        md = ctx.to_device(mask) if mask is not None else None
        for keep in ((1,) if mask is None else (0, 1)):
            yhat, stats = ctx.score(Xd, coef, 0.75, y=yd, row_mask=md, mask_keep=keep)
            yh = yhat.to_host()
            sel = slice(None) if mask is None else (mask == keep)
            assert np.max(np.abs(yh[sel] - p[sel])) <= np.max(np.abs(p)) * 1e-6
            if mask is not None:
                assert np.all(yh[mask != keep] == 0.0)
            so = orc.score_stats(y[sel], p[sel])
            assert np.max(np.abs(stats - so) / np.maximum(np.abs(so), 1e-300)) < 1e-12
            yhat.free()
        if md is not None:
            md.free()
    Xd.free(); yd.free()


def test_reference_shape_train_model_at_scale(ctx):
    """The reference's own shape (one feature) at 50 M rows: masked fit (narrow Gram) + hold-out metrics (narrow score)
    recover the generator's truth, and the two passes see complementary row sets."""
    n = 50_000_000 + 123
    X, y = ctx.synth(n, 1, seed=2024)
    mask = ctx.to_device((np.arange(n, dtype=np.int64) % 5 != 0).astype(np.uint8))     # 80 / 20 like stage_1...:98-103
    est = b2.B200LinearRegression(ctx=ctx)
    est.fit(X, y, row_mask=mask, mask_keep=1, with_spectrum=False)
    assert abs(est.coef_[0] - 0.5) < 2e-4 and abs(est.intercept_ - 1.0) < 2e-2
    _, stats = ctx.score(X, est.coef_, float(est.intercept_), y=y, row_mask=mask, mask_keep=0, want_yhat=False)
    assert stats[5] == n - int(round(ctx.gram_export()[1, 1]))              # hold-out rows = all rows - training rows
    mape, r2, mx = s1.metrics_from_stats(stats)
    assert 0.65 < r2 < 0.70                 # var(0.5 x) / (var(0.5 x) + 100) = 208.3 / 308.3
    X.free(); y.free(); mask.free()


def test_score_into_a_preallocated_buffer(ctx):
    X, y = orc.generate_dataset(30_000, 128, seed=77, dtype=np.float32)
    coef = np.linspace(0.2, 0.8, 128)
    Xd = ctx.to_device(X)
    ref, _ = ctx.score(Xd, coef, 1.0)
    out = ctx.empty((30_000,), "f32")
    got, _ = ctx.score(Xd, coef, 1.0, out=out)
    assert got is out and np.array_equal(out.to_host(), ref.to_host())
    host_out = np.empty(30_000, dtype=np.float32)
    got_h, _ = ctx.score(X, coef, 1.0, out=host_out)                   # host rows, host buffer
    assert got_h is host_out and np.array_equal(host_out, ref.to_host())
    with pytest.raises(RuntimeError):
        ctx.score(Xd, coef, 1.0, out=np.empty(30_000, dtype=np.float32))
    Xd.free(); ref.free(); out.free()


def test_streaming_score_large_batch(ctx):
    """2 M x 128 device-resident rows (TMA ring + a 3-row register-fed tail) against the fp64 oracle."""
    n, d = 2_000_003, 128
    X, y = ctx.synth(n, d, seed=21)
    coef = np.linspace(0.1, 0.9, d)
    yh, st = ctx.score(X, coef, 0.5, y=y)
    Xh, yh_host = X.to_host(), yh.to_host()
    p = orc.predict(Xh[:50_000], coef, 0.5)
    assert np.max(np.abs(yh_host[:50_000] - p)) <= np.max(np.abs(p)) * 1e-6
    tail = slice(n - 5000, n)
    assert np.max(np.abs(yh_host[tail] - orc.predict(Xh[tail], coef, 0.5))) <= np.max(np.abs(p)) * 1e-6
    so = orc.score_stats(y.to_host(), orc.predict(Xh, coef, 0.5))
    assert np.max(np.abs(st - so) / np.maximum(np.abs(so), 1e-300)) < 1e-11
    X.free(); y.free(); yh.free()


def test_model_metrics_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "ref_model_metrics.npz"))
    m = s1.model_metrics(g["y"], g["p"])
    assert list(m.columns) == ["date", "MAPE", "r_squared", "max_residual"]
    # one clamped |y| ~ 0 row dominates MAPE (division by eps): fp32 staging moves it by ~1e-7 relative
    assert m["MAPE"].iloc[0] == pytest.approx(float(g["MAPE"]), rel=1e-5)
    assert m["r_squared"].iloc[0] == pytest.approx(float(g["r_squared"]), rel=1e-5)
    assert m["max_residual"].iloc[0] == pytest.approx(float(g["max_residual"]), rel=1e-5)


# ------------------------------------------------------------------------------------------------
# the stage: train_model vs the unmodified reference's outputs
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", ["d1_day1", "d1_30days", "d1_small"])
def test_train_model_matches_reference_golden(golden_dir, tag):
    import pandas as pd
    g = np.load(os.path.join(golden_dir, f"ref_train_model_{tag}.npz"))
    df = pd.DataFrame({"date": "2021-04-08", "y": g["y"], "X": g["X"][:, 0]})
    model, metrics = s1.train_model(df)
    assert str(model) == "LinearRegression()"
    assert np.max(np.abs(model.coef_ - g["coef"])) < 1e-5
    assert abs(model.intercept_ - float(g["intercept"])) < 1e-3
    assert model.rank_ == int(g["rank"])
    np.testing.assert_allclose(model.singular_, g["singular"], rtol=1e-5)
    for k in ("MAPE", "r_squared", "max_residual"):
        assert metrics[k].iloc[0] == pytest.approx(float(g[k]), rel=2e-5), k


@pytest.mark.parametrize("tag", ["n10k_d8", "n4k_d32_f32", "n3k_d128_f32"])
def test_train_model_multi_feature_golden(golden, tag):
    import pandas as pd
    g = golden(f"sk_train_model_{tag}.npz")
    d = g["X"].shape[1]
    df = pd.DataFrame(g["X"], columns=[f"X{j}" for j in range(d)])
    df["y"] = g["y"]
    model, metrics = s1.train_model(df)
    o = orc.train_model(g["X"], g["y"])                # fp64 fit of the same rows
    assert np.max(np.abs(model.coef_ - o["coef"])) < 1e-4
    assert metrics["r_squared"].iloc[0] == pytest.approx(o["r_squared"], rel=1e-4)
    assert metrics["MAPE"].iloc[0] == pytest.approx(o["MAPE"], rel=1e-4)


def test_stage_entrypoint_file_in_model_out(tmp_path, monkeypatch):
    """bodywork.yaml drop-in: tranche CSVs in -> regressor-<date>.joblib + metrics CSV out; the artefact is
    consumed the way stage_2_serve_model.py:65,76-79 does."""
    import joblib
    import pandas as pd
    bucket = tmp_path / "bucket"
    (bucket / "datasets").mkdir(parents=True)
    frames = []
    for k, day in enumerate(("2021-04-07", "2021-04-08", "2021-04-09")):
        X, y = orc.generate_dataset(1440, 1, seed=40 + k, alpha=orc.alpha_of_day(97 + k), drop_negative=True)
        df = pd.DataFrame({"date": day, "y": y, "X": X[:, 0]})
        df.to_csv(bucket / "datasets" / f"regression-dataset-{day}.csv", index=False)
        frames.append(df)
    monkeypatch.chdir(tmp_path)
    monkeypatch.setattr(s1, "BUCKET_DIR", str(bucket))
    assert s1.run() == 0
    model_file = bucket / "models" / "regressor-2021-04-09.joblib"
    metrics_file = bucket / "model-metrics" / "regressor-2021-04-09.csv"
    model = joblib.load(io.BytesIO(model_file.read_bytes()))
    allrows = pd.concat(frames)
    o = orc.train_model(allrows["X"].to_numpy(), allrows["y"].to_numpy())
    pred = model.predict(np.array(50, ndmin=2))[0]                      # stage_2: np.array(features, ndmin=2)
    assert pred == pytest.approx(o["intercept"] + 50 * o["coef"][0], abs=1e-3)
    assert str(model) == "LinearRegression()"
    m = pd.read_csv(metrics_file)
    assert list(m.columns) == ["date", "MAPE", "r_squared", "max_residual"]
    assert m["r_squared"].iloc[0] == pytest.approx(o["r_squared"], rel=1e-4)
    # failure path: exit status 1 (stage_1_train_model.py:176-178)
    monkeypatch.setattr(s1, "BUCKET_DIR", str(tmp_path / "nope"))
    assert s1.run() == 1


def test_incremental_refit_equals_full_refit(ctx):
    est = b2.B200LinearRegression(ctx=ctx)
    ctx.gram_reset(16)
    Xs, ys = [], []
    for day in range(5):
        X, y = orc.generate_dataset(20_000, 16, seed=day, alpha=orc.alpha_of_day(1 + day), dtype=np.float32)
        est.partial_fit(X, y)
        Xs.append(X); ys.append(y)
    full = orc.fit_from_stats(orc.gram_stats(np.concatenate(Xs), np.concatenate(ys)))
    assert np.max(np.abs(est.coef_ - full["coef"])) < COEF_TOL


# ------------------------------------------------------------------------------------------------
# synthetic rows + BASELINE-size properties
# ------------------------------------------------------------------------------------------------
def test_synth_is_deterministic_and_shardable(ctx):
    Xa, ya = ctx.synth(10_000, 128, seed=7)
    Xb, yb = ctx.synth(4_000, 128, seed=7, row_offset=6_000)
    A, B = Xa.to_host(), Xb.to_host()
    assert np.array_equal(A[6_000:], B) and np.array_equal(ya.to_host()[6_000:], yb.to_host())
    assert 0.0 <= A.min() and A.max() < 100.0 and abs(A.mean() - 50.0) < 0.1
    resid = ya.to_host() - (1.0 + 0.5 * A.astype(np.float64).sum(axis=1))
    assert abs(resid.mean()) < 0.5 and abs(resid.std() - 10.0) < 0.5
    Xc, _ = ctx.synth(10_000, 128, seed=8)
    assert not np.array_equal(A, Xc.to_host())


@pytest.mark.parametrize("kind", ["f32", "bf16"])
def test_baseline_config_10m_x_128_properties(ctx, kind):
    """BASELINE.json configs[1] at full size: exact row count, additivity over two halves, recovery of the
    generating coefficients within sampling error, and agreement with the fp64 CUDA-core kernel on a
    slice (the oracle itself is pinned to the same kernel at small sizes above)."""
    n, d = 10_000_000, 128
    X, y = ctx.synth(n, d, seed=1234, kind=kind)
    ctx.set_kernel(b2.KERNEL_TCGEN05)
    ctx.gram_reset(d)
    ctx.gram_accumulate(X, y)
    S = ctx.gram_export()
    assert S[d, d] == n
    coef, b0 = ctx.solve()
    assert np.max(np.abs(coef - 0.5)) < 6 * 10.0 / (28.87 * np.sqrt(n))      # 6 sigma of the OLS sampling error
    assert abs(b0 - 1.0) < 1.0
    # slice check against the fp64 SIMT kernel
    m = 200_000
    Xh = X.to_host()[:m]
    yh = y.to_host()[:m]
    Xs, ys = ctx.to_device(Xh, kind), ctx.to_device(yh)
    ctx.gram_reset(d); ctx.gram_accumulate(Xs, ys); tc = ctx.gram_export()
    ctx.set_kernel(b2.KERNEL_SIMT)
    ctx.gram_reset(d); ctx.gram_accumulate(Xs, ys); ref = ctx.gram_export()
    ctx.set_kernel(b2.KERNEL_AUTO)
    assert _rel(tc, ref) < 2e-6
    for a in (X, y, Xs, ys):
        a.free()


# ------------------------------------------------------------------------------------------------
# 30-day concept-drift replay (BASELINE.json configs[4]); binary tranches through the stage
# ------------------------------------------------------------------------------------------------
def _drift_tranches(days, n, d, dtype=np.float32):
    out = []
    for day in range(days):
        X, y = orc.generate_dataset(n, d, seed=500 + day, alpha=orc.alpha_of_day(1 + 7 * day), dtype=dtype,
                                    drop_negative=(d == 1))
        out.append((X, y))
    return out


@pytest.mark.parametrize("n,d,days", [(1440, 1, 30), (50_000, 128, 6)])
def test_replay_incremental_equals_refit_on_the_same_train_rows(ctx, n, d, days):
    from bodywork_mlops_demo_b200 import incremental
    tranches = _drift_tranches(days, n, d)
    res = incremental.replay(tranches, d, mode="incremental", ctx=ctx)
    assert len(res) == days and res[0].test_mape is None and res[1].test_mape is not None
    Xs, ys = [], []
    for k, (X, y) in enumerate(tranches):
        m = s1.split_mask(len(y))
        Xs.append(X[m == 1]); ys.append(y[m == 1])
        fo = orc.fit_lstsq(np.concatenate(Xs).astype(np.float64), np.concatenate(ys).astype(np.float64))
        assert res[k].n_train_total == sum(len(v) for v in ys)
        assert np.max(np.abs(res[k].coef - fo["coef"])) < COEF_TOL, k
        if k + 1 < days:   # day k+1's tranche scored with model(k): stage_4 semantics
            Xn, yn = tranches[k + 1]
            mo = orc.metrics(yn, orc.predict(Xn, fo["coef"], fo["intercept"]))
            assert res[k + 1].test_r2 == pytest.approx(mo["r_squared"], rel=1e-3, abs=1e-4)
            assert res[k + 1].test_max_residual == pytest.approx(mo["max_residual"], rel=1e-3)


def test_replay_exact_mode_reproduces_the_reference_split(ctx):
    from bodywork_mlops_demo_b200 import incremental
    tranches = _drift_tranches(5, 3000, 8)
    res = incremental.replay(tranches, 8, mode="exact", ctx=ctx)
    allX = np.concatenate([t[0] for t in tranches]); ally = np.concatenate([t[1] for t in tranches])
    o = orc.train_model(allX, ally)            # the reference's global RandomState(42) split over all history
    assert res[-1].n_train_total == o["n_train"]
    assert np.max(np.abs(res[-1].coef - o["coef"])) < COEF_TOL


def test_stage_reads_binary_tranches(tmp_path, monkeypatch):
    import datetime as dt
    import joblib
    from bodywork_mlops_demo_b200 import tranche_io as tio
    bucket = tmp_path / "bucket"
    (bucket / "datasets").mkdir(parents=True)
    Xs, ys = [], []
    for k in range(3):
        X, y = orc.generate_dataset(40_000, 16, seed=70 + k, dtype=np.float32)
        tio.write_tranche(str(bucket / "datasets" / f"regression-dataset-2021-05-0{k + 1}.b2t"), X, y,
                          dt.date(2021, 5, k + 1))
        Xs.append(X); ys.append(y)
    monkeypatch.chdir(tmp_path)
    monkeypatch.setattr(s1, "BUCKET_DIR", str(bucket))

    def no_frames(path):                                   # binary tranches go file -> pinned memory -> HBM
        raise AssertionError(f"a DataFrame was materialised for {path}")
    monkeypatch.setattr(s1, "_read_tranche_frame", no_frames)
    data, day = s1.download_latest_dataset(str(bucket))
    assert isinstance(data, s1.TrancheRows) and len(data) == 120_000 and str(day) == "2021-05-03"
    assert data.X.dtype == np.float32 and data.X.flags.c_contiguous
    data.free()
    assert s1.run() == 0
    model = joblib.load(bucket / "models" / "regressor-2021-05-03.joblib")
    o = orc.train_model(np.concatenate(Xs), np.concatenate(ys))
    assert np.max(np.abs(model.coef_ - o["coef"])) < COEF_TOL and model.n_features_in_ == 16
    metrics = open(bucket / "model-metrics" / "regressor-2021-05-03.csv").read().splitlines()
    assert metrics[0] == "date,MAPE,r_squared,max_residual"
    assert abs(float(metrics[1].split(",")[2]) - o["r_squared"]) < 2e-5


# ------------------------------------------------------------------------------------------------
# batch scoring companion of stage_2 + stage_4's service-test metrics
# ------------------------------------------------------------------------------------------------
def test_score_payload_follows_the_service_shape_rules(ctx):
    from sklearn.linear_model import LinearRegression
    from bodywork_mlops_demo_b200 import stage_2_scoring as s2
    X, y = orc.generate_dataset(2000, 3, seed=6)
    model = LinearRegression().fit(X, y)
    for features in ([50.0, 2.0, 7.0], [[50.0, 2.0, 7.0], [1.0, 2.0, 3.0]]):
        want = model.predict(np.array(features, ndmin=2))                  # stage_2_serve_model.py:77-78
        got = s2.score_payload(model, {"X": features}, ctx)
        assert got["prediction"] == pytest.approx(want[0], rel=1e-6)
        np.testing.assert_allclose(got["predictions"], want, rtol=1e-6)
        assert got["model_info"] == "LinearRegression()"
    X1, y1 = orc.generate_dataset(500, 1, seed=8)
    m1 = LinearRegression().fit(X1, y1)
    assert s2.score_payload(m1, {"X": 50}, ctx)["prediction"] == pytest.approx(m1.predict(np.array(50, ndmin=2))[0],
                                                                                    rel=1e-6)
    with pytest.raises(ValueError):
        s2.score_batch(model, [[1.0, 2.0]], ctx)


@pytest.mark.parametrize("n,d", [(1317, 1), (200_000, 128)])
def test_service_test_matches_stage_4_metric_definitions(ctx, n, d):
    from sklearn.linear_model import LinearRegression
    from bodywork_mlops_demo_b200 import stage_2_scoring as s2
    X, y = orc.generate_dataset(n + 500, d, seed=9, dtype=np.float32, drop_negative=(d == 1))
    model = LinearRegression().fit(X[:500].astype(np.float64), y[:500].astype(np.float64))
    Xt, yt = X[500:], y[500:]
    rec = s2.service_test(model, Xt, yt, ctx=ctx)
    want = orc.service_test_metrics(yt.astype(np.float64), model.predict(Xt.astype(np.float64)))
    assert rec["MAPE"].iloc[0] == pytest.approx(want["MAPE"], rel=1e-5)
    assert rec["r_squared"].iloc[0] == pytest.approx(want["r_squared"], rel=1e-6)
    assert rec["max_residual"].iloc[0] == pytest.approx(want["max_residual"], rel=1e-4)
    assert rec["mean_response_time"].iloc[0] < 8.22e-3      # the reference's recorded 8.22 ms per row over HTTP
    np.testing.assert_allclose(s2.score_batch(model, Xt, ctx), model.predict(Xt.astype(np.float64)), rtol=2e-6)


# ------------------------------------------------------------------------------------------------
# raw C-ABI: strided rows (ldx > d), unaligned buffers, argument errors
# ------------------------------------------------------------------------------------------------
def _raw_accumulate(ctx, Xdev_ptr, ydev_ptr, n, d, ldx, x_dtype=0, mask_ptr=None, keep=1):
    lib = b2.native.load()
    return lib.b2_gram_accumulate(ctx._h, Xdev_ptr, x_dtype, ydev_ptr, n, d, ldx, b2.native.MEM_DEVICE, mask_ptr, keep)


@pytest.mark.parametrize("kernel", [b2.KERNEL_TCGEN05, b2.KERNEL_SIMT])
def test_strided_rows_ldx_greater_than_d(ctx, kernel):
    """X given as the first 64 columns of a wider row-major matrix (ldx = 96): TMA global stride / SIMT pitch."""
    n, d, ldx = 50_001, 64, 96
    wide, y = orc.generate_dataset(n, ldx, seed=12, dtype=np.float32)
    Xd, yd = ctx.to_device(wide), ctx.to_device(y)
    ctx.set_kernel(kernel)
    ctx.gram_reset(d)
    assert _raw_accumulate(ctx, Xd.ptr, yd.ptr, n, d, ldx) == 0, b2.native.last_error()
    S = ctx.gram_export()
    ctx.set_kernel(b2.KERNEL_AUTO)
    assert _rel(S, orc.gram_stats(wide[:, :d], y)) < (2e-6 if kernel == b2.KERNEL_TCGEN05 else 1e-12)
    # scoring with the same pitch
    lib = b2.native.load()
    coef = np.linspace(0.1, 0.9, d)
    stats = np.zeros(10)
    yhat = ctx.empty((n,), "f32")
    rc = lib.b2_score(ctx._h, Xd.ptr, 0, n, d, ldx, b2.native.MEM_DEVICE, coef.ctypes.data, 2.0, yd.ptr, None, 1,
                      yhat.ptr, stats.ctypes.data)
    assert rc == 0, b2.native.last_error()
    p = orc.predict(wide[:, :d], coef, 2.0)
    assert np.max(np.abs(yhat.to_host() - p)) <= np.max(np.abs(p)) * 1e-6
    np.testing.assert_allclose(stats, orc.score_stats(y, p), rtol=1e-10)


def test_unaligned_buffers_fall_back_to_the_simt_kernel(ctx):
    """AUTO picks the CUDA-core kernel when X / y are not 16-byte aligned; forcing tcgen05 is refused."""
    n, d = 10_000, 8
    X, y = orc.generate_dataset(n + 1, d, seed=13, dtype=np.float32)
    Xd, yd = ctx.to_device(X), ctx.to_device(y)
    xp, yp = Xd.ptr + d * 4, yd.ptr + 4          # skip one row: y is now 4-byte aligned only
    ctx.gram_reset(d)
    assert _raw_accumulate(ctx, xp, yp, n, d, d) == 0, b2.native.last_error()
    assert _rel(ctx.gram_export(), orc.gram_stats(X[1:], y[1:])) < 1e-12
    ctx.set_kernel(b2.KERNEL_TCGEN05)
    ctx.gram_reset(d)
    assert _raw_accumulate(ctx, xp, yp, n, d, d) == -6      # B2_E_UNSUPPORTED
    assert "tcgen05 path needs" in b2.native.last_error()
    ctx.set_kernel(b2.KERNEL_AUTO)


def test_argument_errors_return_codes_not_crashes(ctx):
    lib = b2.native.load()
    X, y = orc.generate_dataset(100, 4, seed=1, dtype=np.float32)
    Xd, yd = ctx.to_device(X), ctx.to_device(y)
    ctx.gram_reset(4)
    assert _raw_accumulate(ctx, Xd.ptr, yd.ptr, 100, 5, 5) == -1          # d differs from the statistic's d
    assert _raw_accumulate(ctx, Xd.ptr, yd.ptr, 100, 4, 3) == -1          # ldx < d
    assert _raw_accumulate(ctx, Xd.ptr, yd.ptr, -1, 4, 4) == -1
    assert _raw_accumulate(ctx, Xd.ptr, yd.ptr, 100, 4, 4, x_dtype=7) == -1
    assert _raw_accumulate(ctx, None, yd.ptr, 100, 4, 4) == -1            # null X
    assert lib.b2_gram_reset(ctx._h, 129) == -1 and lib.b2_gram_reset(ctx._h, 0) == -1
    assert lib.b2_ctx_set_drain_rows(ctx._h, 100) == -1                   # not a multiple of the 64-row tile
    with pytest.raises(RuntimeError, match="alpha must be >= 0"):
        ctx.gram_reset(4); ctx.gram_accumulate(Xd, yd); ctx.solve(alpha=-1.0)
    assert _raw_accumulate(ctx, Xd.ptr, yd.ptr, 0, 4, 4) == 0             # empty block is a no-op
    ctx.gram_reset(4)
    ctx.gram_accumulate(Xd, yd)
    assert ctx.gram_export()[4, 4] == 100


def test_masked_tail_tile_on_the_tensor_core_path(ctx):
    """n not a multiple of the 64-row tile AND a row mask: TMA zero-fill + mask bytes + the E warp's row validity."""
    n, d = 64 * 500 + 37, 128
    X, y = orc.generate_dataset(n, d, seed=14, dtype=np.float32)
    mask = (np.random.RandomState(2).rand(n) < 0.7).astype(np.uint8)
    S = _gram(ctx, X, y, b2.KERNEL_TCGEN05, mask=mask, keep=1)
    assert S[d, d] == int(mask.sum())
    assert _rel(S, orc.gram_stats(X[mask == 1], y[mask == 1])) < 2e-6
    S0 = _gram(ctx, X, y, b2.KERNEL_TCGEN05, mask=mask, keep=0)
    assert S0[d, d] == n - int(mask.sum())


@pytest.mark.parametrize("kind", ["f32", "bf16"])
def test_single_bf16_operand_mode_meets_the_contract_at_large_n(ctx, kind):
    """B2_PRECISION_BF16 ('bf16-accum', BASELINE.json configs[1]): one bf16 operand, fp32 accumulate.  The operand
    rounding error is zero-mean, so the coefficient error falls as 1/sqrt(n): asserted < 1e-4 (the contract) at
    n = 2 M and compared with the default split mode on the same rows."""
    n, d = 2_000_000, 128
    X, y = ctx.synth(n, d, seed=21, kind=kind)
    Xh, yh = X.to_host(), y.to_host()
    Xf = (Xh if kind == "f32" else b2.native.from_bf16_bits(Xh)).astype(np.float64)
    fo = orc.fit_from_stats(orc.gram_stats(Xf, yh.astype(np.float64)))
    errs = {}
    for mode in (b2.PRECISION_SPLIT, b2.PRECISION_BF16):
        ctx.set_precision(mode)
        ctx.set_kernel(b2.KERNEL_TCGEN05)
        try:
            ctx.gram_reset(d); ctx.gram_accumulate(X, y)
            coef, _ = ctx.solve()
            assert ctx.gram_export()[d, d] == n
        finally:
            ctx.set_precision(b2.PRECISION_SPLIT); ctx.set_kernel(b2.KERNEL_AUTO)
        errs[mode] = float(np.max(np.abs(coef - fo["coef"])))
    assert errs[b2.PRECISION_SPLIT] < COEF_TOL
    assert errs[b2.PRECISION_BF16] < 1e-4
    X.free(); y.free()


def test_plain_c_client_fits_through_the_c_abi(c_client):
    """tests/c_client/fit_client.c: C99, pageable host rows, b2_gram_accumulate(B2_MEM_HOST) + b2_solve vs a
    double-precision normal-equation solve written out in the client."""
    import subprocess
    proc = subprocess.run([c_client], capture_output=True, text=True, timeout=300)
    assert proc.returncode == 0, proc.stdout + proc.stderr
    assert "worst coefficient error" in proc.stdout


def test_non_finite_input_is_refused_like_sklearn(ctx):
    X, y = orc.generate_dataset(5000, 8, seed=3, dtype=np.float32)
    X[17, 3] = np.nan
    with pytest.raises(ValueError, match="NaN"):
        b2.B200LinearRegression(ctx=ctx).fit(X, y)
    X[17, 3] = 1.0
    y[5] = np.inf
    with pytest.raises(ValueError, match="NaN"):
        b2.B200LinearRegression(ctx=ctx).fit(X, y)
    y[5] = 0.0
    assert np.all(np.isfinite(b2.B200LinearRegression(ctx=ctx).fit(X, y).coef_))     # the context is still usable


# ------------------------------------------------------------------------------------------------
# DataFrame columns -> device rows (b2_upload_columns): the gather + conversion train_model uses
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,dtype", [(1, 1, np.float64), (1000, 3, np.float64), (70_001, 128, np.float64),
                                       (300_000, 40, np.float32), (263_000, 128, np.float64)])
def test_upload_columns_equals_numpy_conversion(ctx, n, d, dtype):
    """Strided float64 / float32 columns (a consolidated pandas block, a Fortran-ordered array, every other element of a
    longer vector) arrive as exactly ``np.stack(columns, 1).astype(float32)``, across the 262 144-row bounce blocks."""
    rng = np.random.RandomState(n + d)
    block = (rng.rand(d, n) * 100).astype(dtype)                  # pandas: one (d, n) block, columns contiguous
    cols = [block[j] for j in range(d)]
    if d >= 3:
        wide = (rng.rand(2 * n) * 100).astype(dtype)
        cols[1] = wide[::2]                                        # a strided column
        cols[2] = np.asfortranarray(rng.rand(n, 2).astype(dtype))[:, 1]
    Xd = ctx.upload_columns(cols)
    got = Xd.to_host()
    Xd.free()
    assert got.shape == (n, d) and got.dtype == np.float32
    assert np.array_equal(got, np.stack(cols, axis=1).astype(np.float32))
    with pytest.raises(RuntimeError):
        ctx.upload_columns([cols[0], cols[0][:-1]] if n > 1 else [np.zeros(3, np.int32)])


def test_train_model_takes_dataframe_columns_without_a_host_copy(ctx, monkeypatch):
    """train_model(DataFrame) must not materialise the (n, d) matrix on the host: the columns go to b2_upload_columns."""
    import pandas as pd
    X, y = orc.generate_dataset(50_000, 16, seed=5, dtype=np.float64)
    df = pd.DataFrame({"date": "2021-01-01", "y": y, **{f"X{j}": X[:, j] for j in range(16)}})

    def no_stack(*a, **k):
        raise AssertionError("train_model stacked the columns on the host")
    monkeypatch.setattr(np, "stack", no_stack)
    model, metrics = s1.train_model(df)
    monkeypatch.undo()
    mask = s1.split_mask(len(y))
    ref = orc.fit_from_stats(orc.gram_stats(X[mask == 1].astype(np.float32), y[mask == 1].astype(np.float32)))
    assert np.max(np.abs(model.coef_ - ref["coef"])) < COEF_TOL
    assert 0.9 < float(metrics["r_squared"][0]) <= 1.0


def test_estimator_fit_on_float64_host_rows(ctx):
    """float64 host rows (what scikit-learn users pass) are converted by b2_upload_columns on the way up and fitted
    resident: same coefficients as the oracle's fit of the float32-rounded rows, masks honoured, buffers released."""
    X, y = orc.generate_dataset(120_000, 32, seed=21, dtype=np.float64)
    est = b2.B200LinearRegression(ctx=ctx).fit(X, y)
    ref = orc.fit_from_stats(orc.gram_stats(X.astype(np.float32), y.astype(np.float32)))
    assert np.max(np.abs(est.coef_ - ref["coef"])) < COEF_TOL and est.rank_ == 32
    mask = (np.arange(len(y)) % 4 != 0).astype(np.uint8)
    est2 = b2.B200LinearRegression(ctx=ctx).fit(np.asfortranarray(X), y, row_mask=mask, mask_keep=1)
    ref2 = orc.fit_from_stats(orc.gram_stats(X[mask == 1].astype(np.float32), y[mask == 1].astype(np.float32)))
    assert np.max(np.abs(est2.coef_ - ref2["coef"])) < COEF_TOL
    with pytest.raises(ValueError):
        b2.B200LinearRegression(ctx=ctx).fit(X, y[:-1])

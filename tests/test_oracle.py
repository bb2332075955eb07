"""Pin the CPU oracle: golden vectors produced by the unmodified reference + scikit-learn itself."""
import glob
import os

import numpy as np
import pytest

from oracle import ols_oracle as orc


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name), allow_pickle=False)


@pytest.mark.parametrize("tag", ["d1_day1", "d1_30days", "d1_small"])
def test_train_model_matches_reference_golden(golden_dir, tag):
    g = _load(golden_dir, f"ref_train_model_{tag}.npz")
    out = orc.train_model(g["X"], g["y"])
    np.testing.assert_allclose(out["coef"], g["coef"], rtol=0, atol=1e-12)
    assert abs(out["intercept"] - float(g["intercept"])) < 1e-10
    assert out["rank"] == int(g["rank"])
    np.testing.assert_allclose(out["singular"], g["singular"], rtol=1e-12)
    assert abs(out["MAPE"] - float(g["MAPE"])) < 1e-12
    assert abs(out["r_squared"] - float(g["r_squared"])) < 1e-12
    assert abs(out["max_residual"] - float(g["max_residual"])) < 1e-10
    assert list(g["columns"]) == ["date", "MAPE", "r_squared", "max_residual"]


def test_metrics_match_reference_golden(golden_dir):
    g = _load(golden_dir, "ref_model_metrics.npz")
    m = orc.metrics(g["y"], g["p"])
    assert m["MAPE"] == pytest.approx(float(g["MAPE"]), rel=1e-13)
    assert m["r_squared"] == pytest.approx(float(g["r_squared"]), rel=1e-13)
    assert m["max_residual"] == pytest.approx(float(g["max_residual"]), rel=1e-15)


@pytest.mark.parametrize("tag,tol", [("n10k_d8", 1e-11), ("n4k_d32_f32", 2e-5), ("n3k_d128_f32", 2e-4)])
def test_train_model_multi_feature_golden(golden, tag, tol):
    # the f32 goldens were fitted by sklearn in float32; the oracle is float64 -> looser bound
    g = golden(f"sk_train_model_{tag}.npz")
    out = orc.train_model(g["X"], g["y"])
    assert np.max(np.abs(out["coef"] - g["coef"])) < tol
    assert out["rank"] == int(g["rank"])


@pytest.mark.parametrize("n", [5, 57, 1440, 10_001])
def test_split_indices_bit_exact(golden_dir, n):
    g = _load(golden_dir, f"sk_split_n{n}.npz")
    tr, te = orc.split_indices(n)
    assert np.array_equal(tr, g["train"]) and np.array_equal(te, g["test"])
    assert orc.split_sizes(n) == (g["train"].size, g["test"].size)


def test_docstring_known_answer(golden_dir):
    g = _load(golden_dir, "sk_docstring.npz")
    f = orc.fit_lstsq(g["X"], g["y"])
    np.testing.assert_allclose(f["coef"], [1.0, 2.0], atol=1e-12)
    assert f["intercept"] == pytest.approx(3.0, abs=1e-12)
    f2 = orc.fit_from_stats(orc.gram_stats(g["X"], g["y"]))
    np.testing.assert_allclose(f2["coef"], g["coef"], atol=1e-10)
    assert f2["intercept"] == pytest.approx(float(g["intercept"]), abs=1e-10)


def test_rank_deficient_min_norm(golden_dir):
    g = _load(golden_dir, "sk_rank_deficient.npz")
    f = orc.fit_lstsq(g["X"], g["y"])
    np.testing.assert_allclose(f["coef"], g["coef"], atol=1e-10)
    assert f["rank"] == int(g["rank"]) == 4
    f2 = orc.fit_from_stats(orc.gram_stats(g["X"], g["y"]))
    np.testing.assert_allclose(f2["coef"], g["coef"], atol=1e-7)
    assert f2["rank"] == 4
    np.testing.assert_allclose(f2["singular"][:4], g["singular"][:4], rtol=1e-9)


@pytest.mark.parametrize("n,d,dtype", [(10_000, 8, np.float64), (50_000, 32, np.float32), (20_000, 128, np.float64)])
def test_gram_route_equals_sklearn(n, d, dtype):
    """The secondary (scalable) oracle -- chunked fp64 Gram + centred solve -- pinned to sklearn."""
    from sklearn.linear_model import LinearRegression
    X, y = orc.generate_dataset(n, d, seed=100 + d, dtype=dtype)
    reg = LinearRegression().fit(X.astype(np.float64), y.astype(np.float64))
    f = orc.fit_from_stats(orc.gram_stats(X, y, chunk=4096))
    assert np.max(np.abs(f["coef"] - reg.coef_)) < 1e-9
    assert abs(f["intercept"] - reg.intercept_) < 1e-6
    np.testing.assert_allclose(f["singular"], reg.singular_, rtol=1e-8)
    assert f["rank"] == reg.rank_


def test_ridge_matches_sklearn_ridge():
    from sklearn.linear_model import Ridge
    X, y = orc.generate_dataset(5000, 16, seed=7)
    for alpha in (1e-3, 1.0, 1e4):
        reg = Ridge(alpha=alpha, solver="cholesky").fit(X, y)
        f = orc.fit_from_stats(orc.gram_stats(X, y), alpha=alpha)
        assert np.max(np.abs(f["coef"] - reg.coef_)) < 1e-9
        assert abs(f["intercept"] - reg.intercept_) < 1e-7


def test_train_model_oracle_equals_sklearn_sequence():
    X, y = orc.generate_dataset(3001, 5, seed=3)
    a = orc.train_model(X, y)
    b = orc.train_model_sklearn(X, y)
    assert np.max(np.abs(a["coef"] - b["coef"])) < 1e-12
    for k in ("MAPE", "r_squared", "max_residual"):
        assert a[k] == pytest.approx(b[k], rel=1e-11)
    assert (a["n_train"], a["n_test"]) == (b["n_train"], b["n_test"])


def test_generator_follows_reference_dgp():
    X, y = orc.generate_dataset(200_000, 1, seed=1, alpha=orc.alpha_of_day(1), drop_negative=True)
    assert 0.0 <= X.min() and X.max() <= 100.0 and (y >= 0).all()
    assert orc.alpha_of_day(1) == 1.0
    f = orc.fit_lstsq(X, y)
    assert abs(f["coef"][0] - 0.5) < 0.07      # dropping y < 0 attenuates the slope (cf. golden 0.45)
    assert len(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz"))) >= 10

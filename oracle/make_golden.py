"""Generate tests/golden/*.npz by running the UNMODIFIED reference.  TEST INFRASTRUCTURE ONLY.

Run with a checkout of the reference project at hand:

    python oracle/make_golden.py REFERENCE_DIR [OUT_DIR]      (OUT_DIR defaults to tests/golden)

What it does
------------
* imports ``REFERENCE_DIR/mlops_simulation/stage_1_train_model.py`` with ``boto3`` /
  ``botocore.exceptions`` stubbed (they are absent from the image and only used for S3 I/O),
* calls the reference's own ``train_model(data)`` (stage_1_train_model.py:93-108) and
  ``model_metrics`` (:79-90) on seeded datasets drawn with the reference's data-generating
  process (stage_3_synthetic_data_generation.py:36-43),
* for D > 1 (the reference itself is D = 1) calls the same scikit-learn entry points the
  reference calls (train_test_split / LinearRegression / the three metrics),
* stores inputs and outputs as small ``.npz`` fixtures; the tests read only the fixtures.  Rows too large to store
  (over ``MAX_STORED_BYTES``) are kept as the seed and shape they are drawn with plus their SHA-256;
  ``tests/conftest.py`` draws them again and checks the digest.
"""
from __future__ import annotations

import hashlib
import importlib.util
import os
import sys
import types

import numpy as np
import pandas as pd

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF_MODULE = os.path.join("mlops_simulation", "stage_1_train_model.py")
MAX_STORED_BYTES = 1_000_000

sys.path.insert(0, ROOT)
from oracle import ols_oracle as orc  # noqa: E402


def load_reference(ref_dir: str):
    boto3 = types.ModuleType("boto3")
    botocore = types.ModuleType("botocore")
    exc = types.ModuleType("botocore.exceptions")
    exc.ClientError = type("ClientError", (Exception,), {})
    botocore.exceptions = exc
    sys.modules.setdefault("boto3", boto3)
    sys.modules.setdefault("botocore", botocore)
    sys.modules.setdefault("botocore.exceptions", exc)
    spec = importlib.util.spec_from_file_location("ref_stage_1", os.path.join(ref_dir, REF_MODULE))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def main(ref_dir: str, out_dir: str) -> None:
    GOLD = out_dir
    os.makedirs(GOLD, exist_ok=True)
    ref = load_reference(ref_dir)
    import sklearn

    # ---- D = 1 through the reference's own train_model -------------------------------
    for tag, n, seed, day in (("d1_day1", 1440, 11, 1), ("d1_30days", 30 * 1440, 12, 45),
                              ("d1_small", 57, 13, 200)):
        X, y = orc.generate_dataset(n, 1, seed=seed, alpha=orc.alpha_of_day(day), drop_negative=True)
        df = pd.DataFrame({"date": np.full(len(y), "2021-04-08"), "y": y, "X": X[:, 0]})
        model, metrics = ref.train_model(df)
        np.savez(os.path.join(GOLD, f"ref_train_model_{tag}.npz"),
                 X=X, y=y, coef=model.coef_, intercept=np.float64(model.intercept_),
                 rank=np.int64(model.rank_), singular=model.singular_,
                 MAPE=np.float64(metrics["MAPE"].iloc[0]),
                 r_squared=np.float64(metrics["r_squared"].iloc[0]),
                 max_residual=np.float64(metrics["max_residual"].iloc[0]),
                 columns=np.array(list(metrics.columns)),
                 sklearn_version=np.array(sklearn.__version__), source=np.array(REF_MODULE + "::train_model"))
        print(tag, model.coef_, model.intercept_, metrics.to_dict("records")[0])

    # ---- model_metrics alone -------------------------------------------------------------
    rng = np.random.RandomState(5)
    ya = rng.normal(50, 20, 301)
    ya[7] = 0.0  # exercises the max(|y|, eps) clamp in MAPE
    yp = ya + rng.normal(0, 3, 301)
    m = ref.model_metrics(ya, yp)
    np.savez(os.path.join(GOLD, "ref_model_metrics.npz"), y=ya, p=yp,
             MAPE=np.float64(m["MAPE"].iloc[0]), r_squared=np.float64(m["r_squared"].iloc[0]),
             max_residual=np.float64(m["max_residual"].iloc[0]))

    # ---- D > 1 through the same sklearn calls (reference's dependency) ----------------------
    for tag, n, d, seed, dtype in (("n10k_d8", 10_000, 8, 21, np.float64),
                                   ("n4k_d32_f32", 4_096, 32, 22, np.float32),
                                   ("n3k_d128_f32", 3_000, 128, 23, np.float32)):
        X, y = orc.generate_dataset(n, d, seed=seed, dtype=dtype)
        out = orc.train_model_sklearn(X, y)
        rows = {"X": X} if X.nbytes <= MAX_STORED_BYTES else {
            "seed": np.int64(seed), "X_shape": np.array(X.shape, dtype=np.int64),
            "X_sha256": np.array(hashlib.sha256(X.tobytes()).hexdigest())}
        np.savez(os.path.join(GOLD, f"sk_train_model_{tag}.npz"), **rows, y=y,
                 coef=out["coef"], intercept=np.float64(out["intercept"]), rank=np.int64(out["rank"]),
                 singular=out["singular"], MAPE=np.float64(out["MAPE"]),
                 r_squared=np.float64(out["r_squared"]), max_residual=np.float64(out["max_residual"]),
                 sklearn_version=np.array(sklearn.__version__))
        print(tag, out["coef"][:3], out["intercept"], out["MAPE"], out["r_squared"])

    # ---- sklearn's docstring known answer (LinearRegression docstring example) ---------------------
    X = np.array([[1, 1], [1, 2], [2, 2], [2, 3]], dtype=np.float64)
    y = X @ np.array([1.0, 2.0]) + 3.0
    from sklearn.linear_model import LinearRegression
    reg = LinearRegression().fit(X, y)
    np.savez(os.path.join(GOLD, "sk_docstring.npz"), X=X, y=y, coef=reg.coef_,
             intercept=np.float64(reg.intercept_))

    # ---- rank-deficient: duplicated + constant column (gelsd minimum-norm) ---------------------------
    X, y = orc.generate_dataset(500, 4, seed=31)
    X = np.concatenate([X, X[:, :1], np.full((500, 1), 7.0)], axis=1)
    reg = LinearRegression().fit(X, y)
    np.savez(os.path.join(GOLD, "sk_rank_deficient.npz"), X=X, y=y, coef=reg.coef_,
             intercept=np.float64(reg.intercept_), rank=np.int64(reg.rank_), singular=reg.singular_)

    # ---- split indices -----------------------------------------------------------------------
    from sklearn.model_selection import train_test_split
    for n in (5, 57, 1440, 10_001):
        idx = np.arange(n)
        tr, te = train_test_split(idx, test_size=0.2, random_state=42)
        np.savez(os.path.join(GOLD, f"sk_split_n{n}.npz"), train=tr, test=te)
    print("golden fixtures written to", GOLD)


if __name__ == "__main__":
    if len(sys.argv) not in (2, 3):
        raise SystemExit("usage: python oracle/make_golden.py REFERENCE_DIR [OUT_DIR]")
    main(sys.argv[1], sys.argv[2] if len(sys.argv) == 3 else os.path.join(ROOT, "tests", "golden"))

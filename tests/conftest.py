import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (a B200: the kernels are built for sm_100a)")


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


def _load_golden(name: str) -> dict:
    """The arrays of tests/golden/<name>.  A fixture whose rows were too large to store (oracle/make_golden.py) keeps
    the seed and shape they were drawn with and their SHA-256: the rows are drawn again and must match the digest."""
    import hashlib
    import numpy as np
    from oracle import ols_oracle as orc
    with np.load(os.path.join(GOLDEN, name), allow_pickle=False) as fh:
        g = dict(fh)
    if "X" not in g:
        n, d = (int(v) for v in g["X_shape"])
        X, y = orc.generate_dataset(n, d, seed=int(g["seed"]), dtype=g["y"].dtype)
        assert hashlib.sha256(X.tobytes()).hexdigest() == str(g["X_sha256"]), f"{name}: redrawn rows differ"
        assert np.array_equal(y, g["y"]), f"{name}: redrawn targets differ"
        g["X"] = X
    return g


@pytest.fixture(scope="session")
def golden():
    """Loader of a golden fixture by file name: ``golden("sk_train_model_n3k_d128_f32.npz")["X"]``."""
    return _load_golden


def _have_gpu() -> bool:
    try:
        import bodywork_mlops_demo_b200 as b2
        return b2.native.device_count() > 0
    except Exception:
        return False


@pytest.fixture(scope="session")
def ctx():
    """One device context shared by the GPU tests (fails loudly if the extension is missing)."""
    import bodywork_mlops_demo_b200 as b2
    c = b2.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="session")
def c_client(tmp_path_factory):
    """tests/c_client/fit_client.c built with gcc against include/b2gram.h and the in-tree libb2gram.so."""
    import shutil
    import subprocess
    import bodywork_mlops_demo_b200 as b2
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    lib_dir = os.path.dirname(b2.native.lib_path())
    exe = str(tmp_path_factory.mktemp("c_client") / "fit_client")
    cmd = [gcc, "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-O2", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "c_client", "fit_client.c"), "-o", exe, "-L", lib_dir, "-lb2gram", "-lm",
           "-Wl,-rpath," + lib_dir]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    assert proc.returncode == 0, proc.stderr
    return exe

"""CPU-side checks of the boundary: the C-ABI library builds/loads and exports
every symbol include/wdx_b200.h declares; without a GPU it fails loudly instead
of computing on the CPU."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    txt = open(os.path.join(ROOT, "include", "wdx_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(wdx_[a-z0-9_]+)\s*\(", txt)))


def test_header_symbols_are_exported():
    from warpdemux_b200 import _lib

    lib = _lib.load()
    declared = _declared_symbols()
    assert "wdx_predict" in declared and "wdx_model_create" in declared
    for sym in declared:
        assert hasattr(lib, sym), f"{sym} declared in include/wdx_b200.h but not exported"
    assert sorted(_lib.EXPORTS) == declared
    assert b"sm_100a" in lib.wdx_version()


_NO_DEVICE_CHILD = """
import numpy as np, pytest
from warpdemux_b200 import _lib, model_io
from warpdemux_b200.models.dtw_svm import DTW_SVM

assert _lib.device_count() == 0
mdl = DTW_SVM(model_io.load_npz("tests/golden/models/WDX4_rna004_v1_0.npz"))
with pytest.raises(_lib.WdxError, match="no CUDA device"):
    mdl.predict(np.zeros((2, 25)))
"""


def test_no_cpu_fallback_without_gpu():
    """In a child process that sees no device (CUDA_VISIBLE_DEVICES empty), so that it holds on GPU machines too."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE_CHILD], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "warpdemux_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert "oracle" not in src.replace("# oracle", ""), f"{f} mentions the oracle"


def test_argument_validation_precedes_device_use(models):
    from warpdemux_b200.models.dtw_svm import DTW_SVM

    mdl = DTW_SVM(models["WDX4_rna004_v1_0"])
    with pytest.raises(ValueError, match="same number of columns"):
        mdl.predict(np.zeros((3, 24)))
    with pytest.raises(ValueError, match="Model not trained yet."):
        DTW_SVM(None).predict(np.zeros((1, 25)))
    with pytest.raises(ValueError):
        DTW_SVM(models["WDX4_rna004_v1_0"], mode="bogus")


def test_sharding_is_contiguous_and_complete():
    from warpdemux_b200.sharding import shard_bounds, shard_of

    for n, w in [(10, 3), (100, 8), (7, 8), (0, 2), (100_000_000, 8), (1, 1)]:
        b = shard_bounds(n, w)
        assert b[0][0] == 0 and b[-1][1] == n
        assert all(b[g][1] == b[g + 1][0] for g in range(w - 1))
        for g, (s, e) in enumerate(b):
            if e > s:
                assert shard_of(s, n, w) == g and shard_of(e - 1, n, w) == g


def test_model_unpickler_admits_exact_globals_only(tmp_path):
    """load_reference_joblib resolves only an exact list of (module, name) pairs: a crafted file cannot reach a callable
    inside an admitted package (numpy.testing._private.utils.runstring is exec)."""
    import pickle

    import numpy as np
    import pytest

    from warpdemux_b200 import model_io

    class Evil:
        def __reduce__(self):
            import numpy.testing._private.utils as u

            return (u.runstring, ("raise SystemExit('code ran')", {}))

    for i, payload in enumerate((Evil(), np.testing.assert_equal)):
        p = tmp_path / f"evil{i}.joblib"
        p.write_bytes(pickle.dumps(payload, protocol=4))
        with pytest.raises(ValueError, match="refusing to unpickle"):
            model_io.load_reference_joblib(str(p))
    for mod, name in model_io._ALLOWED_GLOBALS:
        assert "testing" not in mod and not mod.startswith(("os", "subprocess", "sys"))


def test_shipped_joblib_models_load_as_the_committed_npz():
    """The reference's five shipped DTW_SVM files load through the allow-listing unpickler and give the arrays of
    tests/golden/models.  The .joblib files are the reference package's, not this repository's: WDX_REFERENCE points at
    a checkout of it."""
    import glob

    from warpdemux_b200 import model_io

    ref = os.environ.get("WDX_REFERENCE")
    files = [f for f in glob.glob(os.path.join(ref, "warpdemux/models/model_files/WDX*_rna004_v1_0.joblib")) if "tRNA" not in f] if ref else []
    if not files:
        pytest.skip("the reference's shipped .joblib model files are not at hand (set WDX_REFERENCE)")
    assert len(files) == 5
    for f in files:
        m = model_io.load_reference_joblib(f)
        g = model_io.load_npz(os.path.join(ROOT, "tests", "golden", "models", os.path.basename(f).replace(".joblib", ".npz")))
        assert np.array_equal(m.sv, g.sv) and np.array_equal(m.dual_coef, g.dual_coef) and np.array_equal(m.thresholds, g.thresholds)

"""CPU: the fingerprint oracle (oracle/wdx_oracle.py `fingerprint`) against the
golden outputs of the reference's own `detect_results_to_fpt`
(tests/golden/fingerprint_rna004.npz, produced by oracle/make_golden.py), and
the restated Cython kernels against the reference's compiled ones (oracle/_ref)."""
import glob
import importlib.util
import json
import os

import numpy as np
import pytest

from wdx_testutil import oracle_fingerprints, synth_adapter_signals

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_oracle_fingerprint_matches_reference_golden(golden_fingerprint):
    g = golden_fingerprint
    cfg = json.loads(str(g["cfg"]))
    status, fpt, dwell, stats = oracle_fingerprints(g["signals"], g["adapter_start"], g["adapter_end"], **cfg)
    assert np.array_equal(status != 0, g["status"] != 0)
    ok = g["status"] == 0
    assert ok.sum() >= 30
    assert np.array_equal(dwell[ok], g["dwell"][ok])
    assert np.array_equal(fpt[ok], g["fpt"][ok]), "float64 fingerprints must be bit-identical"
    assert np.array_equal(stats[ok], g["stats"][ok])


def test_golden_inputs_are_reproducible(golden_fingerprint):
    sig, a0, a1 = synth_adapter_signals(32, seed=2)
    assert np.array_equal(sig, golden_fingerprint["signals"], equal_nan=True)
    assert np.array_equal(a0, golden_fingerprint["adapter_start"]) and np.array_equal(a1, golden_fingerprint["adapter_end"])


def _ref_segmentation():
    hits = glob.glob(os.path.join(ROOT, "oracle", "_ref", "ref_c_segmentation*.so"))
    if not hits:
        pytest.skip("oracle/_ref not built (oracle/build_ref.py needs a checkout of the reference, WDX_REFERENCE)")
    spec = importlib.util.spec_from_file_location("ref_c_segmentation", hits[0])
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("w", [1, 5, 12])
def test_restated_cython_kernels_match_the_compiled_reference(w):
    from oracle import wdx_oracle as o

    ref = _ref_segmentation()
    rng = np.random.default_rng(w)
    x = np.repeat(rng.standard_normal(60) * 10 + 80, rng.integers(5, 60, 60)) + rng.normal(0, 2, 0 + 0 or 1)
    x = (x + rng.normal(0, 2, x.size)).astype(np.float32).astype(np.float64)
    assert np.array_equal(o.windowed_t_test(x, w), ref.c_windowed_t_test(x, w))
    segs = np.unique(np.concatenate([[0], rng.integers(1, x.size - 1, 40), [x.size]])).astype(np.int64)
    assert np.array_equal(o.new_means(x, segs), ref.c_new_means(x, segs))

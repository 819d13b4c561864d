"""LLR fallback of the boundary detection (reference combined.py:222-296, llr.py, _c_llr.pyx).
CPU: the restatement (oracle/wdx_oracle_llr.py) against (1) the reference's own compiled Cython gains
(oracle/_ref/ref_c_llr, built by oracle/build_ref.py from a checkout of the reference) and (2) the detection path,
boundaries and verdicts the reference's `combined_detect_cnn` produced for the reads of
test_data/demux/4000_rna004.pod5 that leave the plain CNN path (tests/golden/real4000_rna004_WDX4.npz,
oracle/make_golden_real4000.py: 28 hail-mary validations, 193 LLR re-detections, 35 of them validating)."""
import glob
import importlib.util
import json
import os

import numpy as np
import pytest

from conftest import GOLD, ROOT
from wdx_testutil import real4000_rows


@pytest.fixture(scope="module")
def g4000():
    with np.load(os.path.join(GOLD, "real4000_rna004_WDX4.npz")) as z:
        return {k: z[k] for k in z.files}


def llr_config(g):
    from oracle import wdx_oracle_llr as ol

    c = json.loads(str(g["cfg"]))
    return ol.LLRConfig(max_obs_trace=c["max_obs_trace"], min_obs_adapter=c["min_obs_adapter"], max_obs_adapter=c["max_obs_adapter"],
                        downscale_factor=c["downscale_factor"], sig_norm_outlier_thresh=c["outlier_thresh"],
                        adapter_peak_prominence=c["adapter_peak_prominence"], adapter_peak_rel_height=c["adapter_peak_rel_height"],
                        adapter_peak_width=c["adapter_peak_width"], fallback_to_llr=c["fallback_to_llr"],
                        fallback_to_llr_short_reads=c["fallback_to_llr_short_reads"])


def test_gains_match_reference_cython():
    hits = glob.glob(os.path.join(ROOT, "oracle", "_ref", "ref_c_llr*.so"))
    if not hits:
        pytest.skip("oracle/_ref/ref_c_llr not built (oracle/build_ref.py needs a checkout of the reference, WDX_REFERENCE)")
    spec = importlib.util.spec_from_file_location("ref_c_llr", hits[0])
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    from oracle import wdx_oracle_llr as ol

    rng = np.random.default_rng(7)
    for n, head, tail, start in ((1000, 101, 1, 0), (1000, 1, 1, 333), (517, 5, 5, 0), (40, 1, 1, 7), (12, 5, 5, 0)):
        x = np.concatenate([rng.normal(0.5, 1.0, n // 2), rng.normal(-0.7, 0.3, n - n // 2)]).astype(np.float32).astype(np.float64)
        x[3] = x[4]                                  # a zero-variance pair
        with np.errstate(all="ignore"):
            want, c, c2 = ref.c_llr_trace(x, start, n - 1, head, tail, 1, 0, 0, 0, 0, 0, 0, 1)
        gc, gc2 = ol.cumsums(x)
        assert np.array_equal(gc, c) and np.array_equal(gc2, c2)
        got = ol.gains(gc, gc2, start, n - 1, head, tail)
        assert np.array_equal(got, want, equal_nan=True), (n, head, tail, start)


def test_oracle_reproduces_reference_detection_paths(g4000):
    """Every read of the committed subset (all reads that leave the plain CNN path + every 16th read)."""
    from oracle import wdx_oracle_llr as ol
    from oracle import wdx_oracle_validate as ov

    g = g4000
    idx, rows, _, _ = real4000_rows(g)
    cfg, vcfg = llr_config(g), ov.ValidateConfig()
    off_path = (g["n_validate"] > 1) | (g["success"] == 0)
    assert off_path.sum() == 198 and set(np.flatnonzero(off_path)) <= set(idx.tolist())
    n_hm = n_llr = 0
    for j, i in enumerate(idx):
        res, path, info = ol.detect_one(rows[j], int(g["full_lengths"][i]), g["cnn_preds"][i], cfg, vcfg)
        assert bool(res["success"]) == bool(g["success"][i]), i
        # the fixture's hm_tried = the hail mary found a poly(A) end and its validation ran
        assert (info["hm_polya"] > 0) == bool(g["hm_tried"][i]) and bool(info["llr_tried"]) == bool(g["llr_tried"][i]), i
        assert info["hm_polya"] == g["hm_polya"][i], i
        assert (ov.fail_reason(res["code"], res["checks"]) or "") == str(g["fail_reason"][i]), i
        if g["success"][i]:
            assert path == g["path"][i], i
            assert (res["adapter_start"], res["adapter_end"], res["polya_end"]) == tuple(g["bounds"][i]), i
        assert (info["llr_adapter_end"], info["llr_polya_end"]) == tuple(g["llr_bounds"][i]), i
        n_hm += int(info["hm_polya"] > 0)
        n_llr += int(info["llr_tried"])
    assert n_hm == 28 and n_llr == 193

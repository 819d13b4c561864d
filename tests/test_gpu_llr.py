"""LLR fallback of the boundary detection on the device (wdx_validate_set_llr, csrc/llr_kernel.cuh) and
BASELINE.json configs[0] over the reference's whole test file.

Reference: adapted/detect/combined.py:222-296 (+ llr.py, _c_llr.pyx).  Bar: the path every read takes (CNN validated /
hail mary / full LLR / failed), the boundaries, the fail reasons and the reported statistics are those of the
reference's own `combined_detect_cnn` (tests/golden/real4000_rna004_WDX4.npz, oracle/make_golden_real4000.py);
fingerprints bit-identical, barcode calls identical, with no host hook (`llr_fallback=None`)."""
import dataclasses
import json
import os

import numpy as np
import pytest

from conftest import GOLD
from wdx_testutil import real4000_rows

pytestmark = pytest.mark.gpu
MINIBATCH = 1000        # production minibatch size (the reference's parser default)


@pytest.fixture(scope="module")
def g4000():
    with np.load(os.path.join(GOLD, "real4000_rna004_WDX4.npz")) as z:
        return {k: z[k] for k in z.files}


def _llr_cfg(g):
    from warpdemux_b200.detect import combined

    c = json.loads(str(g["cfg"]))
    return combined.LLRConfig(max_obs_trace=c["max_obs_trace"], min_obs_adapter=c["min_obs_adapter"], max_obs_adapter=c["max_obs_adapter"],
                              downscale_factor=c["downscale_factor"], sig_norm_outlier_thresh=c["outlier_thresh"],
                              adapter_peak_prominence=c["adapter_peak_prominence"], adapter_peak_rel_height=c["adapter_peak_rel_height"],
                              adapter_peak_width=c["adapter_peak_width"], fallback_to_llr=c["fallback_to_llr"],
                              fallback_to_llr_short_reads=c["fallback_to_llr_short_reads"])


def _fp_cfg(g):
    c = json.loads(str(g["cfg"]))
    return {k: c[k] for k in ("padding", "outlier_thresh", "min_obs_per_base", "running_stat_width", "num_events", "barcode_num_events")}


def _check_detection(g, idx, vb, where=""):
    """vb: ValidationBatch of the reads `idx` (full report) against the reference's DetectResults."""
    from warpdemux_b200.detect import combined

    bad = []
    src = vb.source & 3
    for j, i in enumerate(idx):
        want_path = int(g["path"][i])
        reason = vb.fail_reason(j) or ""
        ok = bool(vb.success[j]) == bool(g["success"][i]) and reason == str(g["fail_reason"][i])
        if g["success"][i]:
            ok = ok and tuple(vb.bounds[j]) == tuple(g["bounds"][i]) and int(src[j]) == want_path
        # which validate calls ran (fixture: hm_tried = the hail mary found a poly(A) end and was validated)
        if g["hm_tried"][i]:
            ok = ok and bool(vb.source[j] & 4)
        ok = ok and bool(vb.source[j] & 8) == bool(g["llr_tried"][i])
        # DetectResults.llr_adapter_end / llr_polya_end of the reported result
        want_llr = tuple(g["llr_bounds"][i])
        got_llr = (int(vb.bounds[j, 1]), int(vb.bounds[j, 2])) if src[j] else (0, 0)
        ok = ok and got_llr == want_llr
        # reported statistics (NaN = None): mvs_*, adapter_rna_median_shift, real_adapter_*  and the 18 partition values
        got = np.array([vb.vals[j, 5], vb.vals[j, 6], vb.vals[j, 7], vb.vals[j, 8], vb.vals[j, 9], vb.vals[j, 10], vb.vals[j, 2],
                        vb.vals[j, 3], vb.vals[j, 4]])
        ok = ok and np.array_equal(got, g["fvals"][i], equal_nan=True)
        if vb.parts is not None:
            ok = ok and np.array_equal(vb.parts[j], g["parts"][i], equal_nan=True)
        if not ok:
            bad.append((int(i), bool(vb.success[j]), reason, str(g["fail_reason"][i]), vb.bounds[j].tolist(), g["bounds"][i].tolist(),
                        int(vb.source[j]), want_path, got_llr, want_llr))
    assert not bad, (where, len(bad), bad[:6])
    assert combined.fail_reason(10) == "MAD normalization failed: scale is 0"


def test_gpu_llr_fallback_matches_reference_paths(g4000):
    """Validation + hail mary + LLR on the reference CNN's own boundaries: the committed subset (all 198 reads that leave
    the plain CNN path + every 16th read)."""
    from warpdemux_b200.detect import combined

    g = g4000
    idx, rows, _, _ = real4000_rows(g)
    v = combined.Validator(combined.ValidateConfig(), device=0, llr=_llr_cfg(g))
    vb = v.validate(rows, g["full_lengths"][idx], g["cnn_preds"][idx], partitions=True)
    _check_detection(g, idx, vb, "subset")
    assert ((vb.source & 3) == 1).sum() >= 5 and ((vb.source & 3) == 2).sum() == 30
    # without the fallback the same reads fail, and the verdicts of the others are unchanged
    v0 = combined.Validator(combined.ValidateConfig(), device=0, llr=None)
    vb0 = v0.validate(rows, g["full_lengths"][idx], g["cnn_preds"][idx])
    assert (vb0.source == 0).all()
    assert np.array_equal(vb0.success[(vb.source & 3) == 0], vb.success[(vb.source & 3) == 0])
    assert (vb0.success[(vb.source & 3) == 2] == 0).all()
    # only one of the two fallbacks
    only_llr = dataclasses.replace(_llr_cfg(g), fallback_to_llr_short_reads=False)
    v1 = combined.Validator(combined.ValidateConfig(), device=0, llr=only_llr)
    vb1 = v1.validate(rows, g["full_lengths"][idx], g["cnn_preds"][idx])
    assert ((vb1.source & 4) == 0).all() and (vb1.success >= vb0.success).all() and vb1.success.sum() > vb0.success.sum()
    for h in (v, v0, v1):
        h.close()


def test_gpu_llr_fallback_matches_oracle_on_synthetic_rows():
    """Kernel == oracle/wdx_oracle_llr.detect_one on the synthetic rows of the validation fixture (every fail reason of the
    first validation; short and long reads), three LLR configurations."""
    from oracle import wdx_oracle_llr as ol
    from oracle import wdx_oracle_validate as ov
    from warpdemux_b200.detect import combined
    from wdx_testutil import pack_rows

    rows, lens, preds = [], [], []
    for s in range(360):
        row, fl, pr = ov.synthetic_case(s, stride=11500, k=5)
        rows.append(row)
        lens.append(int(fl))
        preds.append(pr)
    sig, lens, preds = pack_rows(rows), np.array(lens, dtype=np.int64), np.array(preds, dtype=np.int64)
    for kw in (dict(), dict(adapter_peak_width=400, adapter_peak_prominence=0.5), dict(max_obs_trace=8000, fallback_to_llr_short_reads=False)):
        lcfg = combined.LLRConfig(**kw)
        ocfg = ol.LLRConfig(**dataclasses.asdict(lcfg))
        v = combined.Validator(combined.ValidateConfig(), device=0, llr=lcfg)
        vb = v.validate(sig, lens, preds, partitions=True)
        v.close()
        n_src = [0, 0, 0]
        for i in range(len(rows)):
            res, path, info = ol.detect_one(sig[i], int(lens[i]), preds[i], ocfg, ov.ValidateConfig())
            assert bool(vb.success[i]) == bool(res["success"]), (kw, i)
            assert int(vb.code[i]) == int(res["code"]) and int(vb.checks[i]) == int(res["checks"]), (kw, i, vb.code[i], res["code"])
            want_src = 0 if info["primary"] == "cnn" else (2 if path == ol.PATH_LLR else 1)
            assert int(vb.source[i]) & 3 == want_src, (kw, i)
            assert bool(vb.source[i] & 8) == bool(info["llr_tried"]), (kw, i)
            if res["code"] not in (ov.HAS_NAN, ol.MAD_ZERO):
                assert tuple(vb.bounds[i]) == (res["adapter_start"], res["adapter_end"], res["polya_end"]), (kw, i)
                assert np.array_equal(vb.vals[i], res["vals"], equal_nan=True), (kw, i)
                assert np.array_equal(vb.parts[i], res["parts"], equal_nan=True), (kw, i)
            n_src[want_src] += 1
        assert n_src[0] > 100, n_src


def _spc(g):
    from types import SimpleNamespace

    from warpdemux_b200.detect import cnn

    c = json.loads(str(g["cfg"]))
    return SimpleNamespace(core=cnn.CoreConfig(min_obs_adapter=c["min_obs_adapter"], max_obs_adapter=c["max_obs_adapter"],
                                               downscale_factor=c["downscale_factor"], max_obs_trace=c["max_obs_trace"]),
                           cnn_boundaries=cnn.CNNBoundariesConfig(polya_cand_k=c["polya_cand_k"]))


def whole_file_expectations(g, idx):
    """The reference chain's whole-file results for the reads `idx` of real4000_rna004_WDX4.npz (read numbers of the file,
    repeats allowed): CNN predictions, detection verdict, boundaries, path, fingerprint status, fail reasons, fingerprints
    and barcode calls.  Where numpy's unstable argsort of EQUAL t-test scores decided the change points on the machine that
    wrote the fixture, the expected fingerprint and call are the oracle's stable-order ones (`stable_idx`)."""
    good = g["status"] == 0
    pos = np.cumsum(good) - 1
    want_fpt, want_label = g["fpt"].copy(), np.where(good, g["y_pred"][np.maximum(pos, 0)], -1)
    want_fpt[g["stable_idx"]] = g["stable_fpt"]
    want_label[g["stable_idx"]] = g["stable_label"]
    assert set(g["stable_idx"].tolist()) <= set(g["tie_reads"].tolist()) and g["stable_idx"].size <= 2
    want = {key: g[key][idx] for key in ("read_ids", "full_lengths", "calibration_offset", "calibration_scale", "cnn_preds", "success",
                                         "bounds", "path", "status", "fail_reason")}
    want.update(fpt=want_fpt[idx], label=want_label[idx], good=good[idx])
    return want


def chain_mismatches(want, res):
    """MinibatchResults `res` (in order, want_fpt=True) against `whole_file_expectations` -> {field: row positions that differ}."""
    cat = lambda f: np.concatenate([getattr(r, f) for r in res])
    suc, bounds, preds = cat("detect_success"), cat("bounds"), cat("preds")
    labels, status, fpt, src = cat("labels"), cat("fp_status"), cat("fpt"), cat("detect_source")
    good = want["good"]
    bad = {
        "cnn_preds": np.flatnonzero((preds != want["cnn_preds"]).any(axis=1)),
        "detect_success": np.flatnonzero(suc != want["success"]),
        "bounds": np.flatnonzero((bounds != want["bounds"]).any(axis=1) & (want["success"] == 1)),
        "path": np.flatnonzero(((src & 3) != want["path"]) & (want["success"] == 1)),
        "fp_status": np.flatnonzero(status != want["status"]),
        "fpt": np.flatnonzero(good & ~np.all(fpt == want["fpt"], axis=1)),
        "label": np.flatnonzero(good & (labels != want["label"])),
        "label_failed_reads": np.flatnonzero(~good & (labels != -1)),
    }
    out = {k: v for k, v in bad.items() if v.size}
    reasons = [r.fail_reason(i) or "" for r in res for i in range(r.labels.size)]
    failed = np.flatnonzero(want["success"] == 0)
    wrong = [int(i) for i in failed if reasons[i] != str(want["fail_reason"][i])]
    if wrong:
        out["fail_reason"] = np.array(wrong)
    return out


def test_gpu_whole_test_file_raw_signal_to_barcode_calls(g4000, models):
    """BASELINE.json configs[0] on the reads of test_data/demux/4000_rna004.pod5 whose int16 rows the fixture keeps
    (every read that leaves the plain CNN path, every 16th read and the tie read below: 439 of the 4000), in minibatches
    of MINIBATCH, raw ADC rows -> `MinibatchDemuxer.run` (CNN -> validation -> hail mary / LLR -> fingerprint -> DTW + SVC)
    with llr_fallback=None: detection verdict, boundaries, fingerprints (bit-identical) and barcode calls of every one of
    them equal the reference chain's over the whole file.  One caveat, recorded in the fixture: where two EQUAL t-test
    scores compete (106 reads have such ties, for 1 of them the outcome depends on the order) scipy's result hangs on
    numpy's unstable argsort; the kernels use the stable order, and for that read the expected values are the oracle's
    stable-order ones."""
    from warpdemux_b200.detect import cnn, combined
    from warpdemux_b200.file_proc import AdcBatch, MinibatchDemuxer
    from warpdemux_b200.models.dtw_svm import DTW_SVM
    from warpdemux_b200.sig_proc import FingerprintConfig

    g = g4000
    idx, rows, adc, num = real4000_rows(g)
    n = idx.size
    off_path = (g["n_validate"] > 1) | (g["success"] == 0)
    assert set(np.flatnonzero(off_path).tolist()) | set(g["stable_idx"].tolist()) <= set(idx.tolist())
    spc = _spc(g)
    md = cnn.load_cnn_model(os.path.join(GOLD, "models", "cnn_rna004_130bps_v0.2.4.npz"), device=0)
    # everything below is per read of the subset
    want = whole_file_expectations(g, idx)
    good = want["good"]
    mismatches = {}
    # (the third pass: the sequential form of the step, without the fingerprint pass next to the LLR tail)
    for mode, inp, overlap in (("guarded", "float", True), ("exact", "adc", True), ("guarded", "adc", False)):
        mp = DTW_SVM(models["WDX4_rna004_v1_0"], device=0, mode=mode)
        dmx = MinibatchDemuxer(mp, md, core=spc.core, cnn_boundaries=spc.cnn_boundaries, validate_config=combined.ValidateConfig(),
                               fp_config=FingerprintConfig(**_fp_cfg(g)), device=0, llr=_llr_cfg(g), full_detect_report=True,
                               overlap_llr_tail=overlap)
        assert dmx.llr_fallback is None
        res = []
        for lo in range(0, n, MINIBATCH):
            sl = slice(lo, lo + MINIBATCH)
            batch = rows[sl] if inp == "float" else AdcBatch(adc[sl], num[sl], want["calibration_offset"][sl], want["calibration_scale"][sl])
            res.append(dmx.run(batch, want["full_lengths"][sl], want["read_ids"][sl], want_fpt=True))
        key = mode if overlap else mode + "_sequential"
        mismatches[key] = {k: idx[v].tolist() for k, v in chain_mismatches(want, res).items()}      # as read numbers of the file
        df = res[0].predictions
        assert list(df["#read_id"]) == [str(x) for x in want["read_ids"][:MINIBATCH][good[:MINIBATCH]]]
        dmx.close()
    md.close()
    assert mismatches == {"guarded": {}, "exact": {}, "guarded_sequential": {}}, mismatches      # the mismatch list must be empty
    assert (g4000["path"] == 2).sum() == 30 and (g4000["path"] == 1).sum() == 5 and g4000["success"].sum() == 3837

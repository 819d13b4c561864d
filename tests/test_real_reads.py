"""BASELINE.json configs[0]: real reads of the reference's own test file
(test_data/demux/4000_rna004.pod5), boundaries from the reference's own adapter detection,
expected fingerprints / barcode calls from the reference's own sig_proc and DTW_SVM
(tests/golden/real_rna004_WDX4.npz, oracle/make_golden_real.py).  CPU: the oracle against that
fixture.  GPU: the CUDA path against it, through the C ABI."""
import json
import os

import numpy as np
import pytest

from wdx_testutil import oracle_fingerprints, real_fixture_rows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cfg(g):
    cfg = json.loads(str(g["cfg"]))
    cfg.pop("model")
    return cfg


def test_oracle_matches_reference_on_real_reads(golden_real, models):
    from oracle import wdx_oracle as o

    g = golden_real
    rows = real_fixture_rows(g)
    ok_det = g["detect_ok"].astype(bool)
    assert ok_det.sum() >= 450
    status, fpt, dwell, stats = oracle_fingerprints(rows[ok_det], g["adapter_start"][ok_det], g["adapter_end"][ok_det],
                                                    **_cfg(g))
    assert np.array_equal(status, g["status"][ok_det])
    good = status == 0
    assert np.array_equal(fpt[good], g["fpt"][ok_det][good]), "fingerprints of real reads must be bit-identical"
    assert np.array_equal(dwell[good], g["dwell"][ok_det][good])
    assert np.array_equal(stats[good], g["stats"][ok_det][good])
    m = models["WDX4_rna004_v1_0"]
    pred, prob, conf, _ = o.predict(m, g["fpt"][g["status"] == 0])
    assert np.array_equal(pred, g["y_pred"])
    assert np.abs(prob - g["y_prob"]).max() < 2e-6
    assert (pred != -1).mean() > 0.6          # real barcodes are being called, not noise


@pytest.mark.gpu
def test_gpu_path_matches_reference_on_real_reads(golden_real, models):
    from warpdemux_b200.models.dtw_svm import DTW_SVM
    from warpdemux_b200.sig_proc import Fingerprinter, FingerprintConfig

    g = golden_real
    rows = real_fixture_rows(g)
    cfg = _cfg(g)
    fp = Fingerprinter(FingerprintConfig(**cfg), device=0)
    b = fp.extract(rows, g["adapter_start"], g["adapter_end"], detect_ok=g["detect_ok"])
    assert np.array_equal(b.status, g["status"])
    good = g["status"] == 0
    assert np.array_equal(b.fpt[good], g["fpt"][good])
    assert np.array_equal(b.dwell[good], g["dwell"][good])
    assert np.array_equal(b.stats[good], g["stats"][good])
    # barcode calls: separate predict and the fused signals -> calls step
    for mode in ("exact", "guarded"):
        mdl = DTW_SVM(models["WDX4_rna004_v1_0"], device=0, mode=mode)
        y_pred, y_prob = mdl.predict(b.fpt[good], nproc=1)
        assert np.array_equal(y_pred, g["y_pred"]), mode
        assert np.abs(y_prob - g["y_prob"]).max() < (2e-6 if mode == "exact" else 1e-3)
        labels, prob, conf, status = fp.extract_and_predict(mdl, rows, g["adapter_start"], g["adapter_end"],
                                                            detect_ok=g["detect_ok"])
        assert np.array_equal(status, g["status"])
        assert np.array_equal(labels[good], g["y_pred"]) and (labels[~good] == -1).all()
    fp.close()


def test_pod5_reader_self_check():
    """Minimal pod5 reader (warpdemux_b200/io/pod5_min.py) on a synthetic VBZ chunk: the decoder
    inverts an independently written encoder (zig-zag delta -> 1/2-byte stream with key bits -> zstd)."""
    import pyarrow as pa

    from warpdemux_b200.io.pod5_min import decode_vbz

    rng = np.random.default_rng(0)
    x = np.cumsum(rng.integers(-40, 40, 5000)).astype(np.int16)
    x[100] = 3000
    x[101] = -2000
    d = np.diff(np.concatenate([[0], x.astype(np.int32)])).astype(np.int32)
    d = ((d + 32768) % 65536 - 32768).astype(np.int32)                   # int16 wrap-around of the deltas
    u = ((d << 1) ^ (d >> 31)).astype(np.uint32) & 0xFFFF
    keys = (u > 255).astype(np.uint8)
    data = bytearray()
    for v, k in zip(u.tolist(), keys.tolist()):
        data.append(v & 255)
        if k:
            data.append(v >> 8)
    raw = np.packbits(keys, bitorder="little").tobytes() + bytes(data)
    chunk = pa.Codec("zstd").compress(raw, asbytes=True)
    assert np.array_equal(decode_vbz(chunk, x.size), x)
    assert decode_vbz(pa.Codec("zstd").compress(b"", asbytes=True), 0).size == 0


def test_pod5_reader_on_reference_file_if_present(golden_real):
    """The pod5 reader on a file written by the pod5 library itself: the reference's test file, which is not part of this
    repository (WDX_REFERENCE points at a checkout of the reference).  No cut-down copy is stored: none was taken from
    that file, and a file written by this project's own code would check the reader only against itself; the decoder
    keeps its synthetic self-check above."""
    ref = os.environ.get("WDX_REFERENCE")
    path = os.path.join(ref, "test_data", "demux", "4000_rna004.pod5") if ref else ""
    if not os.path.exists(path):
        pytest.skip("the reference's test_data/demux/4000_rna004.pod5 is not at hand (set WDX_REFERENCE)")
    from warpdemux_b200.io.pod5_min import Pod5File

    f = Pod5File(path)
    assert len(f) == 4000
    g = golden_real
    off = g["adc_offsets"]
    for i, r in enumerate(f.reads()):
        if i >= 25:
            break
        assert r.read_id == str(g["read_ids"][i])
        s = r.signal
        assert s.size == r.num_samples and s.dtype == np.int16
        a = int(g["slice_start"][i])
        stored = g["adc"][off[i]:off[i + 1]]
        assert np.array_equal(s[a:a + stored.size], stored)
        assert r.signal_pa.dtype == np.float32


@pytest.mark.gpu
def test_gpu_chain_raw_signal_to_barcode_calls(golden_real, models):
    """BASELINE.json configs[0] end to end on the device: calibrated pA rows of the first reads of
    4000_rna004.pod5 -> boundary CNN -> boundary validation -> fingerprint -> DTW+SVC, against what the
    reference's own chain (combined_detect_cnn -> detect_results_to_fpt -> DTW_SVM.predict) produced for the
    same reads.  Reads whose validation fails are the reference's LLR-fallback reads (stay with the caller)."""
    from types import SimpleNamespace

    from conftest import GOLD
    from warpdemux_b200.detect import cnn, combined
    from warpdemux_b200.models.dtw_svm import DTW_SVM
    from warpdemux_b200.sig_proc import Fingerprinter, FingerprintConfig
    from wdx_testutil import cnn_golden_signals

    g = golden_real
    with np.load(os.path.join(GOLD, "cnn_detect_rna004.npz")) as z:
        gc = {k: z[k] for k in z.files}
    with np.load(os.path.join(GOLD, "validate_rna004.npz")) as z:
        full_lens = z["full_lens"][: int(z["n_real"])]
    m = int(g["preload_size"])            # production preload (parser.py:515 update_sig_preload_size): 11 500 samples
    sig = np.ascontiguousarray(cnn_golden_signals(gc)[:, :m])
    n = sig.shape[0]
    ccfg = json.loads(str(gc["cfg"]))
    spc = SimpleNamespace(core=cnn.CoreConfig(min_obs_adapter=ccfg["min_obs_adapter"], max_obs_adapter=ccfg["max_obs_adapter"],
                                              downscale_factor=ccfg["downscale_factor"]),
                          cnn_boundaries=cnn.CNNBoundariesConfig(polya_cand_k=ccfg["polya_cand_k"]), primary_method="cnn")
    model = cnn.load_cnn_model(os.path.join(GOLD, "models", "cnn_rna004_130bps_v0.2.4.npz"), device=0)
    val = combined.Validator(device=0)
    dets = combined.combined_detect_cnn(sig, full_lens, model, spc, validator=val)
    ok = np.array([d.success for d in dets])
    assert ok.sum() >= n - 3
    a0 = np.array([d.adapter_start if d.success else 0 for d in dets], dtype=np.int64)
    a1 = np.array([d.adapter_end if d.success else 0 for d in dets], dtype=np.int64)
    ref_ok = g["detect_ok"][:n].astype(bool)
    assert not (ok & ~ref_ok).any()                       # a read the CNN path validates is validated by the reference too
    assert np.array_equal(a0[ok], g["adapter_start"][:n][ok]) and np.array_equal(a1[ok], g["adapter_end"][:n][ok])
    assert dets[0].cnn_adapter_end == int(gc["preds"][0, 0])

    fp = Fingerprinter(FingerprintConfig(**_cfg(g)), device=0)
    mdl = DTW_SVM(models["WDX4_rna004_v1_0"], device=0, mode="guarded")
    labels, prob, conf, status = fp.extract_and_predict(mdl, sig, a0, a1, detect_ok=ok.astype(np.uint8))
    assert np.array_equal(status[ok], g["status"][:n][ok])
    good_all = g["status"] == 0
    pos = np.cumsum(good_all) - 1                         # row of y_pred for each read with a fingerprint
    chk = ok & good_all[:n]
    assert chk.sum() >= n - 5
    assert np.array_equal(labels[chk], g["y_pred"][pos[:n][chk]])
    fp.close()
    val.close()
    model.close()


@pytest.mark.gpu
def test_gpu_minibatch_step_matches_reference_worker(golden_real, models):
    """warpdemux_b200.file_proc.MinibatchDemuxer = the compute core of the reference's
    worker_detect_and_predict_on_preloaded_signals (file_proc.py:380-455) on the device; the reads the CNN path
    rejects get their boundaries from an `llr_fallback` callback (here: the reference's own results)."""
    from types import SimpleNamespace

    import torch

    from conftest import GOLD
    from warpdemux_b200.detect import cnn, combined
    from warpdemux_b200.file_proc import MinibatchDemuxer, detect_and_predict_on_preloaded_signals
    from warpdemux_b200.models.dtw_svm import DTW_SVM
    from warpdemux_b200.sig_proc import FingerprintConfig
    from wdx_testutil import cnn_golden_signals

    g = golden_real
    with np.load(os.path.join(GOLD, "cnn_detect_rna004.npz")) as z:
        gc = {k: z[k] for k in z.files}
    with np.load(os.path.join(GOLD, "validate_rna004.npz")) as z:
        full_lens = z["full_lens"][: int(z["n_real"])]
    m = int(g["preload_size"])
    sig = np.ascontiguousarray(cnn_golden_signals(gc)[:, :m])
    n = sig.shape[0]
    ccfg = json.loads(str(gc["cfg"]))
    core = cnn.CoreConfig(min_obs_adapter=ccfg["min_obs_adapter"], max_obs_adapter=ccfg["max_obs_adapter"],
                          downscale_factor=ccfg["downscale_factor"])
    model_detect = cnn.load_cnn_model(os.path.join(GOLD, "models", "cnn_rna004_130bps_v0.2.4.npz"), device=0)
    model_predict = DTW_SVM(models["WDX4_rna004_v1_0"], device=0, mode="guarded")
    read_ids = g["read_ids"][:n]
    calls = []

    def llr_fallback(row, full_len):
        # identify the read by its samples (rows are unique)
        i = next(j for j in range(n) if np.array_equal(sig[j], row, equal_nan=True))
        calls.append(i)
        if not g["detect_ok"][i]:
            return SimpleNamespace(success=False)
        return SimpleNamespace(success=True, adapter_start=int(g["adapter_start"][i]), adapter_end=int(g["adapter_end"][i]), polya_end=0)

    dmx = MinibatchDemuxer(model_predict, model_detect, core=core, cnn_boundaries=cnn.CNNBoundariesConfig(polya_cand_k=ccfg["polya_cand_k"]),
                           validate_config=combined.ValidateConfig(), fp_config=FingerprintConfig(**_cfg(g)), device=0,
                           llr_fallback=llr_fallback)
    res = dmx.run(sig, full_lens, read_ids, want_fpt=True)
    assert np.array_equal(res.fp_status, g["status"][:n])
    good_all = g["status"] == 0
    pos = np.cumsum(good_all) - 1
    good = good_all[:n]
    assert np.array_equal(res.labels[good], g["y_pred"][pos[:n][good]]) and (res.labels[~good] == -1).all()
    assert np.abs(res.prob[good] - g["y_prob"][pos[:n][good]]).max() < 1e-3
    assert np.array_equal(res.fpt[good], g["fpt"][:n][good])           # fingerprints bit-identical through the chain
    assert sorted(calls) == sorted(np.flatnonzero(res.detect_code != 0).tolist()) and res.llr_rescued.sum() == len(
        [i for i in calls if g["detect_ok"][i]])
    df = res.predictions
    assert list(df.columns[:3]) == ["#read_id", "predicted_barcode", "confidence_score"] and df.columns[-1] == "p-1"
    assert list(df["#read_id"]) == list(read_ids[good]) and np.array_equal(df["predicted_barcode"].to_numpy(), res.labels[good])
    # device-resident input, no callback, reference argument order
    dmx2 = MinibatchDemuxer(model_predict, model_detect, core=core, cnn_boundaries=cnn.CNNBoundariesConfig(polya_cand_k=ccfg["polya_cand_k"]),
                            fp_config=FingerprintConfig(**_cfg(g)), device=0)
    res2 = detect_and_predict_on_preloaded_signals((torch.from_numpy(sig).cuda(), None, full_lens, read_ids), model_predict, model_detect,
                                                   SimpleNamespace(primary_method="cnn"), demuxer=dmx2)
    ok2 = res2.detect_success.astype(bool)
    assert np.array_equal(res2.labels[ok2], res.labels[ok2]) and (res2.labels[~ok2] == -1).all()
    assert all(res2.fail_reason(i) == combined.fail_reason(int(res2.detect_code[i]), int(res2.detect_checks[i])) for i in np.flatnonzero(~ok2))
    # pipelined stream of minibatches (upload of i+1 overlaps the kernels of i) == one run() per minibatch
    cuts = [(0, 20), (20, 21), (21, n)]
    mbs = [(sig[a:b], full_lens[a:b], read_ids[a:b]) for a, b in cuts]
    streamed = list(dmx2.stream(mbs, want_fpt=True))
    assert len(streamed) == len(cuts)
    for (a, b), r_s in zip(cuts, streamed):
        r_1 = dmx2.run(sig[a:b], full_lens[a:b], read_ids[a:b], want_fpt=True)
        assert np.array_equal(r_s.labels, r_1.labels) and np.array_equal(r_s.fp_status, r_1.fp_status)
        assert np.array_equal(r_s.bounds, r_1.bounds) and np.array_equal(r_s.preds, r_1.preds)
        assert np.array_equal(r_s.fpt, r_1.fpt, equal_nan=True) and np.array_equal(r_s.prob, r_1.prob, equal_nan=True)
        assert list(r_s.predictions["#read_id"]) == list(r_1.predictions["#read_id"])
    assert list(dmx2.stream([])) == []
    dmx.close()
    dmx2.close()
    model_detect.close()


@pytest.mark.gpu
def test_gpu_minibatch_step_on_second_device(golden_real, models):
    """One process per GPU in production, but nothing in the chain may assume device 0: the same minibatch on cuda:1
    (when the box has one) gives the results of cuda:0."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from conftest import GOLD
    from warpdemux_b200.detect import cnn
    from warpdemux_b200.file_proc import MinibatchDemuxer
    from warpdemux_b200.models.dtw_svm import DTW_SVM
    from warpdemux_b200.sig_proc import FingerprintConfig
    from wdx_testutil import cnn_golden_signals

    g = golden_real
    with np.load(os.path.join(GOLD, "cnn_detect_rna004.npz")) as z:
        gc = {k: z[k] for k in z.files}
    with np.load(os.path.join(GOLD, "validate_rna004.npz")) as z:
        full_lens = z["full_lens"][: int(z["n_real"])]
    sig = np.ascontiguousarray(cnn_golden_signals(gc)[:, : int(g["preload_size"])])
    res = []
    for dev in (0, 1):
        md = cnn.load_cnn_model(os.path.join(GOLD, "models", "cnn_rna004_130bps_v0.2.4.npz"), device=dev)
        mp = DTW_SVM(models["WDX4_rna004_v1_0"], device=dev, mode="guarded")
        dmx = MinibatchDemuxer(mp, md, core=cnn.CoreConfig(), cnn_boundaries=cnn.CNNBoundariesConfig(polya_cand_k=5),
                               fp_config=FingerprintConfig(**_cfg(g)), device=dev)
        res.append(dmx.run(sig, full_lens, want_fpt=True))
        res.append(list(dmx.stream([(sig[:30], full_lens[:30]), (sig[30:], full_lens[30:])], return_df=False)))
        dmx.close()
        md.close()
    a, sa, b, sb = res
    assert np.array_equal(a.labels, b.labels) and np.array_equal(a.bounds, b.bounds) and np.array_equal(a.fpt, b.fpt, equal_nan=True)
    assert np.array_equal(np.concatenate([x.labels for x in sb]), b.labels)
    assert np.array_equal(np.concatenate([x.labels for x in sa]), a.labels)


@pytest.mark.gpu
def test_gpu_minibatch_step_from_raw_adc(golden_real, models):
    """AdcBatch input: int16 ADC samples + calibration instead of float32 pA rows (half the PCIe bytes); the rows made on
    the device are bit-identical to the host calibration, so every result is identical."""
    import torch

    from conftest import GOLD
    from warpdemux_b200 import _lib
    from warpdemux_b200.detect import cnn
    from warpdemux_b200.file_proc import AdcBatch, MinibatchDemuxer
    from warpdemux_b200.models.dtw_svm import DTW_SVM
    from warpdemux_b200.sig_proc import FingerprintConfig
    from wdx_testutil import cnn_golden_signals

    g = golden_real
    with np.load(os.path.join(GOLD, "cnn_detect_rna004.npz")) as z:
        gc = {k: z[k] for k in z.files}
    with np.load(os.path.join(GOLD, "validate_rna004.npz")) as z:
        full_lens = z["full_lens"][: int(z["n_real"])]
    m = int(g["preload_size"])
    sig = np.ascontiguousarray(cnn_golden_signals(gc)[:, :m])
    n = sig.shape[0]
    offs = gc["adc_offsets"]
    adc = np.full((n, m), -7, dtype=np.int16)                         # filler beyond the read must not matter
    num = np.zeros(n, dtype=np.int64)
    for i in range(n):
        row = gc["adc"][offs[i]:offs[i + 1]][:m]
        adc[i, : row.size] = row
        num[i] = row.size
    batch = AdcBatch(adc, num, gc["calibration_offset"], gc["calibration_scale"])
    # the calibration kernel alone
    d_adc = torch.from_numpy(adc).cuda()
    d_num = torch.from_numpy(num.astype(np.int32)).cuda()
    d_off, d_sc = torch.from_numpy(gc["calibration_offset"]).cuda(), torch.from_numpy(gc["calibration_scale"]).cuda()
    d_out = torch.empty((n, m), dtype=torch.float32, device="cuda")
    _lib.check(_lib.load().wdx_calibrate_rows(d_adc.data_ptr(), n, m, d_num.data_ptr(), d_off.data_ptr(), d_sc.data_ptr(), d_out.data_ptr(), m, 0,
                                              torch.cuda.current_stream().cuda_stream), "wdx_calibrate_rows")
    assert np.array_equal(d_out.cpu().numpy(), sig, equal_nan=True)
    with pytest.raises(ValueError):
        _lib.check(_lib.load().wdx_calibrate_rows(adc.ctypes.data, n, m, d_num.data_ptr(), d_off.data_ptr(), d_sc.data_ptr(), d_out.data_ptr(), m, 0, None), "x")
    # the whole step
    md = cnn.load_cnn_model(os.path.join(GOLD, "models", "cnn_rna004_130bps_v0.2.4.npz"), device=0)
    mp = DTW_SVM(models["WDX4_rna004_v1_0"], device=0, mode="guarded")
    dmx = MinibatchDemuxer(mp, md, core=cnn.CoreConfig(), cnn_boundaries=cnn.CNNBoundariesConfig(polya_cand_k=5),
                           fp_config=FingerprintConfig(**_cfg(g)), device=0)
    a = dmx.run(sig, full_lens, want_fpt=True)
    b = dmx.run(batch, full_lens, want_fpt=True)
    for f in ("labels", "fp_status", "bounds", "preds", "detect_code"):
        assert np.array_equal(getattr(a, f), getattr(b, f)), f
    assert np.array_equal(a.fpt, b.fpt, equal_nan=True) and np.array_equal(a.prob, b.prob, equal_nan=True)
    parts = list(dmx.stream([(AdcBatch(adc[:40], num[:40], batch.offset[:40], batch.scale[:40]), full_lens[:40]),
                             (AdcBatch(adc[40:], num[40:], batch.offset[40:], batch.scale[40:]), full_lens[40:])], return_df=False))
    assert np.array_equal(np.concatenate([p.labels for p in parts])[:40], dmx.run(sig[:40], full_lens[:40], return_df=False).labels)
    dmx.close()
    md.close()


@pytest.mark.gpu
def test_gpu_fingerprints_of_the_4000_read_subset_incl_score_ties(models):
    """Fingerprint + barcode call of the committed subset of tests/golden/real4000_rna004_WDX4.npz from the reference's own
    boundaries (incl. the long LLR adapters, which take the second, larger-capacity pass).  Reads where two EQUAL t-test
    scores compete inside the peak distance are ambiguous in the reference itself (numpy's unstable argsort decides);
    the kernel follows the stable order: expected values for those come from the oracle's stable_ties variant."""
    from warpdemux_b200.models.dtw_svm import DTW_SVM
    from warpdemux_b200.sig_proc import Fingerprinter, FingerprintConfig
    from wdx_testutil import real4000_rows

    with np.load(os.path.join(ROOT, "tests", "golden", "real4000_rna004_WDX4.npz")) as z:
        g = {k: z[k] for k in z.files}
    idx, rows, _, _ = real4000_rows(g)
    c = json.loads(str(g["cfg"]))
    cfg = {k: c[k] for k in ("padding", "outlier_thresh", "min_obs_per_base", "running_stat_width", "num_events", "barcode_num_events")}
    want_fpt = g["fpt"].copy()
    want_fpt[g["stable_idx"]] = g["stable_fpt"]
    assert g["stable_idx"].size >= 1 and set(g["stable_idx"].tolist()) <= set(idx.tolist())
    for kw in (dict(), dict(max_slice_len=6720, long_slice_len=10112)):
        fp = Fingerprinter(FingerprintConfig(**cfg, **kw), device=0)
        b = fp.extract(rows, g["bounds"][idx, 0], g["bounds"][idx, 1], detect_ok=g["success"][idx])
        assert np.array_equal(b.status, g["status"][idx]), kw
        good = g["status"][idx] == 0
        assert np.array_equal(b.fpt[good], want_fpt[idx][good]), kw
        assert (g["bounds"][idx, 1] - g["bounds"][idx, 0] > 6600)[good].sum() >= 5      # the long pass is exercised
        fp.close()
    fp = Fingerprinter(FingerprintConfig(max_slice_len=6720, **cfg), device=0)             # without the long pass they fail
    b = fp.extract(rows, g["bounds"][idx, 0], g["bounds"][idx, 1], detect_ok=g["success"][idx])
    assert (b.status == 4).sum() >= 5
    fp.close()


def test_oracle_stable_tie_rule_on_the_ambiguous_read():
    """The read of the 4000-read fixture whose change points depend on the order of two equal scores: numpy's default
    argsort reproduces the reference (same machine, same numpy) and the stable order gives the fixture's second answer."""
    from oracle import wdx_oracle as o
    from wdx_testutil import real4000_rows

    with np.load(os.path.join(ROOT, "tests", "golden", "real4000_rna004_WDX4.npz")) as z:
        g = {k: z[k] for k in z.files}
    idx, rows, _, _ = real4000_rows(g)
    c = json.loads(str(g["cfg"]))
    cfg = {k: c[k] for k in ("padding", "outlier_thresh", "min_obs_per_base", "running_stat_width", "num_events", "barcode_num_events")}
    for q, i in enumerate(g["stable_idx"]):
        j = int(np.flatnonzero(idx == i)[0])
        a0, a1 = int(g["bounds"][i, 0]), int(g["bounds"][i, 1])
        assert o.fingerprint_has_ties(rows[j], a0, a1, **cfg)
        st, f, _, _ = o.fingerprint(rows[j], a0, a1, stable_ties=True, **cfg)
        assert st == 0 and np.array_equal(f, g["stable_fpt"][q]) and not np.array_equal(f, g["fpt"][i])

"""The host-side batch loops in front of the kernels, at the sizes where they switch on.

Every kernel has a parity test at small batch sizes.  Production batches are cut into chunks that are double-buffered,
overlapped across streams and, in `MinibatchDemuxer.stream`, rotated over lanes and buffer slots.  A wrong row offset, a
buffer reused one chunk early or a lane with stale state gives wrong calls only at those sizes.  This file drives each
loop past its first chunk (through the batch size and the handles' chunk-size knobs) and compares with the float64 oracle
or the reference's own results on the rows next to every chunk edge, and with the same call made in one chunk on all rows.

- `wdx_predict`: the chunked loop with host, pinned, float32 and device inputs, with and without distances.
- `wdx_fp_extract_ex` / `wdx_fp_predict`: both staging buffers, device rows with host outputs, consensus batches whose
  chunks mix the parked three-launch form with the single-launch form.
- `wdx_cnn_detect`: device rows of several chunks (prepare / convolution / argmax on three streams) and the GUARDED re-runs.
- `MinibatchDemuxer.stream`: every lane and buffer slot reused, ragged minibatches of every input kind, a threshold change."""
import copy
import json
import os

import numpy as np
import pytest

from conftest import GOLD
from wdx_testutil import cnn_golden_signals, oracle_fingerprints, real4000_rows, real_fixture_rows, synth_adapter_signals, synth_fingerprints

pytestmark = pytest.mark.gpu

PROB_ATOL = 2e-6            # float32 exp of the kernel vs numpy's (test_gpu_predict.py)
CHUNK_READS = 1 << 22       # wdx_model's default chunk size
CNN_GUARD = 1e-3            # wdx_cnn's default guard band
PREDICT_MODELS = ("WDX4_rna004_v1_0", "WDX12_rna002_v0_4_4")


def _edges(n, chunk, k=3):
    """The first and last k rows of every chunk of `chunk` rows, and the last row."""
    idx = {n - 1}
    for r0 in range(0, n, chunk):
        r1 = min(n, r0 + chunk)
        idx.update(range(r0, min(r1, r0 + k)))
        idx.update(range(max(r0, r1 - k), r1))
    return np.array(sorted(idx), dtype=np.int64)


def _labels_match_oracle(labels, want_pred, want_prob, want_conf, thresholds):
    """Labels identical except where the oracle's confidence is within float32-exp noise of its threshold."""
    diff = labels != want_pred
    if diff.any():
        thr = thresholds[np.argmax(want_prob, 1)]
        assert np.all(np.minimum(np.abs(want_conf - thr), want_conf)[diff] < 4 * PROB_ATOL), np.flatnonzero(diff)


# ----------------------------------------------------------------------------------------------------------------------
# A. wdx_predict's chunk loop
# ----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev_models(models):
    from warpdemux_b200.device_model import DeviceModel

    out = {n: DeviceModel(models[n], 0) for n in PREDICT_MODELS}
    yield out
    for d in out.values():
        d.close()


def _predict_raw(d, X, mode, kind, dist=True):
    """wdx_predict with the input as `kind`: 'pageable' / 'f32' (numpy), 'pinned' (torch), 'cuda' (CUDA tensor, host
    outputs) or 'device' (CUDA tensor, device outputs).  Returns numpy (labels, prob, conf, flags, dist or None)."""
    import torch

    from warpdemux_b200 import _lib

    n, k, nsv = X.shape[0], d.params.k, d.params.n_sv
    xd = _lib.WDX_F32 if X.dtype == np.float32 else _lib.WDX_F64
    Xin = np.ascontiguousarray(X)
    if kind == "pinned":
        Xin = torch.from_numpy(Xin).pin_memory()
    elif kind in ("cuda", "device"):
        Xin = torch.from_numpy(Xin).cuda()
    dev = "cuda" if kind == "device" else "cpu"
    lab = torch.empty(n, dtype=torch.int64, device=dev)
    conf = torch.empty(n, dtype=torch.float64, device=dev)
    prob = torch.empty((n, k), dtype=torch.float64, device=dev)
    flags = torch.zeros(n, dtype=torch.uint8, device=dev)
    D = torch.empty((n, nsv), dtype=torch.float32, device=dev) if dist else None
    torch.cuda.synchronize()
    st = torch.cuda.current_stream().cuda_stream if kind == "device" else 0
    d.predict_raw(Xin, n, xd, _lib.MODES[mode], lab, conf, prob, flags, D, stream=st)
    torch.cuda.synchronize()
    return tuple(None if t is None else t.cpu().numpy() for t in (lab, prob, conf, flags, D))


def _same_as_one_chunk(got, ref, where):
    lab, prob, conf, flags, dist = got
    assert np.array_equal(lab, ref[0]), (where, np.flatnonzero(lab != ref[0])[:10])
    # choose_splits depends on the chunk size: the SVC sums may associate differently
    assert np.abs(prob - ref[1]).max() <= 1e-12, where
    assert np.abs(conf - ref[2]).max() <= 1e-12, where
    assert np.array_equal(flags, ref[3]), where
    if dist is not None:
        assert np.array_equal(dist, ref[4]), (where, np.argwhere(dist != ref[4])[:5])


@pytest.mark.parametrize("name", PREDICT_MODELS)
def test_chunked_predict_matches_one_chunk_and_oracle(models, dev_models, name):
    """9 000 reads (past the one-copy small path) in chunks of 1 000, 4 097 and 8 999 reads, for every input kind: EXACT
    distances bit-identical to the oracle on the chunk-edge rows and to the one-chunk call everywhere, probabilities
    within PROB_ATOL of the oracle and 1e-12 of the one-chunk call, labels and FAST distances identical."""
    from oracle import wdx_oracle as o

    m, d = models[name], dev_models[name]
    n = 9000
    chunks = (1000, 4097, 8999)
    X = synth_fingerprints(m.sv, n, seed=31)
    X32 = X.astype(np.float32)
    edges = np.unique(np.concatenate([_edges(n, c) for c in chunks]))
    oracle = {"f64": o.predict(m, X[edges]), "f32": o.predict(m, X32.astype(np.float64)[edges])}
    ref = {"f64": d.predict(X, mode="exact", want_dist=True), "f32": d.predict(X32, mode="exact", want_dist=True),
           "fast": d.predict(X, mode="fast", want_dist=True)}
    for key in ("f64", "f32"):   # the one-chunk call itself against the oracle
        labels, prob, conf, flags, dist = ref[key]
        want_pred, want_prob, want_conf, want_D = oracle[key]
        assert np.array_equal(dist[edges], want_D)
        np.testing.assert_allclose(prob[edges], want_prob, rtol=0, atol=PROB_ATOL)
        _labels_match_oracle(labels[edges], want_pred, want_prob, want_conf, m.thresholds)
    try:
        for c in chunks:
            d.set_chunk_reads(c)
            for kind in ("pageable", "pinned", "f32", "cuda", "device"):
                key = "f32" if kind == "f32" else "f64"
                got = _predict_raw(d, X32 if kind == "f32" else X, "exact", kind)
                _same_as_one_chunk(got, ref[key], (c, kind))
                want_pred, want_prob, _, want_D = oracle[key]
                assert np.array_equal(got[4][edges], want_D), (c, kind)
                np.testing.assert_allclose(got[1][edges], want_prob, rtol=0, atol=PROB_ATOL)
            # host buffers without distances: the chunk loop of the plain host path
            got = d.predict(X, mode="exact")
            _same_as_one_chunk(got + (None,), ref["f64"], (c, "no dist"))
            # FAST: distances are per pair and do not depend on the chunk
            _same_as_one_chunk(d.predict(X, mode="fast", want_dist=True), ref["fast"], (c, "fast"))
    finally:
        d.set_chunk_reads(CHUNK_READS)


def test_distances_one_read_per_chunk(models, dev_models):
    """With distances asked for, even a live-sized batch takes the chunk loop: 300 chunks of one read."""
    from oracle import wdx_oracle as o

    for name in PREDICT_MODELS:
        m, d = models[name], dev_models[name]
        X = synth_fingerprints(m.sv, 300, seed=32)
        want_pred, want_prob, want_conf, want_D = o.predict(m, X)
        ref = d.predict(X, mode="exact", want_dist=True)
        d.set_chunk_reads(1)
        try:
            got = d.predict(X, mode="exact", want_dist=True)
            got_dev = _predict_raw(d, X, "exact", "device")
        finally:
            d.set_chunk_reads(CHUNK_READS)
        for g in (got, got_dev):
            _same_as_one_chunk(g, ref, name)
            assert np.array_equal(g[4], want_D)
            np.testing.assert_allclose(g[1], want_prob, rtol=0, atol=PROB_ATOL)
            _labels_match_oracle(g[0], want_pred, want_prob, want_conf, m.thresholds)


def test_guarded_overflow_in_some_chunks(models, dev_models):
    """GUARDED with every read inside the guard band, 12 000 reads in chunks of 5 000: the 4 096-entry re-run list of the
    first two chunks overflows, the last chunk's does not.  The overflowed reads are redone on the host side and carry
    FLAG_RECOMPUTED; labels equal EXACT."""
    from warpdemux_b200 import _lib

    m, d = models["WDX4_rna004_v1_0"], dev_models["WDX4_rna004_v1_0"]
    n = 12000
    X = synth_fingerprints(m.sv, n, seed=33)
    le, pe, ce, _ = d.predict(X, mode="exact")
    d.set_chunk_reads(5000)
    d.set_guard(10.0)
    try:
        lab, conf, prob = np.empty(n, np.int64), np.empty(n, np.float64), np.empty((n, m.k), np.float64)
        flags = np.zeros(n, np.uint8)
        d.predict_raw(X, n, _lib.WDX_F64, _lib.MODE_FAST_F32_GUARDED, lab, conf, prob, flags)
        over = (flags & _lib.FLAG_GUARD_OVERFLOW) != 0
        assert [int(over[r0:r0 + 5000].sum()) for r0 in (0, 5000, 10000)] == [5000 - 4096, 5000 - 4096, 0]
        # what was listed was redone in EXACT_F64 on the device
        assert np.all((flags[~over] & _lib.FLAG_RECOMPUTED) != 0)
        assert np.array_equal(lab[~over], le[~over])
        lg, pg, cg, fg = d.predict(X, mode="guarded")
    finally:
        d.set_guard(5e-5)
        d.set_chunk_reads(CHUNK_READS)
    assert np.all((fg & _lib.FLAG_RECOMPUTED) != 0) and not np.any(fg & _lib.FLAG_GUARD_OVERFLOW)
    assert np.array_equal(lg, le)
    np.testing.assert_allclose(pg, pe, rtol=0, atol=1e-12)
    np.testing.assert_allclose(cg, ce, rtol=0, atol=1e-12)


# ----------------------------------------------------------------------------------------------------------------------
# B. the fingerprint stage's chunk loop
# ----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def synth300():
    sig, a0, a1 = synth_adapter_signals(300, seed=61, width=9000)
    status, fpt, dwell, stats = oracle_fingerprints(sig, a0, a1)
    assert (status == 0).sum() > 250 and (status != 0).any()
    return dict(sig=sig, a0=a0, a1=a1, status=status, fpt=fpt, dwell=dwell, stats=stats)


@pytest.fixture(scope="module")
def fp():
    from warpdemux_b200.sig_proc import Fingerprinter

    f = Fingerprinter(device=0)
    yield f
    f.close()


def _check_calls(s, labels, prob, conf, status, fpt, want_pred, want_prob, mode, where):
    """Bars of test_gpu_fingerprint.test_fused_extract_and_predict."""
    ok = s["status"] == 0
    assert np.array_equal(status, s["status"]), where
    assert np.array_equal(fpt[ok], s["fpt"][ok]), where
    assert np.array_equal(labels[ok], want_pred), (where, np.flatnonzero(labels[ok] != want_pred))
    assert np.abs(prob[ok] - want_prob).max() < (2e-6 if mode == "exact" else 1e-3), where
    assert (labels[~ok] == -1).all() and np.isnan(conf[~ok]).all(), where


def test_chunked_extract_and_predict(models, fp, synth300):
    """The fused step in chunks of 1, 37 and 299 reads (the model's chunk size bounds the fingerprint chunk), host rows
    (staged) and device rows with host outputs (the branch that synchronises between chunks)."""
    import torch

    from oracle import wdx_oracle as o
    from warpdemux_b200 import _lib
    from warpdemux_b200.models.dtw_svm import DTW_SVM

    s = synth300
    m = models["WDX4_rna004_v1_0"]
    ok = s["status"] == 0
    want_pred, want_prob, _, _ = o.predict(m, s["fpt"][ok])
    n, stride = s["sig"].shape
    d_sig = torch.from_numpy(s["sig"]).cuda()
    d_a0, d_a1 = torch.from_numpy(s["a0"]).cuda(), torch.from_numpy(s["a1"]).cuda()
    torch.cuda.synchronize()
    for mode in ("exact", "guarded"):
        mdl = DTW_SVM(m, device=0, mode=mode)
        dm = mdl._device_model()
        try:
            for chunk in (1, 37, 299):
                dm.set_chunk_reads(chunk)
                labels, prob, conf, status, fpt = fp.extract_and_predict(mdl, s["sig"], s["a0"], s["a1"], want_fpt=True)
                _check_calls(s, labels, prob, conf, status, fpt, want_pred, want_prob, mode, (mode, chunk, "host rows"))
                lab = np.full(n, -1, np.int64)
                cf, pr = np.full(n, np.nan), np.full((n, m.k), np.nan)
                fl, st = np.zeros(n, np.uint8), np.zeros(n, np.int32)
                fpt2 = np.full((n, 25), np.nan)
                fp.predict_raw(dm, d_sig, n, stride, d_a0, d_a1, _lib.MODES[mode], lab, st, conf=cf, prob=pr, flags=fl, fpt=fpt2)
                assert not (fl & _lib.FLAG_GUARD_OVERFLOW).any()
                _check_calls(s, lab, pr, cf, st, fpt2, want_pred, want_prob, mode, (mode, chunk, "device rows"))
                assert np.array_equal(lab, labels) and np.array_equal(pr, prob, equal_nan=True)
        finally:
            dm.set_chunk_reads(CHUNK_READS)
            mdl._drop_device()


def test_extract_in_two_staging_pieces(fp, synth300):
    """7 800 host rows of stride 9 000 are staged in two 256 MB pieces (7 456 + 344 rows): every output equals the tiled
    oracle bit for bit, and the in-place winsorisation lands in the right rows."""
    s = synth300
    reps = 26
    tile = lambda x: np.concatenate([x] * reps, axis=0)
    big = tile(s["sig"])
    assert big.shape[0] > ((256 << 20) // (big.shape[1] * 4))
    a0, a1 = tile(s["a0"]), tile(s["a1"])
    status, fpt, dwell, stats = tile(s["status"]), tile(s["fpt"]), tile(s["dwell"]), tile(s["stats"])
    ok = status == 0
    b = fp.extract(big, a0, a1)
    assert np.array_equal(b.status, status), np.flatnonzero(b.status != status)[:10]
    assert np.array_equal(b.dwell[ok], dwell[ok])
    assert np.array_equal(b.fpt[ok], fpt[ok]) and np.isnan(b.fpt[~ok]).all()
    assert np.array_equal(b.stats[ok], stats[ok])
    clipped = s["sig"].copy()
    fp.extract(clipped, s["a0"], s["a1"], clip_in_place=True)       # one chunk
    assert not np.array_equal(clipped, s["sig"], equal_nan=True)
    b2 = fp.extract(big, a0, a1, clip_in_place=True)
    assert np.array_equal(big, tile(clipped), equal_nan=True)
    assert np.array_equal(b2.status, status) and np.array_equal(b2.fpt[ok], fpt[ok])


def test_trna_parked_and_single_launch_chunks_in_one_call(models, golden_real):
    """Consensus fingerprints of 4 500 reads in chunks of 2 100: two chunks in the parked three-launch form (>= 2 048
    reads), then one of 300 in the single-launch form.  Status and fingerprints equal the tiled golden values."""
    from test_gpu_trna import make_fp

    from warpdemux_b200.models.dtw_svm import DTW_SVM

    with np.load(os.path.join(GOLD, "fingerprint_trna.npz")) as z:
        g = {k: z[k] for k in z.files}
    rows = real_fixture_rows(golden_real)
    reps = 9
    tile = lambda x: np.concatenate([x] * reps, axis=0)
    big = tile(rows)
    assert big.shape[0] == 4500
    a0, a1, det = tile(golden_real["adapter_start"]), tile(golden_real["adapter_end"]), tile(golden_real["detect_ok"])
    f, _ = make_fp(g)
    mdl = DTW_SVM(models["WDX4_rna004_v1_0"], device=0, mode="exact")
    dm = mdl._device_model()
    ok1 = g["real_status"] == 0
    want_lab, _, _, _ = dm.predict(g["real_fpt"][ok1], mode="exact")
    dm.set_chunk_reads(2100)
    try:
        labels, prob, conf, status, fpt = f.extract_and_predict(mdl, big, a0, a1, detect_ok=det, want_fpt=True)
    finally:
        dm.set_chunk_reads(CHUNK_READS)
        f.close()
        mdl._drop_device()
    want_status = tile(g["real_status"])
    ok = want_status == 0
    assert np.array_equal(status, want_status), np.flatnonzero(status != want_status)[:10]
    assert np.array_equal(fpt[ok], tile(g["real_fpt"])[ok])
    assert np.array_equal(labels[ok], tile(want_lab)) and (labels[~ok] == -1).all()


# ----------------------------------------------------------------------------------------------------------------------
# C. the boundary CNN on device rows of several chunks
# ----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cnn_setup():
    from oracle import wdx_oracle_cnn as oc
    from warpdemux_b200.detect import cnn

    with np.load(os.path.join(GOLD, "cnn_detect_rna004.npz")) as z:
        gold = {k: z[k] for k in z.files}
    ocfg = oc.CnnConfig(**json.loads(str(gold["cfg"])))
    path = os.path.join(GOLD, "models", "cnn_rna004_130bps_v0.2.4.npz")
    model = cnn.load_cnn_model(path, device=0)
    core = cnn.CoreConfig(min_obs_adapter=ocfg.min_obs_adapter, max_obs_adapter=ocfg.max_obs_adapter,
                          downscale_factor=ocfg.downscale_factor)
    base = cnn_golden_signals(gold)
    rng = np.random.default_rng(71)
    reps = -(-4500 // base.shape[0])
    sig = np.concatenate([base + rng.standard_normal(base.shape).astype(np.float32) * np.float32(0.3 + 0.02 * r) for r in range(reps)])
    yield dict(ocfg=ocfg, weights=oc.load_weights_npz(path), model=model, core=core, k=int(ocfg.polya_cand_k), sig=sig)
    model.close()


def _cnn_call(c, sig, mode, where, scores):
    """wdx_cnn_detect with the rows `where` ('host': numpy, 'device': CUDA tensor with device preds / flags) and scores
    None, 'host' or 'device' -> numpy (preds, flags, scores or None)."""
    import torch

    from warpdemux_b200.detect import cnn

    n, stride = sig.shape
    _, t_out = cnn.score_len(c["model"], c["core"], c["k"], stride)
    if where == "host":
        preds, flags = np.zeros((n, 1 + c["k"]), np.int64), np.zeros(n, np.uint8)
        sc = None if scores is None else np.zeros((n, 2, t_out), np.float32)
        cnn.detect_raw(c["model"], c["core"], c["k"], sig, n, stride, preds, scores=sc, flags=flags, mode=mode)
        return preds, flags, sc
    d_sig = torch.from_numpy(sig).cuda()
    preds = torch.zeros((n, 1 + c["k"]), dtype=torch.int64, device="cuda")
    flags = torch.zeros(n, dtype=torch.uint8, device="cuda")
    sc = None
    if scores == "device":
        sc = torch.zeros((n, 2, t_out), dtype=torch.float32, device="cuda")
    elif scores == "host":
        sc = np.zeros((n, 2, t_out), np.float32)
    torch.cuda.synchronize()
    cnn.detect_raw(c["model"], c["core"], c["k"], d_sig, n, stride, preds, scores=sc, flags=flags, mode=mode,
                   stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    sc = None if sc is None else (sc if isinstance(sc, np.ndarray) else sc.cpu().numpy())
    return preds.cpu().numpy(), flags.cpu().numpy(), sc


@pytest.mark.parametrize("n", [1025, 2600, 4500])
def test_cnn_device_rows_past_one_chunk(cnn_setup, n):
    """Device rows of more than 1 024 reads take the overlapped path (prepare / convolution / argmax on three streams,
    scores alternating between two buffers): preds, flags and scores bit-identical to the same call on host rows, which
    takes the one-stream path; on the chunk-edge rows the boundaries equal the oracle's."""
    from oracle import wdx_oracle_cnn as oc

    c = cnn_setup
    sig = np.ascontiguousarray(c["sig"][:n])
    edges = _edges(n, 1024)
    with np.errstate(all="ignore"):
        want_scores = oc.cnn_scores(oc.prepare_data(sig[edges], c["ocfg"]), c["weights"])
    want = oc.cnn_detect_from_scores(want_scores, c["ocfg"])
    for mode in ("exact", "fast", "guarded"):
        hp, hf, hs = _cnn_call(c, sig, mode, "host", "host")
        for scores in ("device", None):
            dp, df, ds = _cnn_call(c, sig, mode, "device", scores)
            assert np.array_equal(dp, hp), (mode, scores, np.flatnonzero((dp != hp).any(axis=1))[:10])
            assert np.array_equal(df, hf), (mode, scores)
            if scores:
                assert np.array_equal(ds, hs), (mode, np.argwhere(ds != hs)[:5])
        if mode != "fast":      # FAST may differ at near-ties; GUARDED removes them
            assert np.array_equal(hp[edges], want), (mode, edges[(hp[edges] != want).any(axis=1)])
        tol = 2e-5 * max(1.0, float(np.abs(want_scores).max()))    # float32 summation order vs torch's CPU convolution
        assert np.abs(hs[edges] - want_scores).max() <= tol, mode


@pytest.mark.parametrize("n", [2600, 4500])
def test_cnn_guarded_redo_of_every_read(cnn_setup, n):
    """A guard band that holds every read: GUARDED re-runs all of them in EXACT_F32 and must equal EXACT bit for bit,
    through the asynchronous re-run (device scores, <= 4 096 reads), the host-count re-run in pieces of 1 024 rows
    (> 4 096 reads) and the row-by-row patch of host scores."""
    from warpdemux_b200 import _lib
    from warpdemux_b200.detect import cnn

    c = cnn_setup
    sig = np.ascontiguousarray(c["sig"][:n])
    h = c["model"]._handle(c["core"], c["k"])
    calls = [("device", "device"), ("device", None), ("host", "host"), ("device", "host")]
    ref = {cl: _cnn_call(c, sig, "exact", *cl) for cl in calls}
    _lib.check(_lib.load().wdx_cnn_set_guard(h, 1e30), "wdx_cnn_set_guard")
    try:
        got = {cl: _cnn_call(c, sig, "guarded", *cl) for cl in calls}
    finally:
        _lib.check(_lib.load().wdx_cnn_set_guard(h, CNN_GUARD), "wdx_cnn_set_guard")
    for cl in calls:
        (pe, fe, se), (pg, fg, sg) = ref[cl], got[cl]
        assert np.all((fg & cnn.FLAG_RECOMPUTED) != 0), cl
        assert np.array_equal(pg, pe), (cl, np.flatnonzero((pg != pe).any(axis=1))[:10])
        if se is not None:
            assert np.array_equal(sg, se), (cl, np.argwhere(sg != se)[:5])
    assert np.array_equal(ref[calls[0]][0], ref[calls[2]][0]) and np.array_equal(ref[calls[0]][2], ref[calls[2]][2])


# ----------------------------------------------------------------------------------------------------------------------
# D / E. MinibatchDemuxer.stream over every lane and buffer slot
# ----------------------------------------------------------------------------------------------------------------------
FIELDS = ("labels", "conf", "prob", "fp_status", "detect_success", "detect_code", "detect_checks", "bounds", "preds", "llr_rescued",
          "fpt", "detect_source")
# 12 minibatches over the 439 committed reads: more than twice the 6 buffer slots of 4 lanes, sizes that grow and shrink
RAGGED = (1, 64, 7, 200, 33, 2, 41, 9, 3, 30, 45, 4)
KINDS = ("numpy", "pinned", "cuda", "adc", "vbz")


@pytest.fixture(scope="module")
def chain4000():
    from test_gpu_llr import _fp_cfg, _llr_cfg, _spc, whole_file_expectations

    from warpdemux_b200.detect import cnn

    with np.load(os.path.join(GOLD, "real4000_rna004_WDX4.npz")) as z:
        g = dict(z)
    idx, rows, adc, num = real4000_rows(g)
    assert sum(RAGGED) == idx.size
    md = cnn.load_cnn_model(os.path.join(GOLD, "models", "cnn_rna004_130bps_v0.2.4.npz"), device=0)
    yield dict(g=g, idx=idx, rows=rows, adc=adc, num=num, want=whole_file_expectations(g, idx), md=md, spc=_spc(g),
               fp_cfg=_fp_cfg(g), llr=_llr_cfg(g))
    md.close()


def _demuxer(c, mp, lanes, overlap):
    from warpdemux_b200.detect import combined
    from warpdemux_b200.file_proc import MinibatchDemuxer
    from warpdemux_b200.sig_proc import FingerprintConfig

    return MinibatchDemuxer(mp, c["md"], core=c["spc"].core, cnn_boundaries=c["spc"].cnn_boundaries,
                            validate_config=combined.ValidateConfig(), fp_config=FingerprintConfig(**c["fp_cfg"]), device=0,
                            llr=c["llr"], full_detect_report=True, lanes=lanes, overlap_llr_tail=overlap)


def _minibatch(c, pos, kind):
    """(signals, full_lengths, read_ids) of the subset rows `pos` as the input kind `kind`."""
    import torch

    from vbz_testutil import make_vbz_batch

    from warpdemux_b200.file_proc import AdcBatch

    w = c["want"]
    full, ids = w["full_lengths"][pos], w["read_ids"][pos]
    off, sc = w["calibration_offset"][pos], w["calibration_scale"][pos]
    if kind == "numpy":
        sig = c["rows"][pos]
    elif kind == "pinned":
        sig = torch.from_numpy(c["rows"][pos]).pin_memory()
    elif kind == "cuda":
        sig = torch.from_numpy(c["rows"][pos]).cuda()
    elif kind == "adc":
        sig = AdcBatch(c["adc"][pos], c["num"][pos], off, sc)
    else:
        sig = make_vbz_batch([[a[:k]] for a, k in zip(c["adc"][pos], c["num"][pos])], off, sc, c["adc"].shape[1], level=1)
    return sig, full, ids


def _ragged(c, shift=0):
    out, lo = [], 0
    for i, size in enumerate(RAGGED):
        out.append(_minibatch(c, np.arange(lo, lo + size), KINDS[(i + shift) % len(KINDS)]))
        lo += size
    return out


def _same_result(a, b, where):
    for f in FIELDS:
        assert np.array_equal(getattr(a, f), getattr(b, f), equal_nan=True), (where, f)
    assert a.predictions.equals(b.predictions), where


@pytest.mark.parametrize("lanes", [1, 2, 4])
@pytest.mark.parametrize("overlap", [True, False])
def test_stream_reuses_every_lane_and_slot(models, chain4000, lanes, overlap):
    """12 ragged minibatches of every input kind through `stream`: each result equals `run` of the same minibatch, and
    together they equal the reference chain's whole-file results."""
    from test_gpu_llr import chain_mismatches

    from warpdemux_b200.models.dtw_svm import DTW_SVM

    c = chain4000
    dmx = _demuxer(c, DTW_SVM(models["WDX4_rna004_v1_0"], device=0, mode="guarded"), lanes, overlap)
    try:
        mbs = _ragged(c, shift=lanes)
        got = list(dmx.stream(mbs, want_fpt=True))
        assert len(got) == len(mbs) and len(dmx._lane_objs) == lanes
        for i, (mb, r) in enumerate(zip(mbs, got)):
            _same_result(dmx.run(*mb, want_fpt=True), r, (i, KINDS[(i + lanes) % len(KINDS)]))
        assert chain_mismatches(c["want"], got) == {}
    finally:
        dmx.close()


def test_stream_of_tiled_minibatches(models, chain4000):
    """Single minibatches of 1 317 and 4 500 rows (the reads tiled) take the CNN's overlapped path and, past 4 096 reads,
    its host-count GUARDED re-run inside the chain."""
    from test_gpu_llr import chain_mismatches

    from warpdemux_b200.models.dtw_svm import DTW_SVM

    c = chain4000
    m = c["idx"].size
    dmx = _demuxer(c, DTW_SVM(models["WDX4_rna004_v1_0"], device=0, mode="guarded"), 4, True)
    try:
        pos = [np.arange(1317) % m, np.arange(4500) % m]
        mbs = [_minibatch(c, pos[0], "numpy"), _minibatch(c, pos[1], "adc")]
        got = list(dmx.stream(mbs, want_fpt=True))
        for p, mb, r in zip(pos, mbs, got):
            _same_result(dmx.run(*mb, want_fpt=True), r, p.size)
            want = {k: v[p] for k, v in c["want"].items()}
            assert chain_mismatches(want, [r]) == {}, p.size
    finally:
        dmx.close()


def test_threshold_change_reaches_every_lane(models, chain4000):
    """Lanes 1-3 hold replicas built from lane 0's params.  After `model_predict.thresholds` is replaced, every lane must
    call with the new thresholds: labels equal `run` and the oracle on the returned fingerprints."""
    from oracle import wdx_oracle as o
    from warpdemux_b200.models.dtw_svm import DTW_SVM

    c = chain4000
    params = copy.deepcopy(models["WDX4_rna004_v1_0"])
    mp = DTW_SVM(params, device=0, mode="guarded")
    dmx = _demuxer(c, mp, 4, True)
    try:
        mbs = _ragged(c)
        first = list(dmx.stream(mbs, want_fpt=True))
        assert len(dmx._lane_objs) == 4
        good = np.concatenate([r.fp_status for r in first]) == 0
        conf = np.concatenate([r.conf for r in first])
        fpt = np.concatenate([r.fpt for r in first])[good]
        before = copy.deepcopy(params)
        mp.thresholds = np.full(params.k, np.quantile(conf[good], 0.6))
        assert params.thresholds is mp.thresholds
        # the new thresholds change at least a fifth of the oracle's calls
        assert (o.predict(before, fpt)[0] != o.predict(params, fpt)[0]).mean() >= 0.2
        second = list(dmx.stream(mbs, want_fpt=True))
        for i, (mb, r) in enumerate(zip(mbs, second)):
            ref = dmx.run(*mb, want_fpt=True)
            assert np.array_equal(r.labels, ref.labels), (i, i % 4)
            ok = r.fp_status == 0
            if ok.any():
                want_pred, want_prob, want_conf, _ = o.predict(params, r.fpt[ok])
                _labels_match_oracle(r.labels[ok], want_pred, want_prob, want_conf, params.thresholds)
            assert (r.labels[~ok] == -1).all()
    finally:
        dmx.close()

"""pod5 VBZ decoding on the device (csrc/wdx_vbz.cu): the zstd frame decoder against pyarrow byte for byte, the
streamvbyte-16 rows against io.pod5_min.decode_vbz, malformed frames as status codes, and the whole minibatch step fed
with compressed chunks against the same reads as raw ADC rows."""
import os

import numpy as np
import pytest

from conftest import GOLD
from vbz_testutil import (ST, corpus, frame_modes, hand_frames, make_vbz_batch, malformed_frames, svb16_encode, synth_signal,
                          vbz_encode, write_pod5, zstd_decompress)
from wdx_testutil import real4000_rows

pytestmark = pytest.mark.gpu

CLAIMED_MODES = {"single_segment", "window_descriptor", "fcs", "no_fcs", "block_raw", "block_rle", "block_compressed",
                 "lit_raw", "lit_rle", "lit_huf1", "lit_huf4", "lit_treeless"} | {
                    f"seq_{c}_{m}" for c in ("LL", "OF", "ML") for m in ("predefined", "rle", "fse", "repeat")}


def test_gpu_zstd_matches_pyarrow_full_and_prefix():
    from warpdemux_b200.vbz import zstd_decompress as dev_decompress

    frames = corpus() + [(f, raw) for _, f, raw in hand_frames()]
    modes = set()
    for f, raw in frames:
        modes |= set(frame_modes(f))
        assert zstd_decompress(f) == raw
    assert CLAIMED_MODES <= modes, CLAIMED_MODES - modes
    full = dev_decompress([f for f, _ in frames], capacities=[len(r) for _, r in frames])
    for i, ((st, out), (_, raw)) in enumerate(zip(full, frames)):
        assert st == 0 and out == raw, (i, st, len(out), len(raw))
    rng = np.random.default_rng(11)
    lims = [int(rng.integers(0, len(r) + 1)) for _, r in frames]
    pre = dev_decompress([f for f, _ in frames], limits=lims, capacities=[x + 7 for x in lims])
    for (st, out), (_, raw), lim in zip(pre, frames, lims):
        assert st == 0 and out == raw[:lim]


def test_gpu_zstd_malformed_frames_give_their_status():
    from warpdemux_b200.vbz import zstd_decompress as dev_decompress

    raw = svb16_encode(synth_signal(np.random.default_rng(0), 5000, 20))
    good = vbz_encode(synth_signal(np.random.default_rng(0), 5000, 20))
    cases = malformed_frames(good)
    res = dev_decompress([f for _, f, _ in cases] + [good, good], capacities=[len(raw) + 10] * len(cases) + [len(raw) - 1, len(raw)])
    for (name, _, want), (st, _) in zip(cases, res):
        assert st == want, name
    assert res[-2][0] == ST["TOO_LARGE"] and res[-1] == (0, raw)


def _chunked_reads(rng, n, stride):
    """Reads of every shape the row decoder meets: multi-chunk, shorter / longer than stride, empty chunks, +-30000 jumps."""
    reads = []
    for k in range(n):
        length = int(rng.choice([0, 1, 7, 300, stride - 1, stride, stride + 1, 3 * stride]))
        x = synth_signal(rng, length, 20).astype(np.int32)
        if k % 3 == 0 and length > 4:
            j = rng.integers(1, length, 4)
            x[j] += rng.choice([-30000, 30000], 4)
        x = ((x + 32768) % 65536 - 32768).astype(np.int16)
        cuts = sorted(rng.integers(0, length + 1, int(rng.integers(0, 4))).tolist())
        reads.append([x[a:b] for a, b in zip([0] + cuts, cuts + [length])])
    return reads


def test_gpu_vbz_rows_match_decode_vbz():
    import torch

    from warpdemux_b200.io.pod5_min import decode_vbz
    from warpdemux_b200.vbz import decode_rows

    rng = np.random.default_rng(5)
    stride = 2500
    reads = _chunked_reads(rng, 160, stride)
    batch = make_vbz_batch(reads, rng.normal(0, 5, len(reads)), rng.uniform(0.1, 0.3, len(reads)), stride, level=3)
    rows, nv, st = decode_rows(batch, device=0)
    torch.cuda.synchronize()
    rows, nv, st = rows.cpu().numpy(), nv.cpu().numpy(), st.cpu().numpy()
    assert not st.any()
    for r, chunks in enumerate(reads):
        parts = []
        for c in range(batch.read_chunks[r], batch.read_chunks[r + 1]):
            b = batch.data[batch.chunk_offsets[c]:batch.chunk_offsets[c + 1]].tobytes()
            parts.append(decode_vbz(b, int(batch.chunk_samples[c])))
        want = np.concatenate(parts)[:stride] if parts else np.zeros(0, np.int16)
        assert nv[r] == want.size == min(sum(len(c) for c in chunks), stride)
        assert np.array_equal(rows[r, :want.size], want) and not rows[r, want.size:].any(), r


def test_gpu_vbz_bad_chunks_fail_their_read_only():
    import torch

    from warpdemux_b200 import _lib
    from warpdemux_b200.vbz import decode_rows, zstd_decompress_raw

    rng = np.random.default_rng(9)
    stride = 3000
    good_sig = [synth_signal(rng, 2000, 20) for _ in range(12)]
    good = vbz_encode(good_sig[0])
    bad = [f for _, f, _ in malformed_frames(good)] + [vbz_encode(np.zeros(100, np.int16)) for _ in range(2)]
    want_st = [w for _, _, w in malformed_frames(good)] + [ST["TOO_LARGE"], ST["SAMPLES"]]
    chunk_lists, frames, samples_override = [], [], {}
    for k in range(len(bad)):
        chunk_lists.append([good_sig[k % 12][:1000], good_sig[k % 12][:2000]])
        frames.append([None, bad[k]])
    # TOO_LARGE: 2000 samples' frame declared as 10 samples; SAMPLES: 100 one-byte samples declared as 90
    chunk_lists[-2][1] = good_sig[0][:10]
    frames[-2][1] = vbz_encode(good_sig[0][:2000] * 0 + np.int16(20000))
    chunk_lists[-1][1] = np.zeros(90, np.int16)
    frames[-1][1] = bad[-1]
    chunk_lists += [[s] for s in good_sig]
    frames += [None] * len(good_sig)
    batch = make_vbz_batch(chunk_lists, np.zeros(len(chunk_lists)), np.ones(len(chunk_lists)), stride, frames=frames)
    rows, nv, st = decode_rows(batch, device=0)
    torch.cuda.synchronize()
    st, nv, rows = st.cpu().numpy(), nv.cpu().numpy(), rows.cpu().numpy()
    assert st[:len(bad)].tolist() == want_st
    assert not nv[:len(bad)].any() and not rows[:len(bad)].any()
    for k, s in enumerate(good_sig):
        assert st[len(bad) + k] == 0 and nv[len(bad) + k] == s.size and np.array_equal(rows[len(bad) + k, :s.size], s)
    # invalid arguments of the C ABI
    d = torch.zeros(64, dtype=torch.int64, device="cuda:0")
    h = torch.zeros(64, dtype=torch.int64)
    with pytest.raises(ValueError):
        zstd_decompress_raw(h.view(torch.uint8), h[:3], h[:2], h.view(torch.uint8), h[:3], h[:2], h.view(torch.int32)[:2], 0, 0)
    with pytest.raises(ValueError):
        _lib.check(_lib.load().wdx_zstd_decompress(d.data_ptr(), d.data_ptr(), -1, d.data_ptr(), d.data_ptr(), d.data_ptr(),
                                                   d.data_ptr(), d.data_ptr(), 0, None), "wdx_zstd_decompress")
    with pytest.raises(ValueError):
        _lib.check(_lib.load().wdx_vbz_decode_rows(d.data_ptr(), d.data_ptr(), d.data_ptr(), 1, d.data_ptr(), 1, d.data_ptr(),
                                                   d.data_ptr(), d.data_ptr(), 0, d.data_ptr(), d.data_ptr(), 0, None), "wdx_vbz_decode_rows")
    with pytest.raises(ValueError):
        _lib.check(_lib.load().wdx_vbz_decode_rows(h.data_ptr(), h.data_ptr(), h.data_ptr(), 1, h.data_ptr(), 1, h.data_ptr(),
                                                   h.data_ptr(), h.data_ptr(), 16, h.data_ptr(), h.data_ptr(), 0, None), "wdx_vbz_decode_rows")


@pytest.fixture(scope="module")
def chain(models):
    from test_gpu_llr import _fp_cfg, _llr_cfg, _spc

    from warpdemux_b200.detect import cnn, combined
    from warpdemux_b200.file_proc import AdcBatch, MinibatchDemuxer
    from warpdemux_b200.models.dtw_svm import DTW_SVM
    from warpdemux_b200.sig_proc import FingerprintConfig

    with np.load(os.path.join(GOLD, "real4000_rna004_WDX4.npz")) as z:
        g = dict(z)
    idx, rows, adc, num = real4000_rows(g)
    spc = _spc(g)
    md = cnn.load_cnn_model(os.path.join(GOLD, "models", "cnn_rna004_130bps_v0.2.4.npz"), device=0)
    mp = DTW_SVM(models["WDX4_rna004_v1_0"], device=0, mode="guarded")
    dmx = MinibatchDemuxer(mp, md, core=spc.core, cnn_boundaries=spc.cnn_boundaries, validate_config=combined.ValidateConfig(),
                           fp_config=FingerprintConfig(**_fp_cfg(g)), device=0, llr=_llr_cfg(g), full_detect_report=True)
    sel = lambda key: g[key][idx]
    return dict(g=g, idx=idx, adc=adc, num=num, dmx=dmx, off=sel("calibration_offset"), sc=sel("calibration_scale"),
                full=sel("full_lengths"), ids=sel("read_ids"), AdcBatch=AdcBatch)


FIELDS = ("labels", "conf", "prob", "fp_status", "detect_success", "detect_code", "detect_checks", "bounds", "preds", "llr_rescued",
          "fpt", "detect_source")


def _vbz_batches(c, split, mb):
    rng = np.random.default_rng(21)
    out = []
    for lo in range(0, c["idx"].size, mb):
        sl = slice(lo, lo + mb)
        reads = []
        for a, k in zip(c["adc"][sl], c["num"][sl]):
            x = a[:k]
            if split and k > 3:
                cuts = sorted(rng.choice(np.arange(1, k), int(rng.integers(1, 3)), replace=False).tolist())
                reads.append([x[p:q] for p, q in zip([0] + cuts, cuts + [k])])
            else:
                reads.append([x])
        out.append((make_vbz_batch(reads, c["off"][sl], c["sc"][sl], c["adc"].shape[1], level=1), c["full"][sl], c["ids"][sl]))
    return out


@pytest.mark.parametrize("split", [False, True])
def test_gpu_vbz_chain_equals_adc_chain_on_real_reads(chain, split):
    import torch

    c = chain
    dmx, AdcBatch = c["dmx"], c["AdcBatch"]
    mb = 200
    vb = _vbz_batches(c, split, mb)
    # the calibrated float32 rows are the ADC path's, bit for bit, NaN padding included
    with torch.cuda.device(0):
        ja = dmx._upload(0, AdcBatch(c["adc"][:mb], c["num"][:mb], c["off"][:mb], c["sc"][:mb]), c["full"][:mb], None)
        jv = dmx._upload(1, vb[0][0], vb[0][1], None)
        torch.cuda.synchronize()
        assert torch.equal(ja["d_sig"].view(torch.int32), jv["d_sig"].view(torch.int32))
    ref = [dmx.run(AdcBatch(c["adc"][lo:lo + mb], c["num"][lo:lo + mb], c["off"][lo:lo + mb], c["sc"][lo:lo + mb]),
                   c["full"][lo:lo + mb], c["ids"][lo:lo + mb], want_fpt=True) for lo in range(0, c["idx"].size, mb)]
    got = [dmx.run(b, fl, ids, want_fpt=True) for b, fl, ids in vb]
    streamed = list(dmx.stream(vb, want_fpt=True))
    for res in (got, streamed):
        for a, b in zip(ref, res):
            for f in FIELDS:
                assert np.array_equal(getattr(a, f), getattr(b, f), equal_nan=True), f
            assert a.predictions.equals(b.predictions)


def test_gpu_vbz_bad_chunk_raises_naming_the_read(chain):
    from warpdemux_b200 import _lib

    c = chain
    b, fl, ids = _vbz_batches(c, False, 50)[0]
    k = 7
    data = b.data.copy()
    data[b.chunk_offsets[k]:b.chunk_offsets[k] + 4] = 0          # bad magic
    b.data = data
    with pytest.raises(_lib.WdxError, match=f"read {ids[k]}.*not a zstd frame"):
        c["dmx"].run(b, fl, ids)


def test_gpu_pod5_file_stream_equals_adc(chain, tmp_path):
    """pod5 file -> vbz_minibatches -> MinibatchDemuxer.stream equals the same reads as AdcBatch minibatches."""
    import uuid

    from warpdemux_b200.io.pod5_min import Pod5File

    c = chain
    n = 120
    reads = [(uuid.UUID(str(c["ids"][j])).bytes, c["adc"][j, :c["num"][j]], float(c["off"][j]), float(c["sc"][j])) for j in range(n)]
    path = str(tmp_path / "real.pod5")
    write_pod5(path, reads, chunk_size=4000, seed=1)
    f = Pod5File(path)
    stride = c["adc"].shape[1]
    got = list(c["dmx"].stream(f.vbz_minibatches(batch_size=50, preload=stride)))
    AdcBatch = c["AdcBatch"]
    # full_lengths from the file are the rows' sample counts here (the fixture keeps preload samples of each read)
    ref = [c["dmx"].run(AdcBatch(c["adc"][lo:lo + 50][:n - lo], c["num"][lo:lo + 50][:n - lo], c["off"][lo:lo + 50][:n - lo],
                                 c["sc"][lo:lo + 50][:n - lo]), c["num"][lo:min(lo + 50, n)], c["ids"][lo:min(lo + 50, n)])
           for lo in range(0, n, 50)]
    for a, b in zip(ref, got):
        for fld in FIELDS[:-2]:
            assert np.array_equal(getattr(a, fld), getattr(b, fld), equal_nan=True), fld
        assert a.predictions.equals(b.predictions)

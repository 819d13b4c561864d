"""pod5 -> VbzBatch minibatches (host side, no GPU): `Pod5File.vbz_minibatches` gathers the compressed chunks of each
minibatch from the Arrow buffers; read for read it must agree with `Pod5File.reads()` + `decode_vbz`."""
import numpy as np
import pytest

pa = pytest.importorskip("pyarrow")

from vbz_testutil import synth_signal, write_pod5  # noqa: E402


def _reads(rng, n):
    out = []
    for k in range(n):
        length = int(rng.choice([0, 1, 900, 5000, 11500, 11501, 23000, 40000]))
        sig = synth_signal(rng, length, 20)
        if k % 5 == 3 and length > 10:          # explicit uneven chunks, one of them empty
            cut = sorted(rng.integers(1, length, 2).tolist())
            sig = [sig[:cut[0]], sig[cut[0]:cut[0]], sig[cut[0]:cut[1]], sig[cut[1]:]]
        out.append((rng.bytes(16), sig, float(rng.normal(10, 3)), float(rng.uniform(0.1, 0.3))))
    return out


@pytest.mark.parametrize("preload", [11500, 3000])
@pytest.mark.parametrize("shuffle", [True, False])
def test_vbz_minibatches_match_reads_and_decode_vbz(tmp_path, preload, shuffle):
    from warpdemux_b200.file_proc import VbzBatch
    from warpdemux_b200.io.pod5_min import Pod5File, decode_vbz

    rng = np.random.default_rng(7)
    reads = _reads(rng, 37)
    path = str(tmp_path / "synth.pod5")
    rows_of = write_pod5(path, reads, chunk_size=4096, seed=3, batch_rows=5, shuffle=shuffle)
    f = Pod5File(path)
    ref = list(f.reads())
    data = open(path, "rb").read()
    end = data.index(b"ARROW1", 16) + 6                                      # the first IPC file: the signal table
    sig_tab = pa.ipc.open_file(pa.BufferReader(data[8:end])).read_all()
    chunk_bytes = sig_tab.column("signal").to_pylist()
    chunk_samples = sig_tab.column("samples").to_pylist()
    got = list(f.vbz_minibatches(batch_size=8, preload=preload))
    assert [len(g[2]) for g in got] == [8, 8, 8, 8, 5]
    i = 0
    for batch, full_lengths, ids in got:
        assert isinstance(batch, VbzBatch) and batch.stride == preload
        assert batch.chunk_offsets[0] == 0 and batch.chunk_offsets[-1] == batch.data.size
        for j in range(len(ids)):
            r = ref[i]
            assert ids[j] == r.read_id and full_lengths[j] == r.num_samples
            assert batch.offset[j] == np.float32(r.calibration_offset) and batch.scale[j] == np.float32(r.calibration_scale)
            assert r.signal_rows == rows_of[r.read_id]
            # chunks starting below preload, in the read's order
            starts = np.cumsum([0] + [chunk_samples[c] for c in r.signal_rows])[:-1]
            want_rows = [c for c, s0 in zip(r.signal_rows, starts) if s0 < preload]
            cs = range(batch.read_chunks[j], batch.read_chunks[j + 1])
            assert len(cs) == len(want_rows)
            parts = []
            for c, row in zip(cs, want_rows):
                b = batch.data[batch.chunk_offsets[c]:batch.chunk_offsets[c + 1]].tobytes()
                assert b == chunk_bytes[row] and batch.chunk_samples[c] == chunk_samples[row]
                parts.append(decode_vbz(b, int(batch.chunk_samples[c])))
            sig = r.signal
            dec = np.concatenate(parts) if parts else np.zeros(0, np.int16)
            assert np.array_equal(dec, sig[:dec.size]) and dec.size >= min(sig.size, preload)
            i += 1
    assert i == len(ref)


def test_scratch_layout_covers_what_each_chunk_gives_the_row():
    from warpdemux_b200.vbz import REGION_HDR, scratch_layout

    samples = np.array([100, 0, 5000, 7000, 20, 300], dtype=np.int32)
    rc = np.array([0, 3, 3, 6])                 # read 0: chunks 0-2, read 1: none, read 2: chunks 3-5
    soff = scratch_layout(samples, rc, 5050)
    size = np.diff(soff)
    assert np.all(soff % 16 == 0)
    # read 0: chunk 2 starts at sample 100 and gives 4950 samples; read 2: chunk 3 fills the row, 4 and 5 are past it
    want = [REGION_HDR + 13 + 200, REGION_HDR, REGION_HDR + 625 + 2 * 4950, REGION_HDR + 875 + 2 * 5050, 0, 0]
    assert np.all(size >= want) and np.all(size - np.array(want) < 16)
    with pytest.raises(ValueError):
        scratch_layout(samples, np.array([0, 2]), 100)

"""VBZ test material: a streamvbyte-16 encoder (the inverse of io.pod5_min.decode_vbz), a seeded corpus of zstd frames
written by pyarrow, a header walk that names the zstd modes a frame uses, and small hand-built frames for the modes
pyarrow's encoder does not emit on that corpus (RLE literals, RLE literal-length table)."""
import collections

import numpy as np


def svb16_encode(x) -> bytes:
    """int16 samples -> streamvbyte-16 bytes of zig-zag deltas (pod5 VBZ before zstd)."""
    x = np.asarray(x, dtype=np.int16)
    d = np.diff(np.concatenate([[0], x.astype(np.int32)])).astype(np.int32)
    d = ((d + 32768) % 65536 - 32768).astype(np.int32)
    u = ((d << 1) ^ (d >> 31)).astype(np.uint32) & 0xFFFF
    keys = (u > 255).astype(np.uint8)
    w = 1 + keys.astype(np.int64)
    off = np.cumsum(w) - w
    data = np.zeros(int(w.sum()), np.uint8)
    data[off] = u & 255
    data[off[keys == 1] + 1] = u[keys == 1] >> 8
    return np.packbits(keys, bitorder="little").tobytes() + data.tobytes()


def vbz_encode(x, level: int = 1) -> bytes:
    import pyarrow as pa

    return pa.Codec("zstd", compression_level=level).compress(svb16_encode(x), asbytes=True)


def zstd_stream(raw: bytes) -> bytes:
    """A frame as pyarrow's streaming writer makes it: window descriptor, no content size."""
    import pyarrow as pa

    bio = pa.BufferOutputStream()
    s = pa.CompressedOutputStream(bio, "zstd")
    s.write(raw)
    s.close()
    return bio.getvalue().to_pybytes()


def zstd_decompress(frame: bytes) -> bytes:
    import pyarrow as pa

    return bytes(pa.CompressedInputStream(pa.BufferReader(frame), "zstd").read())


def synth_signal(rng, n, sigma):
    return (np.cumsum(rng.normal(0, sigma, n)) % 2000 + 300).astype(np.int16)


LEVELS = (-5, 1, 3, 9, 19)


def corpus_inputs(seed=1):
    """Uncompressed inputs: svb16 signals of several lengths and noise levels, and a few byte patterns."""
    rng = np.random.default_rng(seed)
    out = [svb16_encode(synth_signal(rng, n, s)) for n in (0, 1, 7, 100, 5000, 11500, 102400, 300000) for s in (2, 20, 200)]
    out += [bytes(300000), svb16_encode(np.full(50000, 500, np.int16)), rng.integers(0, 256, 200000, dtype=np.uint8).tobytes(),
            b"abcdefgh" * 40000, bytes(rng.integers(0, 4, 400000, dtype=np.uint8))]
    return out


def corpus(seed=1):
    """[(frame, raw)]: every input at every level of LEVELS, plus the streaming writer's frame."""
    import pyarrow as pa

    frames = []
    for raw in corpus_inputs(seed):
        for lvl in LEVELS:
            frames.append((pa.Codec("zstd", compression_level=lvl).compress(raw, asbytes=True), raw))
        frames.append((zstd_stream(raw), raw))
    return frames


def frame_modes(b: bytes) -> collections.Counter:
    """Walk a frame's headers: which block types, literal types and sequence table modes it uses."""
    C = collections.Counter()
    assert int.from_bytes(b[:4], "little") == 0xFD2FB528
    fhd = b[4]
    fcs_flag, single, did = fhd >> 6, (fhd >> 5) & 1, fhd & 3
    p = 5 + (0 if single else 1) + [0, 1, 2, 4][did] + [1 if single else 0, 2, 4, 8][fcs_flag]
    C["single_segment" if single else "window_descriptor"] += 1
    C["fcs" if (fcs_flag or single) else "no_fcs"] += 1
    while True:
        h = int.from_bytes(b[p:p + 3], "little")
        last, bt, sz = h & 1, (h >> 1) & 3, h >> 3
        p += 3
        C["block_" + ["raw", "rle", "compressed", "reserved"][bt]] += 1
        if bt == 2:
            q = p
            b0 = b[q]
            lt, sf = b0 & 3, (b0 >> 2) & 3
            if lt in (0, 1):
                C["lit_" + ["raw", "rle"][lt]] += 1
                if sf in (0, 2):
                    rs, hs = b0 >> 3, 1
                elif sf == 1:
                    rs, hs = (b0 >> 4) + (b[q + 1] << 4), 2
                else:
                    rs, hs = (b0 >> 4) + (b[q + 1] << 4) + (b[q + 2] << 12), 3
                q += hs + (rs if lt == 0 else 1)
            else:
                C["lit_treeless" if lt == 3 else ("lit_huf1" if sf == 0 else "lit_huf4")] += 1
                if sf in (0, 1):
                    cs, hs = (int.from_bytes(b[q:q + 3], "little") >> 14) & 0x3FF, 3
                elif sf == 2:
                    cs, hs = (int.from_bytes(b[q:q + 4], "little") >> 18) & 0x3FFF, 4
                else:
                    cs, hs = (int.from_bytes(b[q:q + 5], "little") >> 22) & 0x3FFFF, 5
                q += hs + cs
            n0 = b[q]
            if n0 == 0:
                C["seq_none"] += 1
            else:
                q += 1 if n0 < 128 else (2 if n0 < 255 else 3)
                m = b[q]
                for nm, sh in (("LL", 6), ("OF", 4), ("ML", 2)):
                    C["seq_%s_%s" % (nm, ["predefined", "rle", "fse", "repeat"][(m >> sh) & 3])] += 1
        p += 1 if bt == 1 else sz
        if last:
            break
    return C


def _frame(blocks, fcs=None) -> bytes:
    """zstd frame from (type, payload, regenerated size) blocks; single segment with a 4-byte content size."""
    total = sum(r for _, _, r in blocks) if fcs is None else fcs
    out = bytearray((0xFD2FB528).to_bytes(4, "little")) + bytes([0x80 | 0x20]) + total.to_bytes(4, "little")
    for i, (bt, payload, regen) in enumerate(blocks):
        size = regen if bt == 1 else len(payload)
        out += ((size << 3) | (bt << 1) | (i == len(blocks) - 1)).to_bytes(3, "little") + payload
    return bytes(out)


def _bits_backward(fields) -> bytes:
    """Backward bitstream whose reader meets `fields` [(value, nbits)] in order."""
    x = 1
    for v, nb in fields:
        x = (x << nb) | v
    return x.to_bytes((x.bit_length() + 7) // 8, "little")


def _run_sequences(lits: bytes, seqs, out: bytearray, rep):
    """Reference execution of (ll, offset_value, ml) sequences (RFC 8878 3.1.2.5 / repeat offsets)."""
    li = 0
    for ll, ofv, ml in seqs:
        out += lits[li:li + ll]
        li += ll
        if ofv > 3:
            off = ofv - 3
            rep[:] = [off, rep[0], rep[1]]
        else:
            idx = ofv + (1 if ll == 0 else 0)
            if idx == 1:
                off = rep[0]
            elif idx == 2:
                off = rep[1]
                rep[:] = [off, rep[0], rep[2]]
            else:
                off = rep[2] if idx == 3 else rep[0] - 1
                rep[:] = [off, rep[0], rep[1]]
        for _ in range(ml):
            out.append(out[-off])
    out += lits[li:]


def hand_frames():
    """[(name, frame, expected content)] for RLE literals and the RLE literal-length mode (with raw / RLE blocks)."""
    frames = []
    # RLE literals, no sequences; then a raw block and an RLE block
    lit_rle = bytes([(20 << 3) | 1, 0x41, 0])
    frames.append(("rle_literals", _frame([(2, lit_rle, 20), (0, b"xyz", 3), (1, b"\x07", 5)]), b"A" * 20 + b"xyz" + b"\x07" * 5))
    # raw literals, sequences with RLE tables: LL code 16 (16 + 1 bit), OF code 3 (8 + 3 bits), ML code 5 (8)
    lits = bytes(range(40))
    lit_raw = bytes([(1 << 2) | 0 | ((len(lits) & 15) << 4), len(lits) >> 4]) + lits
    seqs = [(16, 8 + 2, 8), (17, 8 + 5, 8)]
    fields = []
    for ll, ofv, ml in seqs:          # per sequence: offset bits, match-length bits, literal-length bits
        fields += [(ofv - 8, 3), (ll - 16, 1)]
    seq_sec = bytes([len(seqs), (1 << 6) | (1 << 4) | (1 << 2), 16, 3, 5]) + _bits_backward(fields)
    out = bytearray()
    _run_sequences(lits, seqs, out, [1, 4, 8])
    frames.append(("rle_ll_of_ml", _frame([(2, lit_raw + seq_sec, len(out))]), bytes(out)))
    # RLE literals followed by sequences whose literal length is 0 (repeat-offset shift) and repeat-offset codes
    # (RLE tables cannot mix codes, so each sequence gets its own block; the repeat offsets carry across blocks)
    seqs = [(4, 3 + 3, 6), (0, 1, 5), (2, 1, 3)]      # offset 3; LL = 0 -> the second repeat offset; then the first
    ofcode = {6: (2, 2), 1: (0, 0)}                   # offset value -> (code, extra bits)
    blocks, out, rep = [(0, b"abcdefgh", 8)], bytearray(b"abcdefgh"), [1, 4, 8]
    for ll, ofv, ml in seqs:
        c, nb = ofcode[ofv]
        lit = bytes([(ll << 3) | 1, 0x5A])
        seq = bytes([1, (1 << 6) | (1 << 4) | (1 << 2), ll, c, ml - 3]) + _bits_backward([(ofv - (1 << c), nb)])
        before = len(out)
        _run_sequences(b"\x5a" * ll, [(ll, ofv, ml)], out, rep)
        blocks.append((2, lit + seq, len(out) - before))
    frames.append(("rle_literals_repeat_offsets", _frame(blocks), bytes(out)))
    return frames


# status codes of include/wdx_b200.h (WDX_VBZ_*)
ST = dict(OK=0, BAD_MAGIC=1, DICTIONARY=2, CHECKSUM=3, RESERVED=4, TRUNCATED=5, CORRUPT=6, TOO_LARGE=7, FRAMES=8, SAMPLES=9,
          SCRATCH=10)


def malformed_frames(good: bytes):
    """[(name, frame, expected status)] derived from a valid single-segment frame `good` (pyarrow's Codec output)."""
    assert good[4] & 0x20, "needs a single-segment frame"
    fhd = good[4]
    with_did = good[:4] + bytes([fhd | 1]) + b"\x07" + good[5:]           # 1-byte dictionary ID = 7
    with_chk = good[:4] + bytes([fhd | 4]) + good[5:]
    hdr = 5 + [1, 2, 4, 8][fhd >> 6]                                       # first block header
    bh = int.from_bytes(good[hdr:hdr + 3], "little")
    reserved_block = good[:hdr] + ((bh & ~6) | (3 << 1)).to_bytes(3, "little") + good[hdr + 3:]
    return [
        ("bad_magic", b"\x00" + good[1:], ST["BAD_MAGIC"]),
        ("dictionary", with_did, ST["DICTIONARY"]),
        ("checksum", with_chk, ST["CHECKSUM"]),
        ("truncated", good[:len(good) * 2 // 3], ST["TRUNCATED"]),
        ("reserved_block", reserved_block, ST["RESERVED"]),
        ("second_frame", good + good, ST["FRAMES"]),
        ("skippable", (0x184D2A50).to_bytes(4, "little") + (4).to_bytes(4, "little") + b"\0" * 4, ST["FRAMES"]),
    ]


def write_pod5(path, reads, chunk_size=None, seed=0, level=1, batch_rows=7, shuffle=True):
    """A minimal pod5 file: signature, signal / run-info / reads Arrow IPC files, signature.  reads: [(read_id bytes16,
    int16 signal, offset, scale)] or [(id, [chunk signals], offset, scale)] for explicit chunks.  Signal-table rows are
    shuffled (a read's chunk rows are then not contiguous) and split into record batches of `batch_rows`.
    Returns {read_id str: list of signal-table rows}."""
    import uuid

    import pyarrow as pa

    rng = np.random.default_rng(seed)
    chunks, owner = [], []
    for k, (rid, sig, _, _) in enumerate(reads):
        parts = sig if isinstance(sig, list) else (
            [sig[i:i + chunk_size] for i in range(0, max(len(sig), 1), chunk_size)] if chunk_size else [sig])
        for p in parts:
            chunks.append(np.asarray(p, dtype=np.int16))
            owner.append(k)
    order = rng.permutation(len(chunks)) if shuffle else np.arange(len(chunks))
    row_of = np.empty(len(chunks), dtype=np.int64)
    row_of[order] = np.arange(len(chunks))
    sig_tab = pa.table({
        "read_id": pa.array([reads[owner[c]][0] for c in order], type=pa.binary(16)),
        "signal": pa.array([vbz_encode(chunks[c], level) for c in order], type=pa.large_binary()),
        "samples": pa.array([len(chunks[c]) for c in order], type=pa.uint32()),
    })
    rows = [[] for _ in reads]
    for c in range(len(chunks)):
        rows[owner[c]].append(int(row_of[c]))
    reads_tab = pa.table({
        "read_id": pa.array([r[0] for r in reads], type=pa.binary(16)),
        "signal": pa.array(rows, type=pa.list_(pa.uint64())),
        "num_samples": pa.array([int(sum(len(chunks[c]) for c in range(len(chunks)) if owner[c] == k)) for k in range(len(reads))], type=pa.uint64()),
        "calibration_offset": pa.array([r[2] for r in reads], type=pa.float32()),
        "calibration_scale": pa.array([r[3] for r in reads], type=pa.float32()),
    })
    run_tab = pa.table({"acquisition_id": pa.array(["run0"]), "sample_rate": pa.array([4000], type=pa.uint16())})

    def ipc(t, max_rows=None):
        sink = pa.BufferOutputStream()
        with pa.ipc.new_file(sink, t.schema) as w:
            for b in t.to_batches(max_chunksize=max_rows):
                w.write_batch(b)
        return sink.getvalue().to_pybytes()

    sigb = b"\x8bPOD\r\n\x1a\n"
    with open(path, "wb") as fh:
        fh.write(sigb + ipc(sig_tab, batch_rows) + ipc(run_tab) + ipc(reads_tab) + sigb)
    return {str(uuid.UUID(bytes=r[0])): rows[k] for k, r in enumerate(reads)}


def make_vbz_batch(chunk_lists, offset, scale, stride, level=1, frames=None):
    """VbzBatch from per-read lists of int16 chunk signals (frames: optional per-read lists of ready-made frames)."""
    from warpdemux_b200.file_proc import VbzBatch

    fr, samples, counts = [], [], []
    for k, chunks in enumerate(chunk_lists):
        counts.append(len(chunks))
        for j, c in enumerate(chunks):
            samples.append(len(c))
            given = frames[k][j] if frames is not None and frames[k] is not None else None
            fr.append(given if given is not None else vbz_encode(c, level))
    off = np.concatenate([[0], np.cumsum([len(f) for f in fr])]).astype(np.int64)
    return VbzBatch(data=np.frombuffer(b"".join(fr), dtype=np.uint8).copy(), chunk_offsets=off,
                    chunk_samples=np.array(samples, dtype=np.int32), read_chunks=np.concatenate([[0], np.cumsum(counts)]).astype(np.int64),
                    offset=np.asarray(offset, dtype=np.float32), scale=np.asarray(scale, dtype=np.float32), stride=int(stride))

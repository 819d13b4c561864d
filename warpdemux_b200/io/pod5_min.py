"""Minimal pod5 reader (host side) — enough to feed the classification path from
the reference's own test file without the `pod5` package.

Replaces, for the fields the path needs, what `warpdemux/file_proc.py:227-279`
gets from `pod5.Reader`: `read_id`, `num_samples` and `signal_pa`
(= (adc + calibration_offset) * calibration_scale, float32).

Format (pod5 v0.2.x/0.3.x container): a signature, then three embedded Arrow IPC
files (signal table, run-info table, reads table), each delimited by `ARROW1`
magic strings.  Signal rows are VBZ chunks: zstd( streamvbyte16( zigzag( delta(
int16 samples )))), with one key BIT per sample (0 = 1 byte, 1 = 2 bytes, LSB
first) ahead of the data bytes.  A read's signal is the concatenation of the
signal-table rows listed in the reads table.

Parity: there is no `pod5` package in this image to compare with; the decoder is
self-checked (decoded length == `samples`, consumed bytes == chunk length) in
tests/test_pod5_reader.py — unpinned by the reference.
"""
from __future__ import annotations

import re
import uuid
from dataclasses import dataclass
from typing import Iterator, List, Optional, Sequence

import numpy as np

_SIGNATURE = b"\x8bPOD\r\n\x1a\n"


def decode_vbz(chunk: bytes, n_samples: int) -> np.ndarray:
    """One VBZ signal chunk -> int16[n_samples]."""
    import pyarrow as pa

    raw = pa.CompressedInputStream(pa.BufferReader(chunk), "zstd").read()
    buf = np.frombuffer(raw, dtype=np.uint8)
    if n_samples == 0:
        return np.zeros(0, dtype=np.int16)
    nk = (n_samples + 7) // 8
    keys = np.unpackbits(buf[:nk], bitorder="little")[:n_samples].astype(np.int64)
    width = 1 + keys
    off = np.cumsum(width) - width
    data = buf[nk:]
    if off[-1] + width[-1] != data.size:
        raise ValueError("VBZ chunk length does not match its key stream")
    lo = data[off].astype(np.uint32)
    hi = data[np.minimum(off + 1, data.size - 1)].astype(np.uint32) * keys.astype(np.uint32)
    u = lo | (hi << 8)
    zz = (u >> 1).astype(np.int32) ^ -(u & 1).astype(np.int32)      # zig-zag
    return np.cumsum(zz, dtype=np.int32).astype(np.int16)            # delta (wraps like int16 arithmetic)


def _uuid_strings(col) -> np.ndarray:
    """A column of 16-byte read ids -> str [n] in uuid.UUID's canonical form, without a per-read Python loop."""
    import pyarrow as pa

    arr = col.combine_chunks() if isinstance(col, pa.ChunkedArray) else col
    if isinstance(arr, pa.ExtensionArray):
        arr = arr.storage
    if pa.types.is_fixed_size_binary(arr.type):
        raw = np.frombuffer(arr.buffers()[1], dtype=np.uint8)[arr.offset * 16:(arr.offset + len(arr)) * 16]
    else:
        raw = np.frombuffer(b"".join(arr.to_pylist()), dtype=np.uint8)
    raw = raw.reshape(-1, 16)
    hexd = np.frombuffer(b"0123456789abcdef", dtype=np.uint8)[np.stack([raw >> 4, raw & 15], axis=-1).reshape(-1, 32)]
    out = np.full((raw.shape[0], 36), ord("-"), dtype=np.uint8)
    for dst, src in ((slice(0, 8), slice(0, 8)), (slice(9, 13), slice(8, 12)), (slice(14, 18), slice(12, 16)),
                     (slice(19, 23), slice(16, 20)), (slice(24, 36), slice(20, 32))):
        out[:, dst] = hexd[:, src]
    return out.view("S36").ravel().astype(str)


@dataclass
class Pod5Read:
    read_id: str
    num_samples: int
    calibration_offset: float
    calibration_scale: float
    signal_rows: List[int]
    _file: "Pod5File"

    @property
    def signal(self) -> np.ndarray:
        """Raw ADC samples, int16."""
        return self._file._signal(self.signal_rows)

    @property
    def signal_pa(self) -> np.ndarray:
        """Calibrated picoampere signal, float32 (pod5 `ReadRecord.signal_pa`)."""
        return ((self.signal.astype(np.float32) + np.float32(self.calibration_offset))
                * np.float32(self.calibration_scale))


class Pod5File:
    def __init__(self, path: str):
        import pyarrow as pa

        self.path = path
        with open(path, "rb") as fh:
            data = fh.read()
        if not (data.startswith(_SIGNATURE) and data.endswith(_SIGNATURE)):
            raise ValueError(f"{path}: not a pod5 file")
        marks = [m.start() for m in re.finditer(b"ARROW1", data)]
        if len(marks) < 6 or len(marks) % 2:
            raise ValueError(f"{path}: cannot locate the embedded Arrow tables")
        tables = {}
        for a, b in zip(marks[0::2], marks[1::2]):
            rd = pa.ipc.open_file(pa.BufferReader(data[a:b + 6]))
            names = set(rd.schema.names)
            if {"signal", "samples"} <= names:
                tables["signal"] = rd
            elif {"num_samples", "calibration_scale"} <= names:
                tables["reads"] = rd
        if set(tables) != {"signal", "reads"}:
            raise ValueError(f"{path}: signal / reads tables not found")
        self._sig = tables["signal"]
        self._reads = tables["reads"].read_all()
        # row index -> (batch, offset in batch) for the signal table
        counts = [self._sig.get_batch(i).num_rows for i in range(self._sig.num_record_batches)]
        self._batch_start = np.concatenate([[0], np.cumsum(counts)])
        self._batch_cache = {}

    def __len__(self) -> int:
        return self._reads.num_rows

    def _signal_row(self, row: int) -> np.ndarray:
        b = int(np.searchsorted(self._batch_start, row, side="right") - 1)
        if b not in self._batch_cache:
            if len(self._batch_cache) > 4:
                self._batch_cache.clear()
            self._batch_cache[b] = self._sig.get_batch(b)
        batch = self._batch_cache[b]
        i = row - int(self._batch_start[b])
        return decode_vbz(batch.column("signal")[i].as_py(), int(batch.column("samples")[i].as_py()))

    def _signal(self, rows: Sequence[int]) -> np.ndarray:
        parts = [self._signal_row(int(r)) for r in rows]
        return parts[0] if len(parts) == 1 else np.concatenate(parts)

    def _vbz_index(self):
        """The signal table as one large_binary column (storage of the `minknow.vbz` extension type) with its offsets and
        bytes as numpy views, and its `samples`; the reads table's flattened signal-row lists.  Built once."""
        if getattr(self, "_vbz", None) is None:
            import pyarrow as pa

            cols, samples = [], []
            for i in range(self._sig.num_record_batches):
                b = self._sig.get_batch(i)
                col = b.column("signal")
                if isinstance(col, pa.ExtensionArray):
                    col = col.storage
                cols.append(col if col.type == pa.large_binary() else col.cast(pa.large_binary()))
                samples.append(np.asarray(b.column("samples").to_numpy(zero_copy_only=False), dtype=np.int64))
            rows = self._reads.column("signal").combine_chunks()
            if isinstance(rows, pa.ExtensionArray):
                rows = rows.storage
            loff = rows.offsets.to_numpy().astype(np.int64)
            sig = pa.concat_arrays(cols) if cols else pa.array([], type=pa.large_binary())
            off = np.frombuffer(sig.buffers()[1], dtype=np.int64)[sig.offset:sig.offset + len(sig) + 1]
            data = np.frombuffer(sig.buffers()[2], dtype=np.uint8) if len(sig) else np.zeros(0, np.uint8)
            self._vbz = dict(signal=sig, off=off, data=data,
                             samples=np.concatenate(samples) if samples else np.zeros(0, np.int64),
                             row_off=loff - loff[0], rows=np.asarray(rows.flatten().to_numpy(zero_copy_only=False), dtype=np.int64))
        return self._vbz

    def vbz_minibatches(self, batch_size: int = 1000, preload: int = 11500):
        """Minibatches of still-compressed signal for the device decoder: yields (file_proc.VbzBatch, full_lengths
        int64 [n] (= num_samples), read_ids [n] str) per `batch_size` reads in file order.  A read keeps the chunks that
        start below `preload` samples (the row length); their bytes are not decoded here: a minibatch whose chunks are
        consecutive signal-table rows gets a view of the column's bytes, other minibatches a gather by Arrow (`take`)."""
        import pyarrow as pa

        from ..file_proc import VbzBatch

        ix = self._vbz_index()
        t = self._reads
        num = np.asarray(t.column("num_samples").to_numpy(), dtype=np.int64)
        cal_off = np.asarray(t.column("calibration_offset").to_numpy(), dtype=np.float32)
        cal_sc = np.asarray(t.column("calibration_scale").to_numpy(), dtype=np.float32)
        ids = _uuid_strings(t.column("read_id"))
        loff, rows_all, samples_all = ix["row_off"], ix["rows"], ix["samples"]
        for a in range(0, t.num_rows, int(batch_size)):
            b = min(a + int(batch_size), t.num_rows)
            nr = b - a
            rows = rows_all[loff[a]:loff[b]]
            cnt = np.diff(loff[a:b + 1])
            s = samples_all[rows]
            read_of = np.repeat(np.arange(nr), cnt)
            excl = np.cumsum(s) - s
            first = (loff[a:b] - loff[a])[read_of]
            keep = (excl - excl[first]) < preload if rows.size else np.zeros(0, dtype=bool)
            rc = np.concatenate([[0], np.cumsum(np.bincount(read_of[keep], minlength=nr))]).astype(np.int64)
            r = rows[keep]
            if r.size == 0 or np.all(np.diff(r) == 1):     # the usual layout: the minibatch's chunks are consecutive rows
                lo_, hi_ = (r[0], r[-1] + 1) if r.size else (0, 0)
                off = ix["off"][lo_:hi_ + 1]
                data = ix["data"][off[0]:off[-1]] if r.size else np.zeros(0, np.uint8)
            else:
                sel = ix["signal"].take(pa.array(r, type=pa.int64()))
                off = np.frombuffer(sel.buffers()[1], dtype=np.int64)[sel.offset:sel.offset + len(sel) + 1]
                data = np.frombuffer(sel.buffers()[2], dtype=np.uint8)[off[0]:off[-1]]
            batch = VbzBatch(data=data, chunk_offsets=(off - off[0]).astype(np.int64), chunk_samples=s[keep].astype(np.int32),
                             read_chunks=rc, offset=cal_off[a:b], scale=cal_sc[a:b], stride=int(preload))
            yield batch, num[a:b].copy(), ids[a:b]

    def reads(self, selection: Optional[Sequence[str]] = None) -> Iterator[Pod5Read]:
        t = self._reads
        ids = t.column("read_id").to_pylist()
        ns = t.column("num_samples").to_pylist()
        off = t.column("calibration_offset").to_pylist()
        sc = t.column("calibration_scale").to_pylist()
        rows = t.column("signal").to_pylist()
        want = set(selection) if selection is not None else None
        for i in range(t.num_rows):
            rid = str(uuid.UUID(bytes=ids[i]))
            if want is not None and rid not in want:
                continue
            yield Pod5Read(rid, int(ns[i]), float(off[i]), float(sc[i]), list(rows[i]), self)

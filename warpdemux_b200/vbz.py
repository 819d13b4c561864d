"""pod5 VBZ signal decoding on the device (csrc/wdx_vbz.cu, include/wdx_b200.h: wdx_zstd_decompress,
wdx_vbz_decode_rows).

    rows, n_valid, status = decode_rows(vbz_batch)          # CUDA int16 [n, stride], int32 [n], int32 [n]

`io.pod5_min.decode_vbz` is the host reference of these kernels; there is no host fallback behind them.
"""
from __future__ import annotations

from typing import Optional

import numpy as np

from . import _lib

# include/wdx_b200.h WDX_VBZ_*
STATUS = {0: "ok", 1: "not a zstd frame", 2: "zstd dictionary", 3: "zstd checksum flag", 4: "reserved zstd field",
          5: "truncated zstd frame", 6: "corrupt zstd frame", 7: "content larger than its bound",
          8: "skippable or second zstd frame", 9: "samples disagree with the streamvbyte keys / data",
          10: "scratch region too small"}
REGION_HDR = 16


def status_name(code: int) -> str:
    return STATUS.get(int(code), f"status {int(code)}")


def scratch_layout(chunk_samples, read_chunks, stride: int) -> np.ndarray:
    """int64 [m+1] offsets of the per-chunk scratch regions wdx_vbz_decode_rows needs: 16 header bytes, the key bytes
    and two data bytes per sample the row takes from the chunk, 16-byte aligned; nothing for chunks past the row."""
    s = np.asarray(chunk_samples, dtype=np.int64).reshape(-1)
    rc = np.asarray(read_chunks, dtype=np.int64).reshape(-1)
    m = s.size
    if rc.size < 1 or rc[0] != 0 or rc[-1] != m or np.any(np.diff(rc) < 0):
        raise ValueError("read_chunks must be a CSR offsets array over all chunks (0 .. m, non-decreasing)")
    if np.any(s < 0):
        raise ValueError("chunk samples must be non-negative")
    excl = np.cumsum(s) - s
    first = np.repeat(rc[:-1], np.diff(rc))               # first chunk of each chunk's read
    soff = excl - excl[first] if m else excl
    t = np.clip(stride - soff, 0, s)
    need = np.where(soff < stride, REGION_HDR + (s + 7) // 8 + 2 * t, 0)
    need = (need + 15) // 16 * 16
    return np.concatenate([[0], np.cumsum(need)]).astype(np.int64)


def zstd_decompress_raw(src, chunk_off, limit, scratch, scratch_off, produced, status, device: int, stream: int) -> None:
    """wdx_zstd_decompress on device tensors (uint8 src / scratch, int64 offsets / limit / produced, int32 status)."""
    m = int(chunk_off.numel()) - 1
    rc = _lib.load().wdx_zstd_decompress(src.data_ptr(), chunk_off.data_ptr(), m, limit.data_ptr(), scratch.data_ptr(),
                                         scratch_off.data_ptr(), produced.data_ptr(), status.data_ptr(), int(device), stream)
    _lib.check(rc, "wdx_zstd_decompress")


def decode_rows_raw(src, chunk_off, samples, read_chunks, scratch, scratch_off, rows, n_valid, status, device: int, stream: int) -> None:
    """wdx_vbz_decode_rows on device tensors; rows int16 [n, stride]."""
    m, n = int(samples.numel()), int(read_chunks.numel()) - 1
    rc = _lib.load().wdx_vbz_decode_rows(src.data_ptr(), chunk_off.data_ptr(), samples.data_ptr(), m, read_chunks.data_ptr(), n,
                                         scratch.data_ptr(), scratch_off.data_ptr(), rows.data_ptr(), int(rows.shape[1]),
                                         n_valid.data_ptr(), status.data_ptr(), int(device), stream)
    _lib.check(rc, "wdx_vbz_decode_rows")


def zstd_decompress(frames, limits=None, capacities=None, device: Optional[int] = None):
    """Host list of zstd frames -> [(status, bytes)] through the device decoder (for tests and tools).  limits: per
    frame prefix length (default: everything); capacities: output bytes per frame (default: the limit, or 1 MiB)."""
    import torch

    dev = torch.device("cuda", 0 if device is None else int(device))
    m = len(frames)
    lim = np.array([np.iinfo(np.int64).max if limits is None or limits[i] is None else limits[i] for i in range(m)], dtype=np.int64)
    cap = np.array([capacities[i] if capacities is not None else (lim[i] if limits is not None and limits[i] is not None else 1 << 20)
                    for i in range(m)], dtype=np.int64)
    off = np.concatenate([[0], np.cumsum([len(f) for f in frames])]).astype(np.int64)
    soff = np.concatenate([[0], np.cumsum(cap)]).astype(np.int64)
    data = np.frombuffer(b"".join(frames), dtype=np.uint8) if off[-1] else np.zeros(1, np.uint8)
    t = lambda a: torch.from_numpy(np.array(a, copy=True)).to(dev)
    d_src, d_off, d_lim, d_soff = t(data), t(off), t(lim), t(soff)
    d_scr = torch.empty(max(int(soff[-1]), 1), dtype=torch.uint8, device=dev)
    d_prod = torch.empty(max(m, 1), dtype=torch.int64, device=dev)
    d_st = torch.empty(max(m, 1), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        st = torch.cuda.current_stream()
        zstd_decompress_raw(d_src, d_off, d_lim, d_scr, d_soff, d_prod, d_st, dev.index, st.cuda_stream)
        scr, prod, status = d_scr.cpu().numpy(), d_prod.cpu().numpy(), d_st.cpu().numpy()
    return [(int(status[i]), scr[soff[i]:soff[i] + prod[i]].tobytes()) for i in range(m)]


def decode_rows(batch, device: Optional[int] = None, stream=None):
    """A `file_proc.VbzBatch` -> (rows int16 [n, stride], n_valid int32 [n], status int32 [n]), CUDA tensors on
    `device`, produced on `stream` (default: the current stream).  status != 0: the read's chunks could not be decoded
    (`status_name`); its row is zero and n_valid 0."""
    import torch

    dev = torch.device("cuda", 0 if device is None else int(device))
    n, stride = int(np.asarray(batch.read_chunks).size) - 1, int(batch.stride)
    soff = scratch_layout(batch.chunk_samples, batch.read_chunks, stride)
    rows = torch.empty((max(n, 0), stride), dtype=torch.int16, device=dev)
    n_valid = torch.empty(max(n, 0), dtype=torch.int32, device=dev)
    status = torch.empty(max(n, 0), dtype=torch.int32, device=dev)
    if n <= 0:
        return rows, n_valid, status
    t = lambda a, dt: torch.from_numpy(np.array(a, dtype=dt, copy=True)).to(dev)
    data = np.asarray(batch.data, dtype=np.uint8).reshape(-1)
    with torch.cuda.device(dev):
        st = stream if stream is not None else torch.cuda.current_stream()
        with torch.cuda.stream(st):
            d_src = t(data if data.size else np.zeros(1, np.uint8), np.uint8)
            d_off, d_s, d_rc, d_soff = t(batch.chunk_offsets, np.int64), t(batch.chunk_samples, np.int32), t(batch.read_chunks, np.int64), t(soff, np.int64)
            d_scr = torch.empty(max(int(soff[-1]), 16), dtype=torch.uint8, device=dev)
            decode_rows_raw(d_src, d_off, d_s, d_rc, d_scr, d_soff, rows, n_valid, status, dev.index, st.cuda_stream)
            for x in (d_src, d_off, d_s, d_rc, d_soff, d_scr):   # freed by the caching allocator only after the kernels ran
                x.record_stream(st)
    return rows, n_valid, status

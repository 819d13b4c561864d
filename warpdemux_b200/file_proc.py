"""The production minibatch step on the GPU — compute core of the reference's
`worker_detect_and_predict_on_preloaded_signals` (warpdemux/file_proc.py:380-455):

    combined_detect_cnn          boundary CNN + validation            wdx_cnn_detect, wdx_validate_run
    barcode_fpt_wrapper (x n)    fingerprint per read                 } wdx_fp_predict (fingerprints stay
    model_predict.predict        DTW distances + SVC + thresholds     }  on the device)
    add_read_id_col_to_predictions                                    host (pandas)

One upload of the NaN-padded float32 minibatch (none when a CUDA tensor is given; asynchronous from a pinned
torch tensor), three kernel stages chained on ONE stream through device-resident buffers (boundaries, verdicts, fingerprints never visit the host), one download of the per-read results.
The queues / counters of the reference worker are orchestration and stay with the caller.

Reads whose CNN boundaries fail validation are re-detected like the reference does (adapted/detect/combined.py:222-290:
hail-mary poly(A) re-detection, then the LLR detector) — on the device, inside the validation call
(`wdx_validate_set_llr`, csrc/llr_kernel.cuh), when the configuration asks for it (`cnn_boundaries.fallback_to_llr*`;
`llr=` overrides).  `llr_fallback` is an optional host hook for the reads that still fail after that (or for all failed
reads when the device fallback is off): it is called for their minibatch rows between validation and fingerprinting
(one host round trip of n verdict bytes).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, List, Optional, Sequence

import numpy as np
import pandas as pd

from . import _lib
from . import vbz as _vbz
from .detect import cnn as _cnn
from .detect import combined as _combined
from .models.utils import predictions_to_df
from .sharding import default_device
from .sig_proc import FAIL_REASON as FP_STATUS_REASON   # one table, the reference's strings
from .sig_proc import FP_NONFINITE, Fingerprinter, FingerprintConfig


def add_read_id_col_to_predictions(predictions: pd.DataFrame, read_ids) -> pd.DataFrame:
    """file_proc.py:769-780."""
    cols = predictions.columns.tolist()
    if "#read_id" in cols:
        raise ValueError("'#read_id' already in dataframe")
    predictions["#read_id"] = read_ids
    return predictions[["#read_id", *cols]]


@dataclass
class AdcBatch:
    """A minibatch as raw ADC samples instead of calibrated pA rows: half the bytes over PCIe, calibrated on the device
    (`wdx_calibrate_rows`: pA = (adc + offset) * scale in float32, as pod5's `signal_pa`; bit-identical rows)."""
    adc: np.ndarray            # int16 [n, stride] (any filler beyond num_samples), numpy or torch CPU tensor (pinned or not)
    num_samples: np.ndarray    # [n] samples present per row (min(read length, stride))
    offset: np.ndarray         # float32 [n] calibration_offset
    scale: np.ndarray          # float32 [n] calibration_scale


@dataclass
class VbzBatch:
    """A minibatch as the still-compressed pod5 signal chunks of its reads (`io.pod5_min.Pod5File.vbz_minibatches`):
    the chunks go to the device as they are and are decoded there into the int16 rows an `AdcBatch` carries
    (`vbz.decode_rows`), then calibrated like them.  Read r = chunks read_chunks[r] .. read_chunks[r+1]-1 in order."""
    data: np.ndarray           # uint8 [bytes] the chunks' zstd frames, concatenated
    chunk_offsets: np.ndarray  # int64 [m+1] frame c = data[chunk_offsets[c]:chunk_offsets[c+1]]
    chunk_samples: np.ndarray  # int32 [m] samples of chunk c (the pod5 signal table's `samples`)
    read_chunks: np.ndarray    # int64 [n+1] CSR: the chunks of each read
    offset: np.ndarray         # float32 [n] calibration_offset
    scale: np.ndarray          # float32 [n] calibration_scale
    stride: int                # row length (the preload size); chunks past it are not needed


@dataclass
class MinibatchResult:
    labels: np.ndarray            # int64 [n] predicted barcode, -1 = unclassified or no fingerprint
    conf: np.ndarray              # float64 [n] confidence margin (NaN without a fingerprint)
    prob: np.ndarray              # float64 [n, k]
    fp_status: np.ndarray         # int32 [n] 0 = fingerprint ok, else the fingerprint stage's status
    detect_success: np.ndarray    # uint8 [n]
    detect_code: np.ndarray       # int32 [n] validation fail code (detect.combined.FAIL_REASONS)
    detect_checks: np.ndarray     # int32 [n]
    bounds: np.ndarray            # int64 [n, 3] adapter_start, adapter_end, polya_end
    preds: np.ndarray             # int64 [n, 1 + k] raw CNN boundaries
    llr_rescued: np.ndarray       # bool [n] boundaries came from the llr_fallback callback
    predictions: Optional[pd.DataFrame]   # reads with a fingerprint: '#read_id', predicted_barcode, confidence_score, pXX..
    fpt: Optional[np.ndarray] = None      # float64 [n, L] when asked for
    detect_source: Optional[np.ndarray] = None   # int32 [n] bits 0-1: boundaries validated (0 CNN, 1 hail mary, 2 device LLR);
                                                 # bit 2 / 3: the hail-mary / full LLR re-detection ran for this read

    @property
    def passed(self) -> np.ndarray:
        return self.fp_status == 0

    def fail_reason(self, i: int) -> Optional[str]:
        if self.fp_status[i] == 0:
            return None
        if not self.detect_success[i]:
            return _combined.fail_reason(int(self.detect_code[i]), int(self.detect_checks[i]))
        return FP_STATUS_REASON.get(int(self.fp_status[i]), "fingerprint failed")


class MinibatchDemuxer:
    """`model_predict`: warpdemux_b200 DTW_SVM; `model_detect`: detect.cnn.BoundariesCNN; `spc`: the reference's
    SigProcConfig (or the three config mirrors given explicitly)."""

    def __init__(self, model_predict, model_detect: "_cnn.BoundariesCNN", spc=None, *, core=None, cnn_boundaries=None,
                 validate_config: Optional["_combined.ValidateConfig"] = None, fp_config: Optional[FingerprintConfig] = None,
                 device: Optional[int] = None, mode: Optional[str] = None, cnn_mode: Optional[str] = None,
                 llr_fallback: Optional[Callable] = None, consensus_query=None, full_detect_report: bool = False,
                 llr="auto", lanes: int = 4, overlap_llr_tail: bool = True):
        import torch  # device memory and streams only

        self._torch = torch
        self.device = default_device() if device is None else int(device)
        self.model_predict, self.model_detect = model_predict, model_detect
        self.core = core if core is not None else (spc.core if spc is not None else _cnn.CoreConfig())
        self.cnn_boundaries = cnn_boundaries if cnn_boundaries is not None else (
            spc.cnn_boundaries if spc is not None else _cnn.CNNBoundariesConfig())
        vcfg = validate_config if validate_config is not None else (
            _combined.ValidateConfig.from_spc(spc) if spc is not None else _combined.ValidateConfig())
        fcfg = fp_config if fp_config is not None else (
            FingerprintConfig.from_spc(spc, consensus_query) if spc is not None else FingerprintConfig())
        # the fingerprint stage needs the verdict and the boundaries only; full_detect_report=True also reproduces the
        # reference's fail_reason / mvs_* values of reads whose first poly(A) candidate fails (all candidates evaluated)
        if isinstance(llr, str):     # "auto": what the configuration says (the reference's defaults: both fallbacks on)
            llr = _combined.LLRConfig.from_spc(spc) if spc is not None else None
        self.validator = _combined.Validator(vcfg, device=self.device, verdict_only=not full_detect_report, llr=llr)
        if fcfg.max_slice_len <= 0:
            # a fixed shared-memory capacity keeps the fingerprint call free of its host synchronisation (the read-back of
            # the longest slice): the CNN's adapter end is < max_obs_adapter, the slice adds the padding on both sides
            import dataclasses

            cap = (int(self.core.max_obs_adapter) + 2 * int(fcfg.padding) + 63) // 64 * 64
            fcfg = dataclasses.replace(fcfg, max_slice_len=min(cap, 16000))
            if llr is not None:
                # an LLR adapter end may lie anywhere below max_obs_trace: those few reads get a second, larger pass
                cap2 = (int(llr.max_obs_trace) + int(fcfg.padding) + 63) // 64 * 64
                if cap2 > fcfg.max_slice_len:
                    fcfg = dataclasses.replace(fcfg, long_slice_len=min(cap2, 16000))
        self.fingerprinter = Fingerprinter(fcfg, device=self.device)
        # Lanes: `stream()` alternates consecutive minibatches between `lanes` compute streams, each with its OWN set of
        # library handles (their workspaces are per handle), so that the latency-bound tail of one minibatch (the few
        # reads of the LLR fallback, the finishing kernels) overlaps the wide kernels of the next.  Lane 0 = the objects
        # given; the others are replicas built from the same host-side parameters (created lazily).
        self.lanes = max(1, int(lanes))
        self.overlap_llr_tail = bool(overlap_llr_tail)   # fingerprints of the validated reads next to the LLR re-detection of the failed ones
        self._lane_objs = [dict(model_predict=model_predict, model_detect=model_detect, validator=self.validator,
                                fingerprinter=self.fingerprinter, stream=None)]
        self._lane_cfg = dict(vcfg=vcfg, fcfg=fcfg, llr=llr, verdict_only=not full_detect_report)
        self.mode = mode or model_predict.mode
        self.cnn_mode = cnn_mode or model_detect.mode
        self.llr_fallback = llr_fallback
        self.k_cand = int(self.cnn_boundaries.polya_cand_k)
        self._stream = None
        self._copy_stream = None
        self._buf = {}
        self._pin = {}

    # -- device plumbing ---------------------------------------------------------
    def _dev(self):
        return self._torch.device("cuda", self.device)

    def _get(self, name, shape, dtype):
        t = self._buf.get(name)
        need = int(np.prod(shape))
        if t is None or t.numel() < need or t.dtype != dtype:
            t = self._torch.empty(max(need, 1), dtype=dtype, device=self._dev())
            self._buf[name] = t
        return t[:need].view(*shape)

    # -- the three phases of one minibatch (slot = one set of device / pinned buffers) -----------------------
    def _streams(self):
        torch = self._torch
        if self._stream is None:
            self._stream = torch.cuda.Stream(device=self._dev(), priority=-1)   # kernels + result download (above the lanes' aux streams)
            self._copy_stream = torch.cuda.Stream(device=self._dev())   # minibatch upload
        return self._stream, self._copy_stream

    def _lane(self, i: int) -> dict:
        """Handles + compute stream of lane i (replicas of lane 0's objects for i > 0)."""
        torch = self._torch
        while len(self._lane_objs) <= i:
            c = self._lane_cfg
            mp0, md0 = self.model_predict, self.model_detect
            self._lane_objs.append(dict(
                model_predict=type(mp0)(mp0.params, device=self.device, mode=mp0.mode),
                model_detect=_cnn.BoundariesCNN(md0.weights, device=self.device, mode=md0.mode),
                validator=_combined.Validator(c["vcfg"], device=self.device, verdict_only=c["verdict_only"], llr=c["llr"]),
                fingerprinter=Fingerprinter(c["fcfg"], device=self.device), stream=None))
        ln = self._lane_objs[i]
        if ln["stream"] is None:
            ln["stream"] = self._streams()[0] if i == 0 else torch.cuda.Stream(device=self._dev(), priority=-1)
        return ln

    def _upload(self, slot: int, signals, full_lengths, read_ids) -> dict:
        """Phase 1 (copy stream): the minibatch goes to the device.  Pageable rows are first copied into the slot's
        pinned staging block so that the H2D transfer itself is asynchronous."""
        torch = self._torch
        st, cst = self._streams()
        job = {"slot": slot, "read_ids": read_ids}
        if isinstance(signals, AdcBatch):
            return self._upload_adc(job, signals, full_lengths)
        if isinstance(signals, VbzBatch):
            return self._upload_vbz(job, signals, full_lengths)
        if isinstance(signals, torch.Tensor):
            if signals.dtype != torch.float32 or signals.dim() != 2 or not signals.is_contiguous():
                raise ValueError("signals tensor must be contiguous float32 [n, stride]")
            h_sig = None if signals.is_cuda else signals
            d_sig = signals if signals.is_cuda else None
        else:
            h_sig, d_sig = torch.from_numpy(_cnn._as_batch(signals)), None
        n, stride = (d_sig if d_sig is not None else h_sig).shape
        lens = np.ascontiguousarray(np.minimum(np.asarray(full_lengths, dtype=np.int64).reshape(-1), np.iinfo(np.int32).max), dtype=np.int32)
        if lens.shape[0] != n:
            raise ValueError("full_lengths must have one entry per signal row")
        job.update(n=n, stride=stride, lens=lens, h_sig=h_sig)
        if d_sig is not None:
            cst.wait_stream(torch.cuda.current_stream())   # the caller produced the tensor on its current stream
        with torch.cuda.stream(cst):
            if d_sig is None:
                if not h_sig.is_pinned():
                    pin = self._pinned(f"{slot}:sig", n * stride, torch.float32).view(n, stride)
                    pin.copy_(h_sig)
                    h_sig = pin
                d_sig = self._get(f"{slot}:sig", (n, stride), torch.float32)
                d_sig.copy_(h_sig, non_blocking=True)
            d_len = self._get(f"{slot}:len", (n,), torch.int32)
            pin_len = self._pinned(f"{slot}:len", n, torch.int32)
            pin_len.copy_(torch.from_numpy(lens))
            d_len.copy_(pin_len, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(cst)
        job.update(d_sig=d_sig, d_len=d_len, ev_h2d=ev)
        return job

    def _upload_adc(self, job: dict, b: AdcBatch, full_lengths) -> dict:
        """Phase 1 for raw ADC input: int16 rows + calibration go up, the float32 pA rows are made on the device."""
        torch = self._torch
        st, cst = self._streams()
        slot = job["slot"]
        adc = b.adc if isinstance(b.adc, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(b.adc, dtype=np.int16))
        if adc.dtype != torch.int16 or adc.dim() != 2 or not adc.is_contiguous() or adc.is_cuda:
            raise ValueError("AdcBatch.adc must be a contiguous int16 [n, stride] host array")
        n, stride = adc.shape
        lens = np.ascontiguousarray(np.minimum(np.asarray(full_lengths, dtype=np.int64).reshape(-1), np.iinfo(np.int32).max), dtype=np.int32)
        small = np.empty((3, n), dtype=np.float32)            # one small upload: n_valid (as int32 bits), offset, scale
        small[0] = np.minimum(np.asarray(b.num_samples, dtype=np.int64).reshape(-1), stride).astype(np.int32).view(np.float32)
        small[1] = np.asarray(b.offset, dtype=np.float32).reshape(-1)
        small[2] = np.asarray(b.scale, dtype=np.float32).reshape(-1)
        if lens.shape[0] != n:
            raise ValueError("full_lengths must have one entry per signal row")
        job.update(n=n, stride=stride, lens=lens, h_sig=None)
        with torch.cuda.stream(cst):
            if not adc.is_pinned():
                pin = self._pinned(f"{slot}:adc", n * stride, torch.int16).view(n, stride)
                pin.copy_(adc)
                adc = pin
            d_adc = self._get(f"{slot}:adc", (n, stride), torch.int16)
            d_adc.copy_(adc, non_blocking=True)
            pin_small = self._pinned(f"{slot}:cal", 3 * n, torch.float32).view(3, n)
            pin_small.copy_(torch.from_numpy(small))
            d_small = self._get(f"{slot}:cal", (3, n), torch.float32)
            d_small.copy_(pin_small, non_blocking=True)
            d_len = self._get(f"{slot}:len", (n,), torch.int32)
            pin_len = self._pinned(f"{slot}:len", n, torch.int32)
            pin_len.copy_(torch.from_numpy(lens))
            d_len.copy_(pin_len, non_blocking=True)
            d_sig = self._get(f"{slot}:sig", (n, stride), torch.float32)
            if n:
                rc = _lib.load().wdx_calibrate_rows(d_adc.data_ptr(), n, stride, d_small[0].data_ptr(), d_small[1].data_ptr(),
                                                    d_small[2].data_ptr(), d_sig.data_ptr(), stride, self.device, cst.cuda_stream)
                _lib.check(rc, "wdx_calibrate_rows")
            ev = torch.cuda.Event()
            ev.record(cst)
        job.update(d_sig=d_sig, d_len=d_len, ev_h2d=ev, h2d_bytes=int(n) * int(stride) * 2)
        return job

    def _upload_vbz(self, job: dict, b: VbzBatch, full_lengths) -> dict:
        """Phase 1 for pod5 VBZ chunks: the compressed bytes and the small arrays go up from one pinned staging block
        (two copies), then wdx_vbz_decode_rows -> int16 rows -> wdx_calibrate_rows, all on the copy stream.  The per-read
        decode status joins the result block (_launch) and is checked in _finalize."""
        torch = self._torch
        st, cst = self._streams()
        slot = job["slot"]
        stride = int(b.stride)
        rc = np.ascontiguousarray(b.read_chunks, dtype=np.int64).reshape(-1)
        n = rc.size - 1
        samples = np.ascontiguousarray(b.chunk_samples, dtype=np.int32).reshape(-1)
        coff = np.ascontiguousarray(b.chunk_offsets, dtype=np.int64).reshape(-1)
        data = np.asarray(b.data, dtype=np.uint8).reshape(-1)
        if stride < 1 or n < 0 or coff.size != samples.size + 1 or (coff.size and (coff[0] != 0 or coff[-1] != data.size or np.any(np.diff(coff) < 0))):
            raise ValueError("VbzBatch: chunk_offsets must be [m+1] non-decreasing offsets into data, chunk_samples [m], stride >= 1")
        soff = _vbz.scratch_layout(samples, rc, stride)
        lens = np.ascontiguousarray(np.minimum(np.asarray(full_lengths, dtype=np.int64).reshape(-1), np.iinfo(np.int32).max), dtype=np.int32)
        if lens.shape[0] != n:
            raise ValueError("full_lengths must have one entry per read")
        # small arrays: one int64-aligned block
        parts = [("coff", coff), ("soff", soff), ("rc", rc), ("samples", samples), ("len", lens),
                 ("offset", np.asarray(b.offset, dtype=np.float32).reshape(-1)), ("scale", np.asarray(b.scale, dtype=np.float32).reshape(-1))]
        if parts[5][1].size != n or parts[6][1].size != n:
            raise ValueError("VbzBatch: offset / scale need one entry per read")
        at, pos = {}, 0
        for name, a in parts:
            at[name] = (pos, a)
            pos += (a.nbytes + 15) // 16 * 16
        nbytes_data = (data.size + 15) // 16 * 16
        job.update(n=n, stride=stride, lens=lens, h_sig=None)
        with torch.cuda.stream(cst):
            pin = self._pinned(f"{slot}:vbz", nbytes_data + pos, torch.uint8)
            hp = pin.numpy()
            hp[:data.size] = data
            for name, (o, a) in at.items():
                hp[nbytes_data + o:nbytes_data + o + a.nbytes] = a.view(np.uint8)
            d_bytes = self._get(f"{slot}:vbz_bytes", (max(nbytes_data, 16),), torch.uint8)
            d_small = self._get(f"{slot}:vbz_small", (max(pos, 16),), torch.uint8)
            if nbytes_data:
                d_bytes[:nbytes_data].copy_(pin[:nbytes_data], non_blocking=True)
            d_small[:pos].copy_(pin[nbytes_data:nbytes_data + pos], non_blocking=True)
            tdt = {np.dtype(np.int64): torch.int64, np.dtype(np.int32): torch.int32, np.dtype(np.float32): torch.float32}
            v = {name: d_small[o:o + a.nbytes].view(tdt[a.dtype]) for name, (o, a) in at.items()}
            d_scr = self._get(f"{slot}:vbz_scratch", (max(int(soff[-1]), 16),), torch.uint8)
            d_adc = self._get(f"{slot}:adc", (n, stride), torch.int16)
            d_dec = self._get(f"{slot}:vbz_dec", (2, n), torch.int32)    # n_valid, status
            d_sig = self._get(f"{slot}:sig", (n, stride), torch.float32)
            if n:
                _vbz.decode_rows_raw(d_bytes, v["coff"], v["samples"], v["rc"], d_scr, v["soff"], d_adc, d_dec[0], d_dec[1],
                                     self.device, cst.cuda_stream)
                rc_ = _lib.load().wdx_calibrate_rows(d_adc.data_ptr(), n, stride, d_dec[0].data_ptr(), v["offset"].data_ptr(),
                                                     v["scale"].data_ptr(), d_sig.data_ptr(), stride, self.device, cst.cuda_stream)
                _lib.check(rc_, "wdx_calibrate_rows")
            ev = torch.cuda.Event()
            ev.record(cst)
        job.update(d_sig=d_sig, d_len=v["len"], ev_h2d=ev, d_vbz_status=d_dec[1], h2d_bytes=int(data.size) + pos)
        return job

    def _launch(self, job: dict, want_fpt: bool) -> None:
        """Phase 2 (the lane's compute stream): CNN -> validation / LLR -> fingerprint + DTW/SVC, then the result download."""
        torch = self._torch
        lane = self._lane(job.get("lane", 0))
        st = lane["stream"]
        dm = lane["model_predict"]._device_model()
        k, L = self.model_predict.params.k, self.model_predict.params.L
        n, stride, slot, lens = job["n"], job["stride"], job["slot"], job["lens"]
        ld = 1 + self.k_cand
        d_sig, d_len = job["d_sig"], job["d_len"]
        g = lambda name, shape, dt: self._get(f"{slot}:{name}", shape, dt)
        with torch.cuda.stream(st):
            st.wait_event(job["ev_h2d"])
            # every per-read result lives in ONE device block (8-byte aligned sections) mirrored by one pinned block
            spec = [("preds", (n, ld), torch.int64), ("bounds", (n, 3), torch.int64), ("lab", (n,), torch.int64),
                    ("conf", (n,), torch.float64), ("prob", (n, k), torch.float64), ("info", (n, 4), torch.int32),
                    ("status", (n,), torch.int32), ("suc", (n,), torch.uint8), ("flags", (n,), torch.uint8)]
            if want_fpt:
                spec.insert(0, ("fpt", (n, L), torch.float64))
            if "d_vbz_status" in job:
                spec.append(("vbz_status", (n,), torch.int32))
            sizes = [(int(np.prod(shape)) * torch.empty(0, dtype=dt).element_size() + 7) // 8 * 8 for _, shape, dt in spec]
            total = sum(sizes)
            d_block = g("results", (max(total, 8),), torch.uint8)
            h_block = self._pinned(f"{slot}:results", max(total, 8), torch.uint8)
            views, hviews, off = {}, {}, 0
            for (name, shape, dt), sz in zip(spec, sizes):
                nbytes = int(np.prod(shape)) * torch.empty(0, dtype=dt).element_size()
                views[name] = d_block[off:off + nbytes].view(dt).view(*shape)
                hviews[name] = h_block[off:off + nbytes].view(dt).view(*shape)
                off += sz
            d_preds, d_bounds, d_lab, d_conf, d_prob = views["preds"], views["bounds"], views["lab"], views["conf"], views["prob"]
            d_info, d_status, d_suc = views["info"], views["status"], views["suc"]
            d_fpt = views.get("fpt")
            if d_fpt is None:     # kept on the device anyway: a guard-list overflow is repaired from it (_finalize)
                d_fpt = g("fpt_dev", (n, L), torch.float64)
            d_flags = views["flags"]
            if "d_vbz_status" in job:
                views["vbz_status"].copy_(job["d_vbz_status"])
            d_a0, d_a1 = g("a0", (n,), torch.int64), g("a1", (n,), torch.int64)
            sp = st.cuda_stream
            rescued = np.zeros(n, dtype=bool)
            if n:
                _cnn.detect_raw(lane["model_detect"], self.core, self.k_cand, d_sig, n, stride, d_preds, mode=self.cnn_mode, stream=sp)
                # Reads that pass the first validation are final there (the LLR re-detection only revisits failed reads), so
                # their fingerprints are computed on a second stream WHILE the re-detection tail runs; the fused call below
                # then only revisits the reads that were failed at that point (status FP_FAIL_DETECT) and may have been rescued.
                early = self.overlap_llr_tail and self.llr_fallback is None and lane["validator"].llr is not None
                if early:
                    if lane.get("aux") is None:
                        # lowest priority: the few CTAs of the re-detection tail are placed first, the fingerprint pass fills the rest
                        lane["aux"] = torch.cuda.Stream(device=self._dev(), priority=0)
                        lane["ev_main"] = torch.cuda.Event()
                        lane["ev_main"].record(st)      # creates the CUDA event (torch does it lazily)
                        lane["ev_p1"] = torch.cuda.Event()
                    d_snap = g("snap_ok", (n,), torch.uint8)
                    lane["validator"].set_early(d_snap, lane["ev_main"])
                lane["validator"].run_raw(d_sig, n, stride, d_len, d_preds, ld, d_suc, d_info, d_bounds, None, stream=sp)
                if early:
                    aux = lane["aux"]
                    with torch.cuda.stream(aux):
                        aux.wait_event(lane["ev_main"])
                        d_a0.copy_(d_bounds[:, 0])
                        d_a1.copy_(d_bounds[:, 1])
                        lane["fingerprinter"].extract_raw(d_sig, n, stride, d_a0, d_a1, d_fpt, d_status, detect_ok=d_snap,
                                                          stream=aux.cuda_stream)
                        lane["ev_p1"].record(aux)
                    st.wait_event(lane["ev_p1"])
                    lane["fingerprinter"].set_resume_status(2)      # WDX_FP_FAIL_DETECT
                if self.llr_fallback is not None:
                    suc_h = d_suc.cpu().numpy()            # synchronises this stream: n bytes
                    failed = np.flatnonzero(suc_h == 0)
                    if failed.size:
                        h_sig = job["h_sig"]
                        rows = d_sig[torch.from_numpy(failed).to(self._dev())].cpu().numpy() if h_sig is None else h_sig.numpy()[failed]
                        b_h = d_bounds.cpu().numpy()
                        for j, i in enumerate(failed):
                            res = self.llr_fallback(rows[j], int(lens[i]))
                            if res is not None and getattr(res, "success", False):
                                b_h[i] = (int(res.adapter_start or 0), int(res.adapter_end), int(res.polya_end or 0))
                                suc_h[i] = 1
                                rescued[i] = True
                        d_bounds.copy_(torch.from_numpy(b_h))
                        d_suc.copy_(torch.from_numpy(suc_h))
                d_a0.copy_(d_bounds[:, 0])
                d_a1.copy_(d_bounds[:, 1])
                lane["fingerprinter"].predict_raw(dm, d_sig, n, stride, d_a0, d_a1, _lib.MODES[self.mode], d_lab, d_status,
                                               conf=d_conf, prob=d_prob, fpt=d_fpt, detect_ok=d_suc, stream=sp, flags=d_flags)
            h_block[:max(total, 8)].copy_(d_block, non_blocking=True)      # one download, does not block the host
            host = hviews
            ev = torch.cuda.Event()
            ev.record(st)
        job.update(host=host, ev_done=ev, rescued=rescued, d_fpt=d_fpt, dev=views)

    def _finalize(self, job: dict, return_df: bool) -> MinibatchResult:
        """Phase 3 (host): wait for the download, copy out of the pinned blocks, build the DataFrame."""
        job["ev_done"].synchronize()
        h = {k: v.numpy().copy() for k, v in job["host"].items()}
        if "vbz_status" in h and h["vbz_status"].any():
            # a pod5 chunk that does not decode is an I/O error of the input file, not a per-read verdict
            bad = np.flatnonzero(h["vbz_status"])
            rid = job["read_ids"]
            name = lambda i: rid[i] if rid is not None else f"row {i}"
            raise _lib.WdxError(f"read {name(bad[0])}: VBZ signal could not be decoded ({_vbz.status_name(h['vbz_status'][bad[0]])}, "
                                f"status {int(h['vbz_status'][bad[0]])}); {bad.size} of {job['n']} reads of the minibatch failed")
        labels, conf, prob, status = h["lab"], h["conf"], h["prob"], h["status"]
        flags = h["flags"]
        over = np.flatnonzero((flags & _lib.FLAG_GUARD_OVERFLOW) != 0)
        if over.size:
            # GUARDED mode listed more boundary reads than its re-run list holds (max(4096, n/64) per launch): those kept
            # their FAST_F32 results; redo them in EXACT_F64 from the fingerprints still on the device
            torch = self._torch
            sel = torch.from_numpy(over).to(self._dev())
            lane = self._lane(job.get("lane", 0))
            with torch.cuda.stream(lane["stream"]):
                x = job["d_fpt"].index_select(0, sel).contiguous()
                k = prob.shape[1]
                lab2 = torch.empty(over.size, dtype=torch.int64, device=self._dev())
                conf2 = torch.empty(over.size, dtype=torch.float64, device=self._dev())
                prob2 = torch.empty((over.size, k), dtype=torch.float64, device=self._dev())
                lane["model_predict"]._device_model().predict_raw(x, over.size, _lib.WDX_F64, _lib.MODE_EXACT_F64, lab2, conf2, prob2,
                                                                  stream=lane["stream"].cuda_stream)
                labels[over], conf[over], prob[over] = lab2.cpu().numpy(), conf2.cpu().numpy(), prob2.cpu().numpy()
        # a fingerprint whose decision values are not finite: the reference's predict raises (sklearn check_array); here the
        # read is reported as failed with its own status instead of silently becoming "unclassified"
        status[(status == 0) & ((flags & _lib.FLAG_NONFINITE) != 0)] = FP_NONFINITE
        predictions = None
        if return_df:
            good = status == 0
            predictions = predictions_to_df(labels[good], prob[good], conf[good], self.model_predict.label_mapper)
            rid = job["read_ids"]
            ids = np.asarray(rid if rid is not None else np.arange(job["n"]))[good]
            predictions = add_read_id_col_to_predictions(predictions, ids)
        return MinibatchResult(labels, conf, prob, status, h["suc"], h["info"][:, 0].copy(), h["info"][:, 1].copy(), h["bounds"],
                               h["preds"], job["rescued"], predictions, h.get("fpt"), detect_source=h["info"][:, 3].copy())

    def _pinned(self, name, numel, dtype):
        t = self._pin.get(name)
        if t is None or t.numel() < numel or t.dtype != dtype:
            t = self._torch.empty(max(int(numel), 1), dtype=dtype).pin_memory()
            self._pin[name] = t
        return t[:numel]

    def run(self, signals, full_lengths, read_ids: Optional[Sequence] = None, return_df: bool = True,
            want_fpt: bool = False) -> MinibatchResult:
        """One minibatch.  signals: float32 [n, stride] NaN-padded rows (numpy; torch CPU tensor, pinned or not; or a CUDA
        tensor), an `AdcBatch` of raw int16 samples or a `VbzBatch` of compressed pod5 signal chunks (a chunk that does
        not decode raises WdxError naming the read); full_lengths: [n] full read lengths (file_proc.py:241-262)."""
        with self._torch.cuda.device(self.device):
            job = self._upload(0, signals, full_lengths, read_ids)
            self._launch(job, want_fpt)
            return self._finalize(job, return_df)

    def stream(self, minibatches, return_df: bool = True, want_fpt: bool = False):
        """Generator over an iterable of minibatches `(signals, full_lengths[, read_ids])`, results in order.
        Three buffer slots: while the kernels of minibatch i run, minibatch i+1 is already launched behind them and
        minibatch i+2 is uploading on the copy stream — the reference overlaps loading and computing with a loader
        process feeding a queue (file_proc.py:333-377)."""
        with self._torch.cuda.device(self.device):
            it = iter(minibatches)

            def up(slot, mb):
                return self._upload(slot, mb[0], mb[1], mb[2] if len(mb) > 2 else None)

            LANES = self.lanes
            SLOTS = LANES + 2     # buffer sets: one per launched minibatch + the upload ahead of them
            pending = []          # uploaded or launched jobs, oldest first
            i = 0                 # minibatches uploaded so far

            def upload_next():
                nonlocal i
                mb = next(it, None)
                if mb is None:
                    return False
                job = up(i % SLOTS, mb)
                job["lane"] = i % LANES
                pending.append([job, False])
                i += 1
                return True

            more = True
            for _ in range(LANES + 1):                  # uploads in flight before the first launch
                more = more and upload_next()
            while pending:
                for pj in pending[:LANES + 1]:          # keep one minibatch per lane launched + one queued behind them
                    if not pj[1]:
                        self._launch(pj[0], want_fpt)
                        pj[1] = True
                done = pending.pop(0)
                res = self._finalize(done[0], return_df)    # frees the oldest slot ...
                if more:
                    more = upload_next()                    # ... for the upload of minibatch i+2
                yield res

    def close(self):
        for ln in self._lane_objs[1:]:
            ln["validator"].close()
            ln["fingerprinter"].close()
            ln["model_detect"].close()
        self._lane_objs = self._lane_objs[:1]
        self.validator.close()
        self.fingerprinter.close()
        self._buf = {}
        self._pin = {}


def detect_and_predict_on_preloaded_signals(preloaded_minibatch, model_predict, model_detect, config,
                                            demuxer: Optional[MinibatchDemuxer] = None) -> MinibatchResult:
    """Argument order of the reference worker (file_proc.py:380-390) without its queues: `preloaded_minibatch` =
    (signals, _, full_lengths, read_ids); `config.sig_proc` is the SigProcConfig."""
    signals, _, full_lengths, read_ids = preloaded_minibatch
    spc = config.sig_proc if hasattr(config, "sig_proc") else config
    if getattr(spc, "primary_method", "cnn") != "cnn":
        raise NotImplementedError("only primary_method = 'cnn' is on the GPU path (llr / start_peak detection stay with the reference)")
    d = demuxer or MinibatchDemuxer(model_predict, model_detect, spc)
    try:
        return d.run(signals, full_lengths, read_ids, return_df=True)
    finally:
        if demuxer is None:
            d.close()


def demux_minibatches_to_dir(minibatches, model_predict, model_detect, spc, writer, predict: bool = True,
                             validator: Optional["_combined.Validator"] = None, fp_config: Optional[FingerprintConfig] = None) -> dict:
    """The reference's demux / prep run over an iterable of preloaded minibatches `(signals, full_lengths, read_ids)`
    with its four outputs written as it writes them (file_proc.py:380-455 per minibatch, :627-724 writers):
    detected_boundaries_*.csv.gz, failed_reads_*.csv.gz, barcode_fpts_*.npz, barcode_predictions_*.csv.gz through
    `writer` (io.results.RunDirWriter; reads it already holds from `continue_from` are skipped, file_proc.py:205-214).
    The full-report path: every DetectResults field of the reference's tables is produced (partition statistics, open
    pores, fail reasons of the last poly(A) candidate), so it runs the three stages as separate calls instead of the
    fused `MinibatchDemuxer` chain."""
    from .sig_proc import batch_detect_results_to_fpt

    v = validator or _combined.Validator(spc, device=getattr(model_detect, "device", None))
    counts = {"reads": 0, "pass": 0, "fail": 0, "skipped": 0}
    try:
        for mb in minibatches:
            signals, full_lengths, read_ids = mb[0], mb[1], mb[2]
            signals = _cnn._as_batch(signals)
            keep = np.array([rid not in writer.processed for rid in read_ids], dtype=bool)
            counts["skipped"] += int((~keep).sum())
            if not keep.all():
                signals, full_lengths = signals[keep], np.asarray(full_lengths)[keep]
                read_ids = [rid for rid, k in zip(read_ids, keep) if k]
            if len(read_ids) == 0:
                continue
            dets = _combined.combined_detect_cnn(signals, full_lengths, model_detect, spc, validator=v, partitions=True)
            results = batch_detect_results_to_fpt(signals, fp_config if fp_config is not None else spc, dets)
            for r, rid in zip(results, read_ids):
                r.set_read_id(rid)
            ok = [r for r in results if r.success]
            predictions = None
            if predict and ok:
                predictions = model_predict.predict(np.vstack([r.barcode_fpt for r in ok]), pbar=False, nproc=1, return_df=True)
                predictions = add_read_id_col_to_predictions(predictions, [r.read_id for r in ok])
            writer.add(results, predictions)
            counts["reads"] += len(results)
            counts["pass"] += len(ok)
            counts["fail"] += len(results) - len(ok)
    finally:
        if validator is None:
            v.close()
    writer.close()
    return counts

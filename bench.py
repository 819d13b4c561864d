#!/usr/bin/env python
"""bench.py — reads/s of the WarpDemuX classification hot path on B200.

    python bench.py --gpus N --steps K --warmup W          # this framework
    python bench.py --impl reference --steps K --warmup W  # reference CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                 # + outputs of the last timed step as DIR/*.npy

Workload (BASELINE.json metric / configs[2]): WDX10_rna004_v1_0 (2601 support
vectors, 11 classes, L=25, window 15) on synthetic barcode fingerprints S1
(support vector + 0.35*N(0,1), SURVEY.md §8d).  100 M reads across 8 GPUs =
12.5 M reads per GPU per step; reads are sharded by contiguous index range, one
process per GPU, no data-path collective (weak scaling).

A "step" = one pass of the fused path (DTW distance to every support vector ->
DTW-kernel SVC probabilities -> thresholded barcode call) over this rank's
batch.  `value` is timed with CUDA events with the batch already in HBM;
`e2e` goes through the reference-facing API `DTW_SVM.predict(X_host)` with
host buffers (H2D and D2H inside the timed region).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL = "WDX10_rna004_v1_0"
METRIC = "reads/s demuxed (WDX10 DTW+SVC)"
READS_PER_GPU = 12_500_000  # 100 M / 8
SIGMA = 0.35
DUMP_ROWS = 1 << 18         # --dump-outputs sample: 2^18 reads x (index, label, confidence, 11 probabilities, flags) x 8 B = 31 MB
DUMP_SEED = 2024


def load_params():
    from warpdemux_b200 import model_io

    return model_io.load_npz(os.path.join(ROOT, "tests", "golden", "models", MODEL + ".npz"))


def synth_host(params, n, seed):
    """S1 fingerprints, generated in 1 M-row blocks (bounded host memory spikes)."""
    rng = np.random.default_rng(seed)
    X = np.empty((n, params.L), dtype=np.float64)
    for r0 in range(0, n, 1 << 20):
        r1 = min(n, r0 + (1 << 20))
        idx = rng.integers(0, params.n_sv, size=r1 - r0)
        X[r0:r1] = params.sv[idx] + SIGMA * rng.standard_normal((r1 - r0, params.L))
    return X


def dump_outputs(out_dir, n, arrays):
    """Per-read results of the last timed step (what DeviceModel.predict returns: label, confidence, class probabilities,
    guard flags) for a fixed, seeded sample of this rank's n reads, as float64 DIR/<name>.npy, plus the sampled read
    indices.  The inputs are seeded as well, so two builds run with the same arguments can be compared file by file."""
    import torch

    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_ROWS, replace=False)) if n > DUMP_ROWS else np.arange(n)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "read_index.npy"), idx.astype(np.float64))
    sel = torch.from_numpy(idx).cuda()
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.index_select(0, sel).cpu().numpy().astype(np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, smax, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); smax.append(float(r[1])); pw.append(float(r[2]))
            except Exception:  # noqa: BLE001
                continue
            for nm, v in zip(names, r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(np.max(smax)), "power_w_max": float(np.max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


# ---- the reference's own Python (baseline/_ref: `pip install --target` of /root/reference, done by __graft_entry__.build()
# in the build container; git-ignored, travels with the working tree) on top of the dtaidistance shim --------------------
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
_REF_MODEL = None


def reference_python_available():
    return os.path.exists(os.path.join(REF_DIR, "warpdemux", "models", "dtw_svm.py")) and os.path.exists(
        os.path.join(REF_DIR, "warpdemux", "models", "model_files", MODEL + ".joblib"))


def _ref_init(model_name):
    """Pool initialiser: import the UNMODIFIED reference package and load its own shipped model file."""
    global _REF_MODEL
    import warnings

    import pandas  # noqa: F401  (before oracle/shim is importable: pandas probes for the real `bottleneck`)
    for q in (REF_DIR, os.path.join(ROOT, "oracle", "shim"), ROOT):
        if q not in sys.path:
            sys.path.insert(0, q)
    import joblib
    from warpdemux.models.dtw_svm import DTW_SVM  # noqa: F401

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        _REF_MODEL = joblib.load(os.path.join(REF_DIR, "warpdemux", "models", "model_files", model_name + ".joblib"))


def _ref_predict(X):
    """One production minibatch through the reference's stock call (file_proc.py:443-450)."""
    df = _REF_MODEL.predict(X, nproc=1, return_df=True)
    return df["predicted_barcode"].to_numpy()


def reference_python_arm(params, workers, seconds_target, steps=1, warmup=0, want_outputs=False):
    """`DTW_SVM.predict(X, nproc=1, return_df=True)` of the reference package, minibatches of <= 1000 reads over a
    ProcessPoolExecutor(workers) — how production runs it (file_proc.py:1197-1245).  dtaidistance (absent third-party C)
    is the shim backed by oracle/wdx_oracle.c; everything else (numpy/pandas glue, 104 MB scratch matrix per call,
    float32 kernel, sklearn's libsvm predict_proba, thresholds) is the reference's own code."""
    import multiprocessing as mp
    from concurrent.futures import ProcessPoolExecutor

    with ProcessPoolExecutor(workers, mp_context=mp.get_context("spawn"), initializer=_ref_init, initargs=(MODEL,)) as ex:
        probe = synth_host(params, 32, seed=123)
        list(ex.map(_ref_predict, [probe] * workers))                  # workers up, model loaded
        t0 = time.perf_counter()
        list(ex.map(_ref_predict, [probe] * workers))
        per_read = (time.perf_counter() - t0) / 32
        mb = int(max(16, min(1000, seconds_target / per_read)))
        n = mb * workers
        X = synth_host(params, n, seed=7)
        chunks = [X[i:i + mb] for i in range(0, n, mb)]
        for _ in range(warmup):
            list(ex.map(_ref_predict, chunks))
        t0 = time.perf_counter()
        for _ in range(steps):
            res = list(ex.map(_ref_predict, chunks))
        dt = (time.perf_counter() - t0) / steps
    if want_outputs:
        return n / dt, n, dt, X, np.concatenate(res)
    return n / dt, n, dt


def cpu_arm(params, threads, seconds_target, steps=1, warmup=0, want_outputs=False):
    """The reference's CPU path as restated in oracle/ (kind "port"): production
    style minibatches of 1000 reads over `threads` single-threaded workers."""
    from oracle import wdx_oracle as o

    o.lib()
    probe = synth_host(params, 64, seed=123)
    t0 = time.perf_counter()
    o.predict_c(params, probe)
    per_read = (time.perf_counter() - t0) / 64
    n = int(max(threads * 50, min(200_000, seconds_target / per_read * threads)))
    n = max(threads, (n // threads) * threads)
    mb = min(1000, max(1, n // threads))
    X = synth_host(params, n, seed=7)
    for _ in range(warmup):
        o.predict_threaded(params, X[: max(threads, n // 8)], threads, mb)
    t0 = time.perf_counter()
    for _ in range(steps):
        res = o.predict_threaded(params, X, threads, mb)
    dt = (time.perf_counter() - t0) / steps
    if want_outputs:
        return n / dt, n, dt, X, res
    return n / dt, n, dt


def _fp_cpu_worker(args):
    """Fingerprint oracle on a slice of reads (one process = one core)."""
    sig, a0, a1 = args
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle import wdx_oracle as o

    ok = 0
    for r in range(sig.shape[0]):
        valid = sig[r][~np.isnan(sig[r])]
        st, _, _, _ = o.fingerprint(valid, int(a0[r]), int(a1[r]))
        ok += st == 0
    return ok


def fingerprint_stage(params_small, local, stream, seconds_cpu=6.0):
    """Secondary measurements (rank 0, N=1): the fingerprint kernel on S4 synthetic
    adapter signals (SURVEY.md 8d), the fused signals -> calls minibatch step
    (BASELINE.json configs[3], WDX4 as the DTW-SVM shape proxy), and the oracle's
    fingerprint chain on the host cores."""
    import torch
    from concurrent.futures import ProcessPoolExecutor

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from wdx_testutil import synth_adapter_signals
    from warpdemux_b200 import _lib
    from warpdemux_b200.models.dtw_svm import DTW_SVM
    from warpdemux_b200.sig_proc import Fingerprinter, FingerprintConfig

    base, reps, width = 1024, 32, 9000
    sig, a0, a1 = synth_adapter_signals(base, seed=21, width=width)
    lens = (~np.isnan(sig)).sum(axis=1)
    sl = np.minimum(lens, a1 + 100) - np.maximum(0, a0 - 100)
    n = base * reps
    sig_h = torch.from_numpy(np.tile(sig, (reps, 1))).pin_memory()
    a0_h, a1_h = np.tile(a0, reps), np.tile(a1, reps)
    sd = sig_h.cuda()
    a0d, a1d = torch.from_numpy(a0_h).cuda(), torch.from_numpy(a1_h).cuda()
    fpt = torch.empty((n, 25), dtype=torch.float64, device="cuda")
    st = torch.empty(n, dtype=torch.int32, device="cuda")
    cap = int((sl.max() + 63) // 64 * 64)
    fp = Fingerprinter(FingerprintConfig(max_slice_len=cap), device=local)
    fp.enable_timing(True)
    for _ in range(3):
        fp.extract_raw(sd, n, width, a0d, a1d, fpt, st, stream=stream)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        fp.extract_raw(sd, n, width, a0d, a1d, fpt, st, stream=stream)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 3
    kms, kl = fp.last_kernel_ms()
    bytes_alg = int(sl.sum()) * 4 * reps + n * 25 * 8
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    out = {
        "workload": f"S4 synthetic adapter signals: {n} reads x {width} samples float32 (mean adapter slice {sl.mean():.0f}), "
                    "rna004_130bps@v1.0 segmentation config",
        "reads_per_s": n / (ms * 1e-3), "kernel_ms": kms, "kernel_launches": kl,
        "ok_fraction": float((st == 0).float().mean().item()),
        "roofline": {"bound": "hbm", "achieved": bytes_alg / (kms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                     "frac": bytes_alg / (kms * 1e-3) / 1e9 / hbm,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
                     "algorithmic_bytes_per_read": bytes_alg / n,
                     "note": "not an HBM-bound kernel in practice: one CTA per read walks ~35 short barrier-separated phases "
                             "(exact medians, float64 t-test in the reference's summation order, peak suppression, top-k, event means); "
                             "issue slots ~55 % busy, FP64 pipe ~20 % (profiles/r02_ncu_full_fingerprint_summary.json)"},
    }
    # end to end from pinned host memory (H2D of the signals inside the timed region)
    out_h = fp.extract(sig_h.numpy()[: 8192], a0_h[:8192], a1_h[:8192], want_dwell=False, want_stats=False)
    t0 = time.perf_counter()
    out_h = fp.extract(sig_h.numpy(), a0_h, a1_h, want_dwell=False, want_stats=False)
    dt = time.perf_counter() - t0
    out["e2e_reads_per_s"] = n / dt
    out["e2e_h2d_bytes"] = int(n * width * 4)
    # fused signals -> barcode calls (fingerprints stay on the device)
    mdl = DTW_SVM(params_small, device=local, mode="guarded")
    lab = torch.empty(n, dtype=torch.int64, device="cuda")
    dm = mdl._device_model()
    for _ in range(2):
        fp.predict_raw(dm, sd, n, width, a0d, a1d, _lib.MODES["guarded"], lab, st, stream=stream)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(3):
        fp.predict_raw(dm, sd, n, width, a0d, a1d, _lib.MODES["guarded"], lab, st, stream=stream)
    e1.record()
    torch.cuda.synchronize()
    out["fused_signals_to_calls"] = {"model": params_small.name if hasattr(params_small, "name") else "WDX4_rna004_v1_0",
                                     "reads_per_s": n / (e0.elapsed_time(e1) / 3 * 1e-3), "mode": "guarded"}
    # CPU: the oracle chain (numpy + scipy find_peaks + restated Cython) on all cores, bounded sample
    cores = os.cpu_count() or 1
    per = 24
    chunks = [(sig[i:i + per], a0[i:i + per], a1[i:i + per]) for i in range(0, min(base, per * cores * 2), per)]
    try:
        with ProcessPoolExecutor(cores) as ex:
            list(ex.map(_fp_cpu_worker, chunks[:cores]))  # warm the workers
            t0 = time.perf_counter()
            list(ex.map(_fp_cpu_worker, chunks))
            dtc = time.perf_counter() - t0
        nc = sum(c[0].shape[0] for c in chunks)
        out["cpu_baseline"] = {"value": nc / dtc, "unit": "reads/s", "cores": cores, "kind": "port",
                               "sample": f"{nc} S4 reads, oracle fingerprint chain (numpy medians, restated Cython t-test, "
                                         f"scipy find_peaks), one process per core"}
    except Exception as e:  # noqa: BLE001
        out["cpu_baseline"] = {"error": str(e)}
    fp.close()
    try:
        out["real_reads"] = fingerprint_real_reads(local, stream, hbm)
    except Exception as e:  # noqa: BLE001
        out["real_reads"] = {"error": str(e)}
    return out


def fingerprint_real_reads(local, stream, hbm):
    """The fingerprint kernel on the 4000 real reads of the reference's test file with the reference's own adapter
    boundaries (tests/golden/real4000_rna004_WDX4.npz), tiled x 8, device-resident: real adapters are shorter (mean slice
    3 300 samples) than the S4 synthetic ones, and 4 % of the reads carry no boundaries (failed detection)."""
    import torch

    from warpdemux_b200.sig_proc import Fingerprinter, FingerprintConfig

    ds = chain_dataset()
    if not ds["kind"].startswith("real"):
        return {"skipped": "tests/golden/_local absent"}
    with np.load(os.path.join(ROOT, "tests", "golden", "real4000_rna004_WDX4.npz")) as z:
        bounds, success = z["bounds"], z["success"]
    sig = ds["sig"]
    a0, a1 = bounds[:, 0].astype(np.int64).copy(), bounds[:, 1].astype(np.int64).copy()
    a0[success == 0] = 0
    a1[success == 0] = 0
    reps, base, width = 8, sig.shape[0], sig.shape[1]
    n = base * reps
    sd = torch.from_numpy(sig).cuda().repeat(reps, 1).contiguous()
    a0d, a1d = torch.from_numpy(a0).cuda().repeat(reps), torch.from_numpy(a1).cuda().repeat(reps)
    okd = torch.from_numpy(success.astype(np.uint8)).cuda().repeat(reps)
    fpt = torch.empty((n, 25), dtype=torch.float64, device="cuda")
    st = torch.empty(n, dtype=torch.int32, device="cuda")
    fp = Fingerprinter(FingerprintConfig(max_slice_len=6720), device=local)   # max_obs_adapter + 2 * padding, as the chain sets it
    fp.enable_timing(True)
    best = 1e30
    for r in range(5):
        fp.extract_raw(sd, n, width, a0d, a1d, fpt, st, detect_ok=okd, stream=stream)
        torch.cuda.synchronize()
        ms, _ = fp.last_kernel_ms()
        if r:
            best = min(best, ms)
    fp.close()
    ok = success == 1
    lens = np.minimum(ds["lens"], width)
    sl = (np.minimum(lens, a1 + 100) - np.maximum(0, a0 - 100))[ok]
    bytes_alg = (int(sl.sum()) * 4 + int(ok.sum()) * 25 * 8) * reps
    return {"workload": f"{n} reads = the 4000 real reads x {reps}, reference boundaries, mean adapter slice {sl.mean():.0f} samples",
            "reads_per_s": n / (best * 1e-3), "kernel_ms": best, "ok_fraction": float((st == 0).float().mean().item()),
            "roofline": {"bound": "hbm", "achieved": bytes_alg / (best * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                         "frac": bytes_alg / (best * 1e-3) / 1e9 / hbm}}


def trna_stage(params_small, local, stream):
    """BASELINE.json configs[3] (rank 0, N=1): consensus-guided (tRNA) fingerprint batch — the
    rna004_130bps@v1.0_tRNA segmentation (120 events, sub-sequence alignment of the consensus,
    second change-point pass, normalize_wrt) on consensus-shaped synthetic adapter signals, alone and
    fused with DTW+SVC (WDX4 as the DTW-SVM shape proxy: the shipped tRNA classifier is CatBoost, out of scope)."""
    import torch

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from wdx_testutil import synth_trna_signals
    from warpdemux_b200 import _lib
    from warpdemux_b200.models.dtw_svm import DTW_SVM
    from warpdemux_b200.sig_proc import Fingerprinter, FingerprintConfig

    with np.load(os.path.join(ROOT, "tests", "golden", "fingerprint_trna.npz")) as z:
        consensus = z["consensus"].astype(np.float64)
    base, reps, width = 512, 64, 9000
    sig, a0, a1 = synth_trna_signals(consensus, base, seed=23, width=width)
    lens = (~np.isnan(sig)).sum(axis=1)
    sl = np.minimum(lens, a1 + 100) - np.maximum(0, a0 - 100)
    n = base * reps
    sd = torch.from_numpy(np.tile(sig, (reps, 1))).cuda()
    a0d, a1d = torch.from_numpy(np.tile(a0, reps)).cuda(), torch.from_numpy(np.tile(a1, reps)).cuda()
    fpt = torch.empty((n, 25), dtype=torch.float64, device="cuda")
    st = torch.empty(n, dtype=torch.int32, device="cuda")
    cap = int((sl.max() + 63) // 64 * 64)
    fp = Fingerprinter(FingerprintConfig.trna(consensus, max_slice_len=cap), device=local)
    fp.enable_timing(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, it=3):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(it):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / it

    ms = timed(lambda: fp.extract_raw(sd, n, width, a0d, a1d, fpt, st, stream=stream))
    kms, kl = fp.last_kernel_ms()
    ok = float((st == 0).float().mean().item())
    bytes_alg = int(sl.sum()) * 4 * reps + n * 25 * 8
    out = {"workload": f"consensus-shaped synthetic adapter signals: {n} reads x {width} samples float32 (mean adapter slice "
                       f"{sl.mean():.0f}), rna004_130bps@v1.0_tRNA segmentation config, consensus of {consensus.size} events",
           "reads_per_s": n / (ms * 1e-3), "kernel_ms": kms, "kernel_launches": kl, "ok_fraction": ok,
           "algorithmic_GBps": bytes_alg / (kms * 1e-3) / 1e9}
    mdl = DTW_SVM(params_small, device=local, mode="guarded")
    lab = torch.empty(n, dtype=torch.int64, device="cuda")
    dm = mdl._device_model()
    ms2 = timed(lambda: fp.predict_raw(dm, sd, n, width, a0d, a1d, _lib.MODES["guarded"], lab, st, stream=stream))
    out["fused_signals_to_calls"] = {"model": "WDX4_rna004_v1_0 (DTW-SVM shape proxy)", "reads_per_s": n / (ms2 * 1e-3),
                                     "mode": "guarded"}
    fp.close()
    return out


_CHAIN_DATA = None


def chain_dataset():
    """Reads for the raw-signal measurements: the 4000 real reads of the reference's own test file
    (test_data/demux/4000_rna004.pod5; first 11 500 samples each as int16 ADC + calibration, written by
    oracle/make_golden_real4000.py into tests/golden/_local — git-ignored, travels with the working tree), where 4.95 % of
    the reads leave the plain CNN path like in production.  Without that file: synthetic adapter + poly(A) + RNA rows
    (scripts/validate_probe.py), on which the real-data CNN misplaces ~20 % of the poly(A) ends (far more fallback work).
    Returns dict(kind, sig float32 [n, 11500] NaN padded, lens int32 [n] full read lengths, adc int16 [n, 11500], num int64 [n],
    offset / scale float32 [n])."""
    global _CHAIN_DATA
    if _CHAIN_DATA is not None:
        return _CHAIN_DATA
    stride = 11500
    local_file = os.path.join(ROOT, "tests", "golden", "_local", "real4000_adc_rows.npz")
    if os.path.exists(local_file):
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from wdx_testutil import real4000_rows

        with np.load(os.path.join(ROOT, "tests", "golden", "real4000_rna004_WDX4.npz")) as z:
            g = {k: z[k] for k in ("preload_size", "full_lengths", "subset", "calibration_offset", "calibration_scale")}
        with np.load(local_file) as z:
            full = {k: z[k] for k in z.files}
        _, sig, adc, num = real4000_rows(g, full)
        _CHAIN_DATA = dict(kind="real: the 4000 reads of test_data/demux/4000_rna004.pod5 (first 11 500 samples)", sig=sig,
                           lens=g["full_lengths"].astype(np.int32), adc=adc, num=num, offset=g["calibration_offset"].astype(np.float32),
                           scale=g["calibration_scale"].astype(np.float32))
    else:
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        from validate_probe import synth_reads

        sig, lens, _, _ = synth_reads(1024, stride)
        cal_scale, cal_off = np.float32(0.1755), np.float32(-243.0)
        adc = np.where(np.isnan(sig), 0, np.rint(np.nan_to_num(sig) / cal_scale - cal_off)).astype(np.int16)
        n = sig.shape[0]
        _CHAIN_DATA = dict(kind="synthetic adapter + poly(A) + RNA rows (tests/golden/_local absent)", sig=sig, lens=lens.astype(np.int32), adc=adc,
                           num=np.minimum(lens, stride).astype(np.int64), offset=np.full(n, cal_off, np.float32), scale=np.full(n, cal_scale, np.float32))
    return _CHAIN_DATA


def raw_signal_chain(params_small, local):
    """The production minibatch step from raw signal (reference file_proc.py:380-455, BASELINE.json configs[0] shape) on
    synthetic reads (adapter + poly(A) plateau + RNA): boundary CNN -> boundary validation -> fingerprint -> DTW+SVC,
    chained on one stream through device buffers (warpdemux_b200.file_proc.MinibatchDemuxer).  Stage times from CUDA
    events with device-resident rows; `e2e` = the public call on PINNED HOST rows (upload + stages + download)."""
    import time

    import torch

    from warpdemux_b200.detect import cnn, combined
    from warpdemux_b200.file_proc import MinibatchDemuxer
    from warpdemux_b200.models.dtw_svm import DTW_SVM

    ds = chain_dataset()
    stride, k = 11500, 5                               # 11 500 = the CLI's sig_preload_size for rna004 (parser.py:515)
    sig, lens = ds["sig"], ds["lens"]
    base = sig.shape[0]
    reps = max(1, 8000 // base)
    n = base * reps
    h_sig = torch.from_numpy(np.tile(sig, (reps, 1))).pin_memory()
    h_len = np.tile(lens, reps)
    model = cnn.load_cnn_model(os.path.join(ROOT, "tests", "golden", "models", "cnn_rna004_130bps_v0.2.4.npz"), device=local)
    mdl = DTW_SVM(params_small, device=local, mode="guarded")
    dmx = MinibatchDemuxer(mdl, model, core=cnn.CoreConfig(), cnn_boundaries=cnn.CNNBoundariesConfig(polya_cand_k=k), device=local,
                           llr=combined.LLRConfig())          # the reference's defaults: hail-mary + LLR fallback on (device)
    best = 1e30
    for it in range(4):
        t0 = time.perf_counter()
        r = dmx.run(h_sig, h_len, return_df=False)
        dt = time.perf_counter() - t0
        if it:
            best = min(best, dt)
    out = {"workload": f"{n} reads x {stride} samples float32 (NaN-padded minibatch rows), rna004 configs, WDX4 model, "
                       "CNN guarded, LLR fallback on the device, DTW guarded",
           "data": ds["kind"],
           "e2e": {"reads_per_s": n / best, "ms": best * 1e3, "h2d_bytes": int(h_sig.numel()) * 4,
                   "api": "MinibatchDemuxer.run(pinned host rows, full_lengths)"},
           "validated_fraction": float(r.detect_success.mean()), "fingerprint_ok_fraction": float((r.fp_status == 0).mean())}
    # production shape: a stream of 1000-read minibatches (parser.py:170-176) from pinned host memory, upload of
    # minibatch i+1 overlapping the kernels of minibatch i (MinibatchDemuxer.stream)
    mb = 1000
    mbs = [(h_sig[a:a + mb], h_len[a:a + mb]) for a in range(0, n - mb + 1, mb)] * 4
    for it in range(2):
        t0 = time.perf_counter()
        got = sum(int(r.labels.size) for r in dmx.stream(mbs, return_df=False))
        dt = time.perf_counter() - t0
    out["e2e_pipelined_minibatches"] = {"reads_per_s": got / dt, "minibatch": mb, "minibatches": len(mbs), "ms_per_minibatch": dt / len(mbs) * 1e3,
                                        "api": "MinibatchDemuxer.stream(iter of (pinned rows, full_lengths)), results consumed in order"}
    # the same stream of minibatches as raw int16 ADC samples + calibration (AdcBatch: half the bytes over PCIe, pA rows
    # made on the device by wdx_calibrate_rows)
    from warpdemux_b200.file_proc import AdcBatch

    h_adc = torch.from_numpy(np.tile(ds["adc"], (reps, 1))).pin_memory()
    num = np.tile(ds["num"], reps)
    offv, scv = np.tile(ds["offset"], reps), np.tile(ds["scale"], reps)
    mbs_adc = [(AdcBatch(h_adc[a:a + mb], num[a:a + mb], offv[a:a + mb], scv[a:a + mb]), h_len[a:a + mb]) for a in range(0, n - mb + 1, mb)] * 4
    for it in range(2):
        t0 = time.perf_counter()
        got = sum(int(r.labels.size) for r in dmx.stream(mbs_adc, return_df=False))
        dt = time.perf_counter() - t0
    out["e2e_pipelined_minibatches_adc"] = {"reads_per_s": got / dt, "minibatch": mb, "ms_per_minibatch": dt / len(mbs_adc) * 1e3,
                                            "h2d_bytes_per_read": stride * 2,
                                            "api": "MinibatchDemuxer.stream(iter of (AdcBatch(pinned int16 rows, calibration), full_lengths))"}
    # stage times, rows resident on the device
    side = torch.cuda.Stream()
    sp = side.cuda_stream
    d_sig = h_sig.cuda()
    d_len = torch.from_numpy(h_len).cuda()
    d_preds = torch.zeros((n, 1 + k), dtype=torch.int64, device="cuda")
    d_suc = torch.zeros(n, dtype=torch.uint8, device="cuda")
    d_info = torch.zeros((n, 4), dtype=torch.int32, device="cuda")
    d_bounds = torch.zeros((n, 3), dtype=torch.int64, device="cuda")
    d_lab = torch.zeros(n, dtype=torch.int64, device="cuda")
    d_st = torch.zeros(n, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    res = None
    with torch.cuda.stream(side):
        for it in range(4):
            ev[0].record()
            cnn.detect_raw(model, dmx.core, k, d_sig, n, stride, d_preds, stream=sp)
            ev[1].record()
            dmx.validator.run_raw(d_sig, n, stride, d_len, d_preds, 1 + k, d_suc, d_info, d_bounds, None, stream=sp)
            ev[2].record()
            a0, a1 = d_bounds[:, 0].contiguous(), d_bounds[:, 1].contiguous()
            dmx.fingerprinter.predict_raw(mdl._device_model(), d_sig, n, stride, a0, a1, 2, d_lab, d_st, detect_ok=d_suc, stream=sp)
            ev[3].record()
            side.synchronize()
            t = [ev[i].elapsed_time(ev[i + 1]) for i in range(3)]
            if it and (res is None or sum(t) < sum(res)):
                res = t
    alg = int(h_len.astype(np.int64).clip(max=stride).sum()) * 4
    # the validation stage alone, without the LLR branch behind it
    v0 = combined.Validator(combined.ValidateConfig(), device=local, verdict_only=True, llr=None)
    best0 = None
    with torch.cuda.stream(side):
        for it in range(3):
            ev[0].record()
            v0.run_raw(d_sig, n, stride, d_len, d_preds, 1 + k, d_suc, d_info, d_bounds, None, stream=sp)
            ev[1].record()
            side.synchronize()
            t0 = ev[0].elapsed_time(ev[1])
            best0 = t0 if best0 is None or (it and t0 < best0) else best0
        dmx.validator.run_raw(d_sig, n, stride, d_len, d_preds, 1 + k, d_suc, d_info, d_bounds, None, stream=sp)   # results of the chain again
        side.synchronize()
    v0.close()
    src = d_info[:, 3].cpu().numpy()
    out["llr_fallback"] = {"validate_without_llr_ms": best0, "llr_and_revalidation_ms": res[1] - best0,
                           "reads_hail_mary_ran": int(((src & 4) != 0).sum()), "reads_llr_ran": int(((src & 8) != 0).sum()),
                           "reads_rescued": int(((src & 3) != 0).sum())}
    out["device_resident"] = {"reads_per_s": n / (sum(res) * 1e-3), "cnn_ms": res[0], "validate_ms": res[1], "fingerprint_predict_ms": res[2],
                              "validate_reads_per_s": n / (res[1] * 1e-3),
                              "validate_roofline": {"bound": "hbm", "achieved": alg / (res[1] * 1e-3) / 1e9, "unit": "GB/s",
                                                    "note": "algorithmic bytes = 4 x valid samples per row, read once"}}
    # the tensor-core kernel of the CNN against the measured dense bf16 / fp16 MMA peak: issued MMA flops (M padded to 128-row
    # tiles, three fp16 products per float32 product) and the useful float32-equivalent flops
    try:
        t_in, _t_out = cnn.score_len(model, dmx.core, k, stride)
        t1 = (t_in - 1) // 3 + 1
        tiles, qtiles = (t1 + 127) // 128, (t1 + 128) // 128
        issued = 2 * tiles * 128 * 64 * 64 * 7 * 2 * 3 + qtiles * 128 * 64 * 16 * 3 * 3 * 2
        useful = 2 * t1 * 64 * 64 * 7 * 2 + t1 * 64 * 2 * 7 * 2
        cnn.enable_timing(model, dmx.core, k, True)
        bestc = None
        with torch.cuda.stream(side):
            for it in range(3):
                cnn.detect_raw(model, dmx.core, k, d_sig, n, stride, d_preds, stream=sp)
                side.synchronize()
                msc, nl = cnn.last_kernel_ms(model, dmx.core, k)
                bestc = msc if bestc is None or (it and msc < bestc) else bestc
        cnn.enable_timing(model, dmx.core, k, False)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:  # noqa: BLE001
            pass
        peak_tf = float(peaks.get("bf16_tflops", 1680.0))
        out["device_resident"]["cnn_tensor_roofline"] = {
            "bound": "tensor", "kernel": "cnn_tc_kernel (tcgen05.mma kind::f16 128x64x16, fp16 hi + lo split, TMEM accumulators)",
            "achieved": issued * n / (bestc * 1e-3) / 1e12, "peak": peak_tf, "unit": "TFLOP/s", "frac": issued * n / (bestc * 1e-3) / 1e12 / peak_tf,
            "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst)" if peaks else "fallback 1680 TFLOP/s",
            "useful_f32_equivalent_tflops": useful * n / (bestc * 1e-3) / 1e12, "conv_kernels_ms": bestc, "conv_kernel_launches": nl,
            "hidden_positions": t1, "issued_mma_flops_per_read": issued,
            "note": "MMA phases are shared-memory-bound (N = 64: 6 KB of operands per 128x64x16 MMA) and alternate with CUDA-core phases "
                    "(conv1, epilogues with the fp16 split) of the same read; DESIGN.md 4.6"}
    except Exception as e:  # noqa: BLE001
        out["device_resident"]["cnn_tensor_roofline"] = {"error": repr(e)}
    # the whole step through the public call on device-resident rows (stages chained, results downloaded, LLR tail
    # overlapped by the fingerprint pass of the validated reads)
    bestw = 1e30
    for it in range(5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dmx.run(d_sig, h_len, return_df=False)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if it:
            bestw = min(bestw, dt)
    out["device_resident"]["whole_step"] = {"ms": bestw * 1e3, "reads_per_s": n / bestw,
                                            "api": "MinibatchDemuxer.run(device tensor rows, full_lengths): wall clock incl. the result download"}
    # CPU beside it (bounded sample, one core): the numpy restatement of validate_boundaries on the same rows and the
    # boundaries the GPU CNN produced for them - the only stage of this chain whose CPU port is timed here (the
    # fingerprint and DTW/SVC stages have their own cpu_baseline entries above)
    try:
        from oracle import wdx_oracle_llr as ol
        from oracle import wdx_oracle_validate as ov

        m_cpu = 96
        pr = d_preds[:m_cpu].cpu().numpy()
        t0 = time.perf_counter()
        o = ov.validate_batch(sig[:m_cpu], h_len[:m_cpu], pr, ov.ValidateConfig())
        dt = time.perf_counter() - t0
        t0 = time.perf_counter()
        full_res = [ol.detect_one(sig[i], int(h_len[i]), pr[i], ol.LLRConfig(), ov.ValidateConfig())[0] for i in range(m_cpu)]
        dt_llr = time.perf_counter() - t0
        gpu_ok = d_suc[:m_cpu].cpu().numpy()
        gpu_b = d_bounds[:m_cpu].cpu().numpy()
        out["validate_cpu_baseline"] = {"value": m_cpu / dt, "unit": "reads/s", "cores": 1, "kind": "port",
                                        "sample": f"{m_cpu} of the same reads, oracle/wdx_oracle_validate.py (numpy), one process",
                                        "with_llr_fallback_reads_per_s": m_cpu / dt_llr,
                                        "gpu_verdict_mismatches_on_sample": int(sum(bool(r["success"]) != bool(g) for r, g in zip(full_res, gpu_ok))),
                                        "gpu_boundary_mismatches_on_sample": int(sum(
                                            bool(r["success"]) and (r["adapter_start"], r["adapter_end"], r["polya_end"]) != tuple(int(v) for v in b)
                                            for r, b in zip(full_res, gpu_b)))}
    except Exception as e:  # noqa: BLE001
        out["validate_cpu_baseline"] = {"error": repr(e)}
    dmx.close()
    model.close()
    return out


def raw_chain_stream_rank(local, minibatches=48, mb=1000, stride=11500, lanes=4):
    """One rank's part of the multi-GPU raw-signal measurement: a stream of production minibatches (1000 reads x 11 500
    int16 ADC samples + calibration, pinned host memory) through MinibatchDemuxer.stream on this rank's GPU.
    Returns (reads, seconds) — the caller takes the max of the seconds over ranks."""
    import torch

    from warpdemux_b200 import model_io as _mio
    from warpdemux_b200.detect import cnn, combined
    from warpdemux_b200.file_proc import AdcBatch, MinibatchDemuxer
    from warpdemux_b200.models.dtw_svm import DTW_SVM

    small = _mio.load_npz(os.path.join(ROOT, "tests", "golden", "models", "WDX4_rna004_v1_0.npz"))
    ds = chain_dataset()
    nb = ds["adc"].shape[0] // mb                      # distinct minibatches in the data set (4 for the real file)
    h_adc = torch.from_numpy(ds["adc"][: nb * mb]).pin_memory()
    md = cnn.load_cnn_model(os.path.join(ROOT, "tests", "golden", "models", "cnn_rna004_130bps_v0.2.4.npz"), device=local)
    mp4 = DTW_SVM(small, device=local, mode="guarded")
    dmx = MinibatchDemuxer(mp4, md, core=cnn.CoreConfig(), cnn_boundaries=cnn.CNNBoundariesConfig(polya_cand_k=5), device=local,
                           llr=combined.LLRConfig(), lanes=lanes, overlap_llr_tail=os.environ.get("WDX_OVERLAP_TAIL", "1") != "0")
    mbs = []
    for i in range(minibatches):
        a = (i % nb) * mb
        mbs.append((AdcBatch(h_adc[a:a + mb], ds["num"][a:a + mb], ds["offset"][a:a + mb], ds["scale"][a:a + mb]), ds["lens"][a:a + mb]))
    sum(int(r.labels.size) for r in dmx.stream(mbs[:8], return_df=False))
    torch.cuda.synchronize()
    return dmx, md, mbs


def config2_wdx4(params4, local, stream, n):
    """BASELINE.json configs[1]: WDX4 on n synthetic fingerprints, 1 B200, EXACT_F64 vs FAST_F32 (and GUARDED);
    label identity of GUARDED vs EXACT over the whole set."""
    import torch
    from warpdemux_b200 import _lib
    from warpdemux_b200.device_model import DeviceModel

    X = torch.from_numpy(synth_host(params4, n, seed=4242)).cuda()
    dm = DeviceModel(params4, local)
    dm.enable_timing(True)
    labs, out = {}, {"model": "WDX4_rna004_v1_0", "reads": n}
    cells = params4.n_sv * params4.band_cells()
    for mode in ("exact", "fast", "guarded"):
        lab = torch.empty(n, dtype=torch.int64, device="cuda")
        dm.predict_raw(X, min(n, 1 << 20), _lib.WDX_F64, _lib.MODES[mode], lab, None, None, None, None, stream=stream)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dm.predict_raw(X, n, _lib.WDX_F64, _lib.MODES[mode], lab, None, None, None, None, stream=stream)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        labs[mode] = lab
        out[mode] = {"reads_per_s": n / (ms * 1e-3), "gcups": n * cells / (ms * 1e-3) / 1e9, "ms": ms}
    out["label_mismatches_fast_vs_exact"] = int((labs["fast"] != labs["exact"]).sum().item())
    out["label_mismatches_guarded_vs_exact"] = int((labs["guarded"] != labs["exact"]).sum().item())
    dm.close()
    return out


def streaming_latency(mdl, params, batches=(1, 8, 64, 512), iters=300):
    """BASELINE.json configs[4]: per-batch latency of DTW_SVM.predict on host
    arrays (H2D + kernels + D2H), model resident, batches of a 512-channel
    flow cell's 100 ms chunk (SURVEY.md 8d S5)."""
    X = synth_host(params, max(batches) * 4, seed=99)
    out = {}
    for b in batches:
        for _ in range(20):
            mdl.predict(X[:b], nproc=1)
        ts = []
        for i in range(iters):
            xb = X[(i % 4) * b:(i % 4) * b + b]
            t0 = time.perf_counter()
            mdl.predict(xb, nproc=1)
            ts.append(time.perf_counter() - t0)
        ts = np.array(ts) * 1e3
        out[str(b)] = {"p50_ms": float(np.percentile(ts, 50)), "p99_ms": float(np.percentile(ts, 99)),
                       "reads_per_s_at_p50": b / (np.percentile(ts, 50) * 1e-3)}
    return out


def streaming_cadence(mdl, params, local, seconds=60.0, period=0.1, batches=(1, 8, 64, 512), raw_batch=512):
    """BASELINE.json configs[4] as SURVEY.md 8(d) S5 defines it: every 100 ms (the cadence of
    minknow_config/RNA2_seq_WDX_live_100ms.toml) a batch of b fingerprints of a 512-channel flow cell arrives, for
    `seconds`; the GPU idles in between (clocks ramp down, L2 goes cold), unlike the back-to-back loop of
    `streaming_latency`.  Each tick issues one DTW_SVM.predict per batch size on host arrays (H2D + kernels + D2H timed by
    the host clock) and one MinibatchDemuxer.run on a raw-signal chunk batch of `raw_batch` reads x 11 500 samples
    (CNN -> validation / LLR -> fingerprint -> DTW + SVC from pinned host rows)."""
    import torch

    from warpdemux_b200 import model_io as _mio
    from warpdemux_b200.detect import cnn, combined
    from warpdemux_b200.file_proc import MinibatchDemuxer
    from warpdemux_b200.models.dtw_svm import DTW_SVM

    X = synth_host(params, max(batches) * 8, seed=99)
    ds = chain_dataset()
    sig, lens = ds["sig"][:raw_batch], ds["lens"][:raw_batch]
    h_sig = torch.from_numpy(np.ascontiguousarray(sig)).pin_memory()
    small = _mio.load_npz(os.path.join(ROOT, "tests", "golden", "models", "WDX4_rna004_v1_0.npz"))
    md = cnn.load_cnn_model(os.path.join(ROOT, "tests", "golden", "models", "cnn_rna004_130bps_v0.2.4.npz"), device=local)
    mp4 = DTW_SVM(small, device=local, mode="guarded")
    dmx = MinibatchDemuxer(mp4, md, core=cnn.CoreConfig(), cnn_boundaries=cnn.CNNBoundariesConfig(polya_cand_k=5), device=local,
                           llr=combined.LLRConfig())
    for _ in range(3):
        for b in batches:
            mdl.predict(X[:b], nproc=1)
        dmx.run(h_sig, lens, return_df=False)
    ts = {str(b): [] for b in batches}
    ts_raw = []
    n_ticks = int(round(seconds / period))
    t_start = time.perf_counter()
    late = 0
    for tick in range(n_ticks):
        due = t_start + tick * period
        now = time.perf_counter()
        if now < due:
            time.sleep(due - now)
        elif now - due > period:
            late += 1
        for b in batches:
            o = ((tick * 7) % 8) * b
            t0 = time.perf_counter()
            mdl.predict(X[o:o + b], nproc=1)
            ts[str(b)].append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        dmx.run(h_sig, lens, return_df=False)
        ts_raw.append(time.perf_counter() - t0)
    out = {"cadence_ms": period * 1e3, "seconds": seconds, "ticks": n_ticks, "late_ticks": late, "model": MODEL, "mode": mdl.mode,
           "api": "DTW_SVM.predict(host array) once per batch size per tick; the GPU idles between ticks"}
    for b in batches:
        a = np.array(ts[str(b)]) * 1e3
        out[str(b)] = {"p50_ms": float(np.percentile(a, 50)), "p99_ms": float(np.percentile(a, 99)), "max_ms": float(a.max()), "samples": int(a.size)}
    a = np.array(ts_raw) * 1e3
    out["raw_chunk_batch"] = {"reads": raw_batch, "samples_per_read": 11500, "p50_ms": float(np.percentile(a, 50)), "p99_ms": float(np.percentile(a, 99)),
                              "max_ms": float(a.max()), "samples": int(a.size), "model": "WDX4_rna004_v1_0", "data": ds["kind"],
                              "api": "MinibatchDemuxer.run(pinned float32 rows, full_lengths), CNN guarded, LLR fallback on, DTW guarded"}
    dmx.close()
    md.close()
    return out


def label_identity_at_scale(dm, params, X_dev, n, lab_g, conf_g, flags_g, stream):
    """SURVEY.md 8(c) acceptance on the headline configuration: the GUARDED results of the timed run against EXACT_F64 over
    the whole step (every mismatch listed), and the FAST_F32 confidence error that the guard band has to cover."""
    import torch
    from warpdemux_b200 import _lib

    k = params.k
    lab_e = torch.empty(n, dtype=torch.int64, device="cuda")
    conf_e = torch.empty(n, dtype=torch.float64, device="cuda")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    dm.predict_raw(X_dev, n, _lib.WDX_F64, _lib.MODE_EXACT_F64, lab_e, conf_e, None, None, None, stream=stream)
    e1.record()
    torch.cuda.synchronize()
    ms_exact = e0.elapsed_time(e1)
    lab_f = torch.empty(n, dtype=torch.int64, device="cuda")
    conf_f = torch.empty(n, dtype=torch.float64, device="cuda")
    dm.predict_raw(X_dev, n, _lib.WDX_F64, _lib.MODE_FAST_F32, lab_f, conf_f, None, None, None, stream=stream)
    torch.cuda.synchronize()
    thr = torch.from_numpy(np.asarray(params.thresholds, dtype=np.float64)).cuda()
    lm = {int(v): i for i, v in enumerate(params.label_map)}

    def listing(mask, lab_x, conf_x):
        idx = torch.nonzero(mask).flatten()[:50].cpu().numpy()
        return [{"read": int(i), "label": int(lab_x[i]), "label_exact": int(lab_e[i]), "conf": float(conf_x[i]), "conf_exact": float(conf_e[i])}
                for i in idx]

    d = (conf_f - conf_e).abs()
    d = d[torch.isfinite(d)]
    edges = [0.0, 1e-9, 1e-8, 1e-7, 1e-6, 1e-5, 5e-5, 1e-4, 1e-3, 1.0]
    hist = torch.histogram(d.cpu(), bins=torch.tensor(edges, dtype=torch.float64)).hist.to(torch.int64).tolist()
    mism_g = lab_g != lab_e
    mism_f = lab_f != lab_e
    guard = 5e-5
    out = {
        "reads": int(n), "model": params.name if hasattr(params, "name") else MODEL,
        "exact_reads_per_s": n / (ms_exact * 1e-3),
        "label_mismatches_guarded_vs_exact": int(mism_g.sum().item()), "mismatch_rate_guarded": float(mism_g.sum().item()) / n,
        "guarded_mismatch_list": listing(mism_g, lab_g, conf_g),
        "label_mismatches_fast_vs_exact": int(mism_f.sum().item()), "fast_mismatch_list": listing(mism_f, lab_f, conf_f),
        "max_abs_conf_fast_minus_exact": float(d.max().item()) if d.numel() else 0.0,
        "abs_conf_error_histogram": {f"<={hi:g}": int(c) for hi, c in zip(edges[1:], hist)},
        "guard_band": guard, "guard_over_max_error": guard / max(float(d.max().item()), 1e-300) if d.numel() else None,
        "reads_recomputed_in_exact": int(((flags_g & 2) != 0).sum().item()),
        "guard_overflow_flags": int(((flags_g & 4) != 0).sum().item()),
        "nonfinite_flags": int(((flags_g & 1) != 0).sum().item()),
        "max_abs_conf_guarded_minus_exact_on_recomputed": float((conf_g - conf_e)[(flags_g & 2) != 0].abs().max().item())
        if bool(((flags_g & 2) != 0).any()) else 0.0,     # same arithmetic, other SV-range split: differs in summation order only
    }
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    params = load_params()
    threads = os.cpu_count() or 1
    total_budget = 120.0
    per_step = max(2.0, min(20.0, total_budget / max(1, args.steps + args.warmup)))
    kind, how = "port", ("minibatches of <=1000 over %d single-threaded workers (oracle/wdx_oracle.c: restated dtaidistance DTW + "
                         "libsvm predict_proba)" % threads)
    if reference_python_available() and not args.port_only:
        try:
            rps, n, dt = reference_python_arm(params, threads, per_step, steps=args.steps, warmup=min(args.warmup, 1))
            kind = "reference"
            how = ("the reference package's own DTW_SVM.predict(X, nproc=1, return_df=True) (baseline/_ref, unmodified) in "
                   "minibatches of <=1000 over a ProcessPoolExecutor(%d); dtaidistance = shim on the restated C (oracle/wdx_oracle.c)" % threads)
        except Exception as e:  # noqa: BLE001
            sys.stderr.write(f"reference python arm failed ({e!r}); timing the oracle port instead\n")
            rps, n, dt = cpu_arm(params, threads, per_step, steps=args.steps, warmup=min(args.warmup, 1))
    else:
        rps, n, dt = cpu_arm(params, threads, per_step, steps=args.steps, warmup=min(args.warmup, 1))
    cells = params.n_sv * params.band_cells()
    line = {
        "impl": "reference", "metric": METRIC, "value": rps, "unit": "reads/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{MODEL} on synthetic S1 fingerprints; bounded sample of {n} reads per step",
                   "model": MODEL, "n_sv": params.n_sv, "classes": params.k, "L": params.L, "window": params.window},
        "gcups": rps * cells / 1e9,
        "cpu_baseline": {"value": rps, "unit": "reads/s", "cores": threads, "kind": kind,
                         "sample": f"{n} S1 reads/step, {how}"},
        "e2e": {"value": rps, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def run_ours(args):
    # Rank 0 prints exactly ONE line on stdout: anything a library writes there (e.g. the NCCL
    # version banner) is sent to stderr instead by pointing fd 1 at fd 2 until the JSON line.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)

    import torch
    import torch.distributed as dist

    from warpdemux_b200 import _lib
    from warpdemux_b200.device_model import DeviceModel
    from warpdemux_b200.models.dtw_svm import DTW_SVM
    from warpdemux_b200.sharding import shard_bounds

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    params = load_params()
    n_total = args.reads_per_gpu * world
    lo, hi = shard_bounds(n_total, world)[rank]  # contiguous index range of this rank
    n = hi - lo
    mode = args.mode
    k = params.k
    cells_per_read = params.n_sv * params.band_cells()

    # this rank's shard of the synthetic set (seeded per shard so any N gives a reproducible set)
    X_host_t = torch.empty((n, params.L), dtype=torch.float64).pin_memory()
    X_host = X_host_t.numpy()
    X_host[:] = synth_host(params, n, seed=1000 + rank)
    X_dev = X_host_t.cuda(non_blocking=False)
    lab_d = torch.empty(n, dtype=torch.int64, device="cuda")
    conf_d = torch.empty(n, dtype=torch.float64, device="cuda")
    prob_d = torch.empty((n, k), dtype=torch.float64, device="cuda")
    flags_d = torch.zeros(n, dtype=torch.uint8, device="cuda")

    dm = DeviceModel(params, local)
    dm.enable_timing(True)
    stream = torch.cuda.current_stream().cuda_stream
    MODE = _lib.MODES[mode]

    def step_device():
        dm.predict_raw(X_dev, n, _lib.WDX_F64, MODE, lab_d, conf_d, prob_d, flags_d, None, stream=stream)

    # ---- value: inputs resident in HBM, CUDA events on the launch stream ----
    for _ in range(args.warmup):
        step_device()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = _lib.kernel_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms, kernel_launches = 0.0, 0
    barrier()
    e0.record()
    for _ in range(args.steps):
        step_device()
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = sum_over_ranks(_lib.kernel_launch_count() - launches0)
    # fused DTW+SVC launches of the LAST step, CUDA events on the launch stream; in GUARDED mode the
    # dominant kernel is the FAST_F32 pass (the EXACT re-run of boundary reads is reported separately)
    kms, kl = dm.last_kernel_ms_mode(mode == "exact")
    kms_all, kl_all = dm.last_kernel_ms()
    ms_per_step = ms_total / args.steps
    value = n_total / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:       # before anything below reuses the result buffers
        dump_outputs(args.dump_outputs, n, {"labels": lab_d, "confidence": conf_d, "probabilities": prob_d, "flags": flags_d})

    # labels gathered host-side in shard order (the only cross-rank exchange of the path)
    labels_host = lab_d.cpu().numpy()
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, labels_host[:1000])
        label_sample = np.concatenate(gathered)
    else:
        label_sample = labels_host[:1000]

    # ---- e2e: host buffers through the reference-facing API ------------------
    mdl = DTW_SVM(params, device=local, mode=mode)
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    mdl.predict(X_host[: min(n, 1 << 18)], nproc=1)  # warm-up: creates the device replica, staging buffers
    mdl.predict(X_host, nproc=1)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        y_pred, y_prob = mdl.predict(X_host, nproc=1, return_df=False)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    barrier()
    e2e_value = n_total / e2e_s
    e2e_match = bool(np.array_equal(y_pred, labels_host))
    # guard bookkeeping of the timed device run (flags were written inside the timed region)
    n_overflow = int(sum_over_ranks(float(((flags_d & 4) != 0).sum().item())))
    n_recomputed = int(sum_over_ranks(float(((flags_d & 2) != 0).sum().item())))

    # ---- e2e from PAGEABLE host memory: what the reference's call sites pass (np.vstack(fpts), file_proc.py:443-450) ----
    X_page = np.array(X_host, copy=True)          # ordinary numpy allocation, not pinned
    mdl.predict(X_page[: min(n, 1 << 18)], nproc=1)
    barrier()
    t0 = time.perf_counter()
    yp2, _ = mdl.predict(X_page, nproc=1, return_df=False)
    torch.cuda.synchronize()
    e2e_page_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    e2e_pageable = {"value": n_total / e2e_page_s, "unit": "reads/s", "labels_equal_device_run": bool(np.array_equal(yp2, labels_host)),
                    "api": "DTW_SVM.predict(X, nproc=1) with X an ordinary (pageable) numpy array, as the reference's workers pass it"}
    del X_page

    # ---- N > 1: the whole sharded call incl. the host-side label gather north_star names (sharding.predict_sharded) ----
    sharded = None
    if world > 1:
        from warpdemux_b200.sharding import predict_sharded

        def fn(x):
            yp, pr = mdl.predict(x, nproc=1, return_df=False)
            return yp, pr.max(axis=1)              # label + top probability per read: what a caller keeps per read

        predict_sharded(fn, X_host[: 1 << 16], x_is_local_shard=True, dst=0)
        barrier()
        t0 = time.perf_counter()
        got = predict_sharded(fn, X_host, x_is_local_shard=True, dst=0)
        torch.cuda.synchronize()
        sh_s = max_over_ranks(time.perf_counter() - t0)
        barrier()
        sharded = {"value": n_total / sh_s, "unit": "reads/s", "seconds": sh_s,
                   "api": "sharding.predict_sharded(lambda x: DTW_SVM.predict(x), this rank's contiguous shard, dst=0): every rank "
                          "classifies its shard from pinned host memory, rank 0 receives all labels + top probabilities in read order",
                   "gathered_bytes": int(n_total * 16)}
        if rank == 0:
            sharded["gathered_reads"] = int(got[0].shape[0])
            sharded["rank0_shard_equals_device_run"] = bool(np.array_equal(got[0][:n], labels_host))

    # ---- raw-signal chain at N GPUs: where host memory / PCIe could break the linear scaling of the fingerprint path ----
    chain = None
    if args.chain_stream:
        try:
            dmx_c, md_c, mbs_c = raw_chain_stream_rank(local)
            for _ in dmx_c.stream(mbs_c[:12], return_df=False):      # untimed: lane replicas, buffers, pinned blocks
                pass
            mbs_c = mbs_c * 4
            barrier()
            t0 = time.perf_counter()
            got_c = sum(int(r.labels.size) for r in dmx_c.stream(mbs_c, return_df=False))
            torch.cuda.synchronize()
            dt_c = max_over_ranks(time.perf_counter() - t0)
            barrier()
            tot_c = sum_over_ranks(float(got_c))
            chain = {"value": tot_c / dt_c, "unit": "reads/s", "n_gpus": world, "reads": int(tot_c), "seconds": dt_c,
                     "h2d_bytes_per_read": 11500 * 2, "host_to_device_gb_per_s": tot_c * 11500 * 2 / dt_c / 1e9,
                     "data": chain_dataset()["kind"],
                     "api": "MinibatchDemuxer.stream(AdcBatch minibatches of 1000 reads x 11 500 int16 samples from pinned host memory) on every "
                            "rank concurrently: calibration -> CNN -> validation / LLR -> fingerprint -> DTW + SVC (WDX4, guarded); "
                            "wall clock, max over ranks"}
            dmx_c.close()
            md_c.close()
        except Exception as e:  # noqa: BLE001
            chain = {"error": repr(e)}

    # ---- other arithmetic modes on a smaller batch (context for `value`) ------
    modes = {}
    if rank == 0 and args.extra_modes:
        n_small = min(n, 1 << 20)
        for mname in ("fast", "exact", "guarded"):
            if mname == mode:
                continue
            M2 = _lib.MODES[mname]
            for _ in range(2):
                dm.predict_raw(X_dev, n_small, _lib.WDX_F64, M2, lab_d, conf_d, prob_d, None, None, stream=stream)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            dm.predict_raw(X_dev, n_small, _lib.WDX_F64, M2, lab_d, conf_d, prob_d, None, None, stream=stream)
            b.record()
            torch.cuda.synchronize()
            modes[mname] = {"reads_per_s": n_small / (a.elapsed_time(b) * 1e-3), "batch": n_small}
    extras = {}
    if rank == 0 and world == 1 and args.extras:
        try:
            extras["label_identity_at_scale"] = label_identity_at_scale(dm, params, X_dev, n, lab_d, conf_d, flags_d, stream)
        except Exception as e:  # noqa: BLE001
            extras["label_identity_at_scale"] = {"error": repr(e)}
        try:
            extras["streaming_latency_ms"] = streaming_latency(mdl, params)
        except Exception as e:  # noqa: BLE001
            extras["streaming_latency_ms"] = {"error": repr(e)}
        if args.cadence_seconds > 0:
            try:
                extras["streaming_100ms_cadence"] = streaming_cadence(mdl, params, local, seconds=args.cadence_seconds)
            except Exception as e:  # noqa: BLE001
                extras["streaming_100ms_cadence"] = {"error": repr(e)}
        if args.single_call_reads > 0:
            try:   # BASELINE.json configs[2]'s whole 100 M-read set given to ONE GPU in ONE wdx_predict call (20 GB of input)
                del X_dev, prob_d
                X_dev = prob_d = None
                torch.cuda.empty_cache()
                nb = args.single_call_reads
                gen = torch.Generator(device="cuda").manual_seed(2024)
                sv_d = torch.from_numpy(params.sv).cuda()
                Xb = torch.empty((nb, params.L), dtype=torch.float64, device="cuda")
                for r0 in range(0, nb, 1 << 22):
                    r1 = min(nb, r0 + (1 << 22))
                    ix = torch.randint(0, params.n_sv, (r1 - r0,), device="cuda", generator=gen)
                    Xb[r0:r1] = sv_d[ix] + SIGMA * torch.randn((r1 - r0, params.L), dtype=torch.float64, device="cuda", generator=gen)
                labb = torch.empty(nb, dtype=torch.int64, device="cuda")
                flb = torch.zeros(nb, dtype=torch.uint8, device="cuda")
                dm.predict_raw(Xb, 1 << 20, _lib.WDX_F64, MODE, labb, None, None, flb, None, stream=stream)
                torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                dm.predict_raw(Xb, nb, _lib.WDX_F64, MODE, labb, None, None, flb, None, stream=stream)
                b.record()
                torch.cuda.synchronize()
                ms = a.elapsed_time(b)
                extras["single_gpu_100M_call"] = {"reads": nb, "seconds": ms * 1e-3, "reads_per_s": nb / (ms * 1e-3), "mode": mode,
                                                  "input_gb": nb * params.L * 8 / 1e9, "guard_overflow_flags": int(((flb & 4) != 0).sum().item()),
                                                  "data": "S1 generated on the device (torch Philox, seed 2024); one wdx_predict call, device buffers",
                                                  "label_histogram_first_1M": {str(int(u)): int(c) for u, c in zip(*np.unique(labb[: 1 << 20].cpu().numpy(), return_counts=True))}}
                del Xb, labb, flb
                torch.cuda.empty_cache()
            except Exception as e:  # noqa: BLE001
                extras["single_gpu_100M_call"] = {"error": repr(e)}
        try:
            from warpdemux_b200 import model_io as _mio
            small = _mio.load_npz(os.path.join(ROOT, "tests", "golden", "models", "WDX4_rna004_v1_0.npz"))
            X_dev = prob_d = None  # make room
            torch.cuda.empty_cache()
            extras["wdx4_10M_exact_vs_fast"] = config2_wdx4(small, local, stream, args.config2_reads)
        except Exception as e:  # noqa: BLE001
            extras["wdx4_10M_exact_vs_fast"] = {"error": repr(e)}
        try:
            extras["fingerprint_stage"] = fingerprint_stage(small, local, stream)
        except Exception as e:  # noqa: BLE001
            extras["fingerprint_stage"] = {"error": repr(e)}
        try:
            extras["trna_consensus_stage"] = trna_stage(small, local, stream)
        except Exception as e:  # noqa: BLE001
            extras["trna_consensus_stage"] = {"error": repr(e)}
        try:
            extras["raw_signal_chain"] = raw_signal_chain(small, local)
        except Exception as e:  # noqa: BLE001
            extras["raw_signal_chain"] = {"error": repr(e)}
    barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (fused DTW+SVC, FP32 CUDA-core issue) ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    sm_max = float(peaks.get("sm_max_mhz", 1965.0))
    n_sm = torch.cuda.get_device_properties(local).multi_processor_count
    exact = mode == "exact"
    slots, lanes = (6, 64) if exact else (5, 128)
    # fused launches of one step process n reads (GUARDED adds the small exact re-run; count the first launch's cells)
    cells_per_launch_set = n * cells_per_read
    kernel_s = kms * 1e-3
    achieved = cells_per_launch_set * slots / kernel_s / 1e12           # T lane-ops/s
    peak = n_sm * lanes * sm_max * 1e6 / 1e12
    sm_now = (clocks or {}).get("sm_mhz") or sm_max
    roofline = {
        "bound": "fp64_alu" if exact else "fp32_alu",
        "kernel": "dtw_svc_kernel<%s,25,15,KM1=%d,%s>" % ("EXACT" if exact else "FAST", 10, "f64" if exact else "packed f32x2 E-form"),
        "achieved": achieved, "peak": peak, "unit": "T lane-op/s", "frac": achieved / peak,
        "frac_at_measured_clock": achieved / (n_sm * lanes * sm_now * 1e6 / 1e12),
        "definition": f"DTW cells/s x {slots} issue slots per cell / ({n_sm} SM x {lanes} lanes x f_SM); "
                      f"peak uses clocks.max.sm={sm_max:.0f} MHz (MEASURED_PEAKS.json), SURVEY.md 8(d)",
        "gcups": cells_per_launch_set / kernel_s / 1e9,
        # stricter readings of the same measurement (DESIGN.md 4.1, profiles/r01_ubench_instruction_mix.txt)
        "frac_of_fma_pipe_cycles": None if exact else (cells_per_launch_set / kernel_s) / (n_sm * 4 * 32 * sm_max * 1e6 / 3.0),
        "frac_of_measured_instruction_mix_ceiling": (cells_per_launch_set / kernel_s) /
                                                    (n_sm * 4 * 32 * sm_max * 1e6 / (18.6 if exact else 4.58)),
        "ceilings_note": "FAST cell = FADD2+FFMA2+FADD2 per 2 cells (3 FMA-pipe cycles per cell) + FMNMX3 (2 ALU cycles); a "
                         "dependency-free loop of exactly this mix sustains 4.58 cycles per cell per SM sub-partition on B200 "
                         "(8.13 T cells/s), the EXACT cell 18.6 cycles (2.0 T cells/s) - scripts/ubench_pipes.cu",
        "kernel_ms_per_step": kms, "kernel_launches_per_step": kl,
        "kernel_share_of_step": kms / ms_per_step,
        "all_fused_launches_ms_per_step": kms_all, "all_fused_launches_per_step": kl_all,
        "traffic": None,
    }
    # HBM side of the same kernel (it is compute-bound; this shows no re-reads are wasted).  Algorithmic bytes per read:
    # the float64 fingerprint in, the k(k-1)/2 one-vs-one decision sums out (fused kernel) and back in (finishing
    # kernel), the per-read results out (label, confidence, k probabilities, flag) - DESIGN.md 4.1.
    n_pairs = k * (k - 1) // 2
    alg_per_read = params.L * 8 + n_pairs * 8      # the fused kernel itself: fingerprint in, decision sums out
    reads_per_launch = min(n, 1 << 22)          # wdx_model_set_chunk_reads default: 2^22 reads per fused launch
    roofline["hbm_algorithmic_bytes_per_read"] = alg_per_read
    roofline["path_hbm_algorithmic_bytes_per_read"] = params.L * 8 + 2 * n_pairs * 8 + (8 + 8 + 8 * k + 1)   # + finishing kernel
    roofline["reads_per_launch"] = reads_per_launch
    roofline["hbm_algorithmic_bytes_per_launch"] = alg_per_read * reads_per_launch
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "latest_traffic.json")))
        if prof.get("reads_in_profiled_launch") == reads_per_launch and prof.get("mode") == mode and prof.get("model") == MODEL:
            roofline["traffic"] = prof.get("dram_bytes_per_launch")            # same variant, same launch size: comparable as printed
        roofline["traffic_bytes_per_read"] = prof.get("dram_bytes_per_read")
        roofline["traffic_profile"] = {k2: prof.get(k2) for k2 in ("kernel", "reads_in_profiled_launch", "mode", "model", "source", "note")}
    except Exception:  # noqa: BLE001
        pass

    # ---- CPU baseline on this box's host cores (bounded sample) ------------------
    cpu = None
    cpu_ref_py = None
    if world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        rps, ns, dt, Xc, (cpu_pred, cpu_prob, cpu_conf) = cpu_arm(params, threads, 15.0, want_outputs=True)
        # the same reads through the GPU path: the parity statement that goes with the speed-up
        gpu_pred, gpu_prob = mdl.predict(Xc, nproc=1)
        cpu = {"value": rps, "unit": "reads/s", "cores": threads, "kind": "port",
               "sample": f"{ns} S1 reads of the same workload, minibatches of <=1000 over {threads} single-threaded "
                         f"workers, {dt:.1f} s (oracle/wdx_oracle.c)",
               "gpu_label_mismatches_on_sample": int((gpu_pred != cpu_pred).sum()),
               "gpu_max_abs_prob_diff_on_sample": float(np.abs(gpu_prob - cpu_prob).max())}
        if reference_python_available():
            # SURVEY.md 8(d): the reference's own Python on the shim, one worker and all cores, bounded samples
            try:
                r1, n1, d1 = reference_python_arm(params, 1, 4.0)
                ra, na, da, Xr, ref_pred = reference_python_arm(params, threads, 6.0, want_outputs=True)
                g_pred, _ = mdl.predict(Xr, nproc=1)
                cpu_ref_py = {"unit": "reads/s", "kind": "reference",
                              "n1": {"value": r1, "cores": 1, "sample": f"{n1} S1 reads, {d1:.1f} s"},
                              "all_cores": {"value": ra, "cores": threads, "sample": f"{na} S1 reads in minibatches of {na // threads} over a "
                                                                                        f"ProcessPoolExecutor({threads}), {da:.1f} s"},
                              "gpu_label_mismatches_on_sample": int((g_pred != ref_pred).sum()),
                              "what": "the unmodified reference package (baseline/_ref, pip --target install of /root/reference): "
                                      "DTW_SVM.predict(X, nproc=1, return_df=True) -> parallel_distances.distance_matrix_to -> "
                                      "dtaidistance SHIM on the restated C (oracle/wdx_oracle.c) -> pdist_kernel -> sklearn "
                                      "SVC.predict_proba -> process_probs -> predictions_to_df"}
            except Exception as e:  # noqa: BLE001
                cpu_ref_py = {"error": repr(e)}
        else:
            cpu_ref_py = {"unavailable": "baseline/_ref not present (install: __graft_entry__.build() where /root/reference exists)"}

    line = {
        "metric": METRIC, "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64" if exact else "f32", "data": "synthetic",
        "config": {"workload": f"{MODEL}: {args.reads_per_gpu} synthetic S1 fingerprints per GPU per step "
                               f"({n_total} total), mode {mode}",
                   "model": MODEL, "n_sv": params.n_sv, "classes": k, "L": params.L, "window": params.window,
                   "reads_per_gpu": args.reads_per_gpu, "mode": mode, "parallelism": f"reads sharded x{world}",
                   "cache": f"input {n * params.L * 8 / 1e6:.0f} MB per step > 126 MB L2 (no flush needed)"},
        "gcups": value * cells_per_read / 1e9,
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "reads/s", "h2d_bytes_per_step": int(n_total * params.L * 8),
                "d2h_bytes_per_step": int(n_total * (8 + 8 + 8 * k + 1)), "steps": e2e_steps,
                "api": "DTW_SVM.predict(X_host, nproc=1) -> (y_pred, y_prob); pinned host input, "
                       "host perf_counter around the blocking calls, max over ranks",
                "labels_equal_device_run": e2e_match},
        "e2e_pageable": e2e_pageable,
        "e2e_sharded_with_label_gather": sharded,
        "raw_signal_chain_stream": chain,
        "guard": {"mode": mode, "band": 5e-5, "reads_recomputed_in_exact_per_step": n_recomputed, "guard_overflow_flags_per_step": n_overflow,
                  "note": "flags written inside the timed region; an overflow (more boundary reads than the re-run list of a launch "
                          "holds) would leave FAST_F32 labels on the flagged reads"},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "cpu_baseline_reference_python": cpu_ref_py,
        "modes": modes,
        "label_histogram": {str(int(a)): int(b) for a, b in zip(*np.unique(label_sample, return_counts=True))},
    }
    line.update(extras)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default=os.environ.get("WDX_BENCH_MODE", "guarded"), choices=["exact", "fast", "guarded"])
    ap.add_argument("--reads-per-gpu", type=int, default=READS_PER_GPU)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-modes", dest="extra_modes", action="store_false")
    ap.add_argument("--config2-reads", type=int, default=10_000_000)
    ap.add_argument("--cadence-seconds", type=float, default=60.0, help="length of the 100 ms-cadence streaming measurement (0 = skip)")
    ap.add_argument("--single-call-reads", type=int, default=100_000_000, help="reads of the one-call single-GPU run (0 = skip)")
    ap.add_argument("--no-chain-stream", dest="chain_stream", action="store_false",
                    help="skip the raw-signal chain stream measured on every rank (multi-GPU scaling of the ADC -> calls path)")
    ap.add_argument("--port-only", action="store_true", help="reference arm: time the C port even if baseline/_ref is present")
    ap.add_argument("--no-extras", dest="extras", action="store_false",
                    help="skip the secondary measurements (streaming latency, fingerprint stage)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step (a seeded sample of rank 0's reads) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours (the reference arm sizes its sample from a timing probe)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: W >= 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

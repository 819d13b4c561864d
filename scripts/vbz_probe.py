"""pod5 VBZ decoding on the device: kernel rate, host batching time and the minibatch step fed from a pod5 file.

    python scripts/vbz_probe.py [OUT.json]

1. wdx_vbz_decode_rows (zstd + streamvbyte-16) on N_READS seeded reads of the median length (21 836 samples), one
   pod5 chunk each (pod5 writes chunks of up to 102 400 samples), rows of 11 500 samples; the compressed input is
   larger than the 126 MB L2.  CUDA events over REPS launches.
2. Pod5File.vbz_minibatches: host time per 1000-read minibatch of a synthetic pod5 file holding those reads.
3. MinibatchDemuxer.stream over the bench's chain reads (bench.chain_dataset, replicated to 8 192 reads) as a pod5
   file (vbz_minibatches in the loop), as prebuilt VbzBatch minibatches and as pinned AdcBatch minibatches, alternated.
Prints one JSON object with the card name and power limit (also written to OUT.json when given).
"""
import json
import os
import subprocess
import sys
import tempfile
import time
import uuid

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

import bench  # noqa: E402
from vbz_testutil import make_vbz_batch, synth_signal, write_pod5  # noqa: E402
from warpdemux_b200 import vbz  # noqa: E402
from warpdemux_b200.file_proc import AdcBatch  # noqa: E402
from warpdemux_b200.io.pod5_min import Pod5File  # noqa: E402

N_READS = int(os.environ.get("N_READS", "8000"))
REPS = int(os.environ.get("REPS", "20"))
MEDIAN, STRIDE, CHUNK = 21836, 11500, 102400
out_path = sys.argv[1] if len(sys.argv) > 1 else None
res = {}
try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    res["gpu"] = q.stdout.strip().splitlines()[0]
except Exception as e:  # noqa: BLE001
    res["gpu"] = f"unknown ({e})"

# 1. kernel rate
rng = np.random.default_rng(123)
sigs = [synth_signal(rng, MEDIAN, 20) for _ in range(N_READS)]
batch = make_vbz_batch([[s] for s in sigs], np.zeros(N_READS), np.ones(N_READS), STRIDE, level=1)
dev = torch.device("cuda", 0)
d = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
soff = vbz.scratch_layout(batch.chunk_samples, batch.read_chunks, STRIDE)
d_src, d_off, d_s, d_rc, d_soff = (d(batch.data, np.uint8), d(batch.chunk_offsets, np.int64), d(batch.chunk_samples, np.int32),
                                   d(batch.read_chunks, np.int64), d(soff, np.int64))
d_scr = torch.empty(int(soff[-1]), dtype=torch.uint8, device=dev)
rows = torch.empty((N_READS, STRIDE), dtype=torch.int16, device=dev)
nv = torch.empty(N_READS, dtype=torch.int32, device=dev)
st = torch.empty(N_READS, dtype=torch.int32, device=dev)
s = torch.cuda.current_stream()
call = lambda: vbz.decode_rows_raw(d_src, d_off, d_s, d_rc, d_scr, d_soff, rows, nv, st, 0, s.cuda_stream)
for _ in range(3):
    call()
torch.cuda.synchronize()
assert not st.any().item() and int(nv.sum().item()) == N_READS * STRIDE
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(REPS):
    call()
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / REPS
res["decode"] = dict(reads=N_READS, read_samples=MEDIAN, stride=STRIDE, compressed_mb=round(batch.data.size / 1e6, 1),
                     ms_per_call=round(ms, 3), reads_per_s=round(N_READS / ms * 1e3), compressed_gb_per_s_in=round(batch.data.size / ms / 1e6, 2),
                     samples_per_s_out=round(N_READS * STRIDE / ms * 1e3))
print(json.dumps(res), flush=True)

with tempfile.TemporaryDirectory() as tmp:
    # 2. host batching
    path = os.path.join(tmp, "median.pod5")
    write_pod5(path, [(uuid.UUID(int=i).bytes, x, 0.0, 1.0) for i, x in enumerate(sigs)], chunk_size=CHUNK, shuffle=False, batch_rows=1000)
    f = Pod5File(path)
    list(f.vbz_minibatches(1000, STRIDE))
    t0 = time.perf_counter()
    nb = sum(1 for _ in f.vbz_minibatches(1000, STRIDE))
    res["host_batching_ms_per_1000_reads"] = round((time.perf_counter() - t0) / nb * 1e3, 3)
    del f, sigs, batch, d_src, d_scr, rows

    # 3. the minibatch step
    dmx, md, mbs = bench.raw_chain_stream_rank(0, minibatches=1, lanes=4)
    ds = bench.chain_dataset()
    rep = 8
    n0 = ds["adc"].shape[0]
    adc = np.concatenate([ds["adc"]] * rep)
    num, off, sc, lens = (np.concatenate([ds[k]] * rep) for k in ("num", "offset", "scale", "lens"))
    n = adc.shape[0]
    path = os.path.join(tmp, "chain.pod5")
    write_pod5(path, [(uuid.UUID(int=i).bytes, adc[i, :num[i]], float(off[i]), float(sc[i])) for i in range(n)], chunk_size=CHUNK,
               shuffle=False, batch_rows=1000)
    f = Pod5File(path)
    h_adc = torch.from_numpy(adc).pin_memory()
    adc_mbs = [(AdcBatch(h_adc[a:a + 1000], num[a:a + 1000], off[a:a + 1000], sc[a:a + 1000]), num[a:a + 1000]) for a in range(0, n, 1000)]
    vbz_mbs = [(b, fl) for b, fl, _ in f.vbz_minibatches(1000, STRIDE)]
    runs = {"adc": lambda: adc_mbs, "vbz_prebuilt": lambda: vbz_mbs, "pod5_file": lambda: f.vbz_minibatches(1000, STRIDE)}
    first = {}
    for k, gen in runs.items():     # warm-up, and the three inputs give the same calls
        first[k] = [r.labels for r in dmx.stream(gen(), return_df=False)]
    same = all(np.array_equal(np.concatenate(first["adc"]), np.concatenate(first[k])) for k in runs)
    times = {k: [] for k in runs}
    for _ in range(3):
        for k, gen in runs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            got = sum(int(r.labels.size) for r in dmx.stream(gen(), return_df=False))
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)
    res["stream"] = dict(reads=n, distinct_reads=n0, data=ds["kind"], labels_equal_adc=bool(same),
                         **{f"{k}_reads_per_s": [round(got / t) for t in v] for k, v in times.items()})
print(json.dumps(res), flush=True)
if out_path:
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        json.dump(res, fh, indent=1)

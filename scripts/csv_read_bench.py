#!/usr/bin/env python
"""Measurements of the CSV text parsed on the device (nsf_csv_row_offsets + nsf_csv_parse), one GPU.

    python scripts/csv_read_bench.py [--out profiles/csv_read_r06.json] [--reps 5]

Inputs: the 60 facial CSVs of bench.py's api_e2e tree (LiveLink-shaped, 1800 rows x 63 columns each) and the 60
audio_features.csv caches of C2's feature rows (60 clips x 30 s at 88.2 kHz, 1801 x 256 each, formatted by
Engine.format_csv, byte for byte pandas' to_csv).
(a) The kernels alone: the five kernels of nsf_csv_parse (row count, scan, row starts, fields, integer columns) on the
    text already in device memory, CUDA events around `reps` calls after two warm-up calls.  Reports ms per call,
    text GB/s and fields/s.
(b) Engine.parse_csv host to host (the upload, the row-offsets wait, the parse, the download), against pandas'
    read_csv of the same files on an 8-thread I/O pool; results asserted bit-identical.
(c) load_data_batched on the 60-take tree (in /dev/shm), uncached and again with the audio_features.csv caches
    present, each against the same call with the pandas readers; examples asserted identical.

The card's name and power limit are read in the same run and written beside the numbers.
"""
import argparse
import contextlib
import io
import json
import os
import shutil
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import csv_cache_bench as ccb  # noqa: E402

DROP = ["Timecode", "BlendshapeCount"]


def pack(files):
    off = np.zeros(len(files) + 1, dtype=np.int64)
    np.cumsum([len(f) for f in files], out=off[1:])
    return np.frombuffer(b"".join(files), dtype=np.uint8), off


def column_map(data, drop):
    names = data.split(b"\n", 1)[0].rstrip(b"\r").decode().split(",")
    kept = [n for n in names if n not in drop]
    return len(names), [-1 if n in drop else kept.index(n) for n in names]


def kernels_alone(eng, files, drop, reps):
    import ctypes as C

    import torch
    from neurosync_trainer_lite_b200 import _native as nv
    text, off = pack(files)
    cols, out_col = column_map(files[0], drop)
    oc = np.asarray(out_col, np.int32)
    out_cols = int(oc.max()) + 1
    s = torch.cuda.current_stream()
    d_text = torch.from_numpy(text).cuda()
    row_off = np.zeros(len(files) + 1, np.int64)
    nv.check(nv.lib.nsf_csv_row_offsets(eng.handle, C.c_void_p(s.cuda_stream), C.c_void_p(d_text.data_ptr()),
                                        off.ctypes.data_as(nv._i64p), len(files), row_off.ctypes.data_as(nv._i64p)))
    out = torch.empty((int(row_off[-1]), out_cols), dtype=torch.float32, device="cuda")
    status = torch.empty(len(files), dtype=torch.int32, device="cuda")

    def call():
        nv.check(nv.lib.nsf_csv_parse(eng.handle, C.c_void_p(s.cuda_stream), nv.F32, C.c_void_p(d_text.data_ptr()),
                                      off.ctypes.data_as(nv._i64p), len(files), cols, oc.ctypes.data_as(nv._i32p),
                                      out_cols, row_off.ctypes.data_as(nv._i64p), C.c_void_p(out.data_ptr()),
                                      out_cols, C.c_void_p(status.data_ptr())))
    call()
    call()
    torch.cuda.synchronize()
    assert int(status.abs().sum()) == 0
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        call()
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / reps
    fields = int(row_off[-1]) * cols
    return {"files": len(files), "text_bytes": int(off[-1]), "rows": int(row_off[-1]), "cols": cols, "reps": reps,
            "ms_per_call": round(ms, 4), "text_GB_per_s": off[-1] / (ms / 1e3) / 1e9, "fields_per_s": fields / (ms / 1e3)}


def host_to_host(eng, files, drop, reps):
    import pandas as pd
    text, off = pack(files)
    cols, out_col = column_map(files[0], drop)
    eng.parse_csv(text, off, cols, out_col, np.float32)
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        rows, r_off, status = eng.parse_csv(text, off, cols, out_col, np.float32)
        times.append(time.perf_counter() - t0)
    assert not status.any()
    read = lambda b: np.ascontiguousarray(pd.read_csv(io.BytesIO(b)).drop(columns=drop).values, dtype=np.float32)  # noqa: E731
    with ThreadPoolExecutor(max_workers=8) as pool:
        t0 = time.perf_counter()
        want = list(pool.map(read, files))
        t_pandas = time.perf_counter() - t0
    for k, w in enumerate(want):
        assert np.array_equal(rows[r_off[k]:r_off[k + 1]].view(np.uint32), w.view(np.uint32)), k
    return {"parse_csv_s": {"min": min(times), "mean": float(np.mean(times)), "runs": reps},
            "pandas_8_threads_s": t_pandas, "speedup_vs_pandas_min": t_pandas / min(times), "rows_identical": True}


def load_data_legs(reps):
    from neurosync_trainer_lite_b200 import synth
    from neurosync_trainer_lite_b200.dataset import data_processing as dp

    def pandas_parse(eng, pool, paths, text, off, drop, dtype):      # the readers before the device parser
        return list(pool.map(lambda p: dp._pandas_rows(p, drop, dtype), paths))

    base = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    work = tempfile.mkdtemp(prefix="nsf_csv_read_", dir=base)
    try:
        ccb.make_tree(os.path.join(work, "t"), synth)

        def run(cached, pandas):
            if not cached:
                for k in range(ccb.N_TAKES):
                    p = os.path.join(work, "t", f"take_{k:03d}", "audio_features.csv")
                    if os.path.exists(p):
                        os.unlink(p)
            original = dp._parse_csvs
            if pandas:
                dp._parse_csvs = pandas_parse
            try:
                with contextlib.redirect_stdout(io.StringIO()):
                    t0 = time.perf_counter()
                    ex, _ = dp.load_data_batched(os.path.join(work, "t"), 88200, set(), cache_format="csv")
                    dt = time.perf_counter() - t0
            finally:
                dp._parse_csvs = original
            assert len(ex) == ccb.N_TAKES
            return dt, dict(dp.last_timing), ex

        result = {"tree": f"{ccb.N_TAKES} takes x {ccb.SECONDS:.0f} s int16 WAV @ 88.2 kHz + facial CSV, in {base}"}
        for cached in (False, True):
            run(cached, False)                                       # warm-up (and, uncached, writes the caches)
            dev = [run(cached, False) for _ in range(reps)]
            ref = [run(cached, True) for _ in range(reps)]
            for (xa, fa), (xb, fb) in zip(dev[-1][2], ref[-1][2]):
                assert np.array_equal(xa, xb) and np.array_equal(fa, fb)
            best_d, best_r = min(dev, key=lambda r: r[0]), min(ref, key=lambda r: r[0])
            result["cached_csv" if cached else "uncached"] = {
                "device_total_s_runs": [round(r[0], 4) for r in dev],
                "pandas_total_s_runs": [round(r[0], 4) for r in ref],
                "device_phases_s_best": {k: round(v, 4) for k, v in best_d[1].items()},
                "pandas_phases_s_best": {k: round(v, 4) for k, v in best_r[1].items()},
                "examples_identical": True}
        return result
    finally:
        shutil.rmtree(work, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "csv_read_r06.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    from neurosync_trainer_lite_b200 import _native as nv
    from neurosync_trainer_lite_b200 import engine, synth
    if nv.lib.nsf_device_count() < 1:
        raise SystemExit("needs an sm_100 device")
    eng = engine.get_engine(88200, *engine.frame_params(88200))
    work = tempfile.mkdtemp(prefix="nsf_csv_files_")
    try:
        ccb.make_tree(work, synth)
        facial = []
        for k in range(ccb.N_TAKES):
            with open(os.path.join(work, f"take_{k:03d}", f"take{k:03d}_iPhone_cal.csv"), "rb") as fh:
                facial.append(fh.read())
    finally:
        shutil.rmtree(work, ignore_errors=True)
    rows, roff = ccb.c2_rows(eng, synth)
    text, t_off = eng.format_csv(rows, roff)
    caches = [text[t_off[k]:t_off[k + 1]].tobytes() for k in range(len(t_off) - 1)]
    result = {"device": ccb.card(),
              "workload": "60 facial CSVs of the api_e2e tree; 60 audio_features.csv caches of C2's rows (float64 text)"}
    result["a_kernels"] = {"facial": kernels_alone(eng, facial, DROP, args.reps),
                           "caches": kernels_alone(eng, caches, [], args.reps)}
    result["b_host_to_host"] = {"facial": host_to_host(eng, facial, DROP, args.reps),
                                "caches": host_to_host(eng, caches, [], args.reps)}
    result["c_load_data"] = load_data_legs(3)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()

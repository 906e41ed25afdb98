#!/usr/bin/env python
"""Measurements of the audio_features.csv cache formatted on the device (nsf_format_csv_host), one GPU.

    python scripts/csv_cache_bench.py [--out profiles/csv_cache_r05.json] [--reps 5]

(a) The two kernels alone (k_csv_lengths + k_csv_write) on C2's rows: the feature rows of 60 clips x 30 s at
    88.2 kHz (108 060 x 256 float32, extracted on the device from synthetic speech-like clips).  Kernel times come from
    torch.profiler's CUDA activity records over `reps` calls after a warm-up call, summed per call.  Reports values/s,
    text GB/s and (rows read by both kernels + text written) over the 7.7 TB/s HBM figure of NVIDIA's HGX B200 data
    sheet (a data-sheet figure, not a measured one).
(b) Engine.format_csv from host rows to host text (pageable buffers), against pandas' to_csv of the same rows in the
    same process (one file per clip), texts compared byte for byte.
(c) load_data_batched on bench.py's api_e2e tree (60 takes of 30 s int16 WAV + facial CSV, in /dev/shm) with
    cache_format="csv": the total and the write_cache phase, against the same call with the pandas writer the
    package used before ("before" leg) on a copy of the tree; every audio_features.csv is asserted byte-identical.

The card's name and power limit are read in the same run and written beside the numbers.
"""
import argparse
import contextlib
import io
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
HBM_BYTES_PER_S = 7.7e12
N_TAKES, SECONDS, FACIAL_ROWS, FACIAL_COLS = 60, 30.0, 1800, 61


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def pandas_text(rows):
    import pandas as pd
    return pd.DataFrame(np.asarray(rows, dtype=np.float64)).to_csv(index=False).encode()


def c2_rows(eng, synth):
    kinds = ("voiced", "voiced", "noise", "voiced", "gated", "voiced")
    clips = [synth.to_int16_pcm(0.8 * synth.synth_clip(SECONDS, 88200, seed=700 + k, kind=kinds[k % 6]))
             for k in range(N_TAKES)]
    from neurosync_trainer_lite_b200 import _native as nv
    from neurosync_trainer_lite_b200.engine import pack_clips
    pcm, off = pack_clips(clips)
    rows = eng.extract_host(pcm, off, nv.PEAK_NORMALIZE)
    assert rows.shape == (108060, 256)
    return rows, eng.row_offsets(off)


def kernels_alone(eng, rows, roff, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    text, _ = eng.format_csv(rows, roff)                      # warm-up: arenas, module load
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            eng.format_csv(rows, roff)
        torch.cuda.synchronize()
    per = {}
    for ev in prof.key_averages():
        if "k_csv_" in ev.key:
            key = "k_csv_lengths" if "k_csv_lengths" in ev.key else "k_csv_write"
            us = max(getattr(ev, a, 0.0) or 0.0 for a in ("device_time_total", "self_device_time_total"))
            per[key] = per.get(key, 0.0) + us / 1e3 / reps          # us -> ms per call
    ms = sum(per.values())
    values, text_bytes = rows.size, len(text)
    moved = 2 * rows.nbytes + text_bytes                        # rows read by both kernels, text written once
    return {"rows": list(rows.shape), "dtype": str(rows.dtype), "files": len(roff) - 1, "reps": reps,
            "kernel_ms_per_call": {k: round(v, 3) for k, v in per.items()}, "kernel_ms": round(ms, 3),
            "values_per_s": values / (ms / 1e3), "text_bytes": text_bytes,
            "text_GB_per_s": text_bytes / (ms / 1e3) / 1e9,
            "hbm_bytes": moved, "hbm_share_of_7.7TBps": moved / HBM_BYTES_PER_S / (ms / 1e3)}


def host_to_host(eng, rows, roff, reps):
    eng.format_csv(rows, roff)
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        text, t_off = eng.format_csv(rows, roff)
        times.append(time.perf_counter() - t0)
    t0 = time.perf_counter()
    want = [pandas_text(rows[roff[k]:roff[k + 1]]) for k in range(len(roff) - 1)]
    t_pandas = time.perf_counter() - t0
    same = all(text[t_off[k]:t_off[k + 1]].tobytes() == want[k] for k in range(len(want)))
    assert same, "device text differs from pandas"
    return {"format_csv_s": {"min": min(times), "mean": float(np.mean(times)), "runs": reps},
            "pandas_to_csv_s": t_pandas, "pandas_to_csv_s_per_file": t_pandas / len(want),
            "speedup_vs_pandas_min": t_pandas / min(times), "text_identical": same, "text_bytes": int(t_off[-1])}


def make_tree(root, synth):
    import pandas as pd
    kinds = ("voiced", "voiced", "noise", "voiced", "gated", "voiced")
    wavs = [synth.wav_bytes(synth.to_int16_pcm(0.8 * synth.synth_clip(SECONDS, 88200, seed=700 + s, kind=kinds[s])),
                            88200) for s in range(6)]
    cols = ["Timecode", "BlendshapeCount"] + [f"bs{i}" for i in range(FACIAL_COLS)]
    csvs = [pd.DataFrame(np.hstack([np.zeros((FACIAL_ROWS, 2)), synth.synth_facial(FACIAL_ROWS, seed=s)]),
                         columns=cols).to_csv(index=False) for s in range(6)]
    for k in range(N_TAKES):
        take = os.path.join(root, f"take_{k:03d}")
        os.makedirs(take)
        with open(os.path.join(take, "audio.wav"), "wb") as fh:
            fh.write(wavs[k % 6])
        with open(os.path.join(take, f"take{k:03d}_iPhone_cal.csv"), "w") as fh:
            fh.write(csvs[k % 6])


def load_data_legs(reps):
    import pandas as pd
    from neurosync_trainer_lite_b200 import synth
    from neurosync_trainer_lite_b200.dataset import data_processing as dp

    def pandas_writer(cache_csv, rows, cache_format, text=None):     # the writer before the device formatter
        pd.DataFrame(np.asarray(rows, dtype=np.float64)).to_csv(cache_csv, index=False)
        print(f"Audio features saved to {cache_csv}")

    base = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    work = tempfile.mkdtemp(prefix="nsf_csv_tree_", dir=base)
    try:
        make_tree(os.path.join(work, "after"), synth)
        shutil.copytree(os.path.join(work, "after"), os.path.join(work, "before"))

        def run(root):
            for k in range(N_TAKES):
                p = os.path.join(root, f"take_{k:03d}", "audio_features.csv")
                if os.path.exists(p):
                    os.unlink(p)
            with contextlib.redirect_stdout(io.StringIO()):
                t0 = time.perf_counter()
                ex, _ = dp.load_data_batched(root, 88200, set(), cache_format="csv")
                dt = time.perf_counter() - t0
            assert len(ex) == N_TAKES
            return dt, dict(dp.last_timing), ex

        run(os.path.join(work, "after"))                              # warm-up: arenas, page cache, module load
        after = [run(os.path.join(work, "after")) for _ in range(reps)]
        original = dp._write_feature_cache
        dp._write_feature_cache = pandas_writer
        try:
            before = run(os.path.join(work, "before"))
        finally:
            dp._write_feature_cache = original
        for k in range(N_TAKES):
            name = os.path.join(f"take_{k:03d}", "audio_features.csv")
            with open(os.path.join(work, "after", name), "rb") as a, open(os.path.join(work, "before", name), "rb") as b:
                assert a.read() == b.read(), name
        for (xa, fa), (xb, fb) in zip(after[-1][2], before[2]):
            assert np.array_equal(xa, xb) and np.array_equal(fa, fb)
        best = min(after, key=lambda r: r[0])
        return {"tree": f"{N_TAKES} takes x {SECONDS:.0f} s int16 WAV @ 88.2 kHz + facial CSV, in {base}",
                "after": {"total_s_runs": [round(r[0], 4) for r in after],
                          "write_cache_s_runs": [round(r[1]["write_cache"], 4) for r in after],
                          "phases_s_best": {k: round(v, 4) for k, v in best[1].items()}},
                "before_pandas_writer": {"total_s": round(before[0], 3),
                                         "phases_s": {k: round(v, 4) for k, v in before[1].items()}},
                "csv_files_byte_identical": True, "examples_identical": True}
    finally:
        shutil.rmtree(work, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "csv_cache_r05.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    from neurosync_trainer_lite_b200 import _native as nv
    from neurosync_trainer_lite_b200 import engine, synth
    if nv.lib.nsf_device_count() < 1:
        raise SystemExit("needs an sm_100 device")
    eng = engine.get_engine(88200, *engine.frame_params(88200))
    rows, roff = c2_rows(eng, synth)
    result = {"device": card(), "workload": "C2 rows: 60 clips x 30 s @ 88.2 kHz -> 108060 x 256 float32"}
    result["a_kernels"] = kernels_alone(eng, rows, roff, args.reps)
    result["b_host_to_host"] = host_to_host(eng, rows, roff, args.reps)
    result["c_load_data"] = load_data_legs(3)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()

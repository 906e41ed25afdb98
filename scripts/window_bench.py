#!/usr/bin/env python
"""Training-window batches from host memory against batches from GPU memory, one GPU, one command.

    python scripts/window_bench.py [--out result.json] [--batches 200]

Two datasets of seeded synthetic rows (256 audio + 61 facial float32 columns, window 128): C3 geometry (60 clips x
2670 rows) and one C4 rank's geometry (60 clips x 6239 rows).  For every batch size:

(a) host route: DataLoader(shuffle=True, collate_fn=AudioFacialDataset.collate_fn) + .to('cuda') of both tensors,
    host clock per batch ending in torch.cuda.synchronize(), over --batches batches after warm-up;
(b) DeviceWindowLoader(shuffle=True) timed the same way (the rows were uploaded once, before the clock);
(c) the gather alone: CUDA events around each of many window_gather calls (its descriptor upload of
    8 (3 (clips + 1) + B) bytes and the kernel), random indices per call and output buffers rotated over >= 256 MB so
    neither side is served from the 126 MB L2; and the kernel alone from torch.profiler in a separate pass.  Bytes
    moved = 2 x B x 128 x (256 + 61) x 4 (every window row read once and written once); the share is taken of
    7.7 TB/s, the HBM3e bandwidth of NVIDIA's HGX B200 data sheet for one GPU (a data-sheet figure, not a
    measured ceiling).

The same run checks that (a) and (b) yield identical batches under one seed, and writes the card's name and power
limit beside the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
HBM_PEAK = 7.7e12
WINDOW, A_COLS, F_COLS = 128, 256, 61
DATASETS = {"c3": (60, 2670), "c4_rank": (60, 6239)}
BATCHES = (32, 128, 512, 2048)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def make_dataset(clips, rows, seed):
    from neurosync_trainer_lite_b200.dataset.dataset import AudioFacialDataset
    ds = AudioFacialDataset.__new__(AudioFacialDataset)
    ds.micro_batch_size = WINDOW
    ds.zero_copy_windows = False
    ds.clips, ds._starts = [], [0]
    rng = np.random.default_rng(seed)
    for _ in range(clips):
        ds.add_clip(rng.standard_normal((rows, A_COLS), dtype=np.float32),
                    rng.standard_normal((rows, F_COLS), dtype=np.float32))
    return ds


def batch_bytes(b):
    return 2 * b * WINDOW * (A_COLS + F_COLS) * 4


def time_loader(loader, n, warmup, to_device):
    """Per-batch host-clock times (ms) of `n` batches after `warmup`, each ending in a synchronize; the loader is
    restarted when an epoch ends."""
    import torch
    it = iter(loader)

    def nxt():
        nonlocal it
        try:
            return next(it)
        except StopIteration:
            it = iter(loader)
            return next(it)

    for _ in range(warmup):
        b = nxt()
        if to_device:
            b = (b[0].to("cuda"), b[1].to("cuda"))
    torch.cuda.synchronize()
    ms = []
    for _ in range(n):
        t0 = time.perf_counter()
        b = nxt()
        if to_device:
            b = (b[0].to("cuda"), b[1].to("cuda"))
        torch.cuda.synchronize()
        ms.append((time.perf_counter() - t0) * 1e3)
        del b
    return ms


def stats(ms):
    a = np.asarray(ms)
    return {"batches": len(a), "mean_ms": round(float(a.mean()), 4), "median_ms": round(float(np.median(a)), 4),
            "p10_ms": round(float(np.percentile(a, 10)), 4), "p90_ms": round(float(np.percentile(a, 90)), 4)}


def same_batches(ds, windows, b, n_check=4, seed=1234):
    import torch
    from torch.utils.data import DataLoader

    from neurosync_trainer_lite_b200.dataset.dataset import AudioFacialDataset, DeviceWindowLoader
    torch.manual_seed(seed)
    host = DataLoader(ds, batch_size=b, shuffle=True, collate_fn=AudioFacialDataset.collate_fn)
    hb = [x for _, x in zip(range(n_check), host)]
    torch.manual_seed(seed)
    dev = DeviceWindowLoader(ds, b, True, windows=windows)
    db = [x for _, x in zip(range(n_check), dev)]
    ok = len(hb) == len(db) and len(host) == len(dev)
    for (ha, hf), (da, df) in zip(hb, db):
        ok = ok and torch.equal(da, ha.to("cuda")) and torch.equal(df, hf.to("cuda"))
    return bool(ok)


def kernel_events(windows, b, launches, rng):
    """CUDA events around each window_gather call (descriptor upload + kernel); random indices, rotating outputs."""
    import torch
    n_out = max(2, -(-(256 << 20) // (batch_bytes(b) // 2)))
    outs = [(torch.empty((b, WINDOW, A_COLS), device="cuda"), torch.empty((b, WINDOW, F_COLS), device="cuda"))
            for _ in range(n_out)]
    idx = [rng.integers(0, len(windows), size=b) for _ in range(64)]
    for k in range(8):
        windows.gather(idx[k % len(idx)], *outs[k % n_out])
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(launches)]
    torch.cuda.synchronize()
    for k in range(launches):
        ev[k][0].record()
        windows.gather(idx[k % len(idx)], *outs[k % n_out])
        ev[k][1].record()
    torch.cuda.synchronize()
    ms = np.array([s.elapsed_time(e) for s, e in ev])
    med = float(np.median(ms))
    return {"launches": launches, "mean_ms": round(float(ms.mean()), 5), "median_ms": round(med, 5),
            "bytes": batch_bytes(b), "gb_per_s_median": round(batch_bytes(b) / (med * 1e-3) / 1e9, 1),
            "share_of_7p7_tb_s_data_sheet": round(batch_bytes(b) / (med * 1e-3) / HBM_PEAK, 3)}


def kernel_profiler(windows, b, launches, rng):
    """Mean CUDA time of k_window_gather itself (torch.profiler, a pass of its own)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    n_out = max(2, -(-(256 << 20) // (batch_bytes(b) // 2)))
    outs = [(torch.empty((b, WINDOW, A_COLS), device="cuda"), torch.empty((b, WINDOW, F_COLS), device="cuda"))
            for _ in range(n_out)]
    idx = [rng.integers(0, len(windows), size=b) for _ in range(64)]
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(launches):
            windows.gather(idx[k % len(idx)], *outs[k % n_out])
        torch.cuda.synchronize()
    rows = [e for e in prof.key_averages() if "k_window_gather" in e.key]
    count = sum(e.count for e in rows)
    if not count:
        return {"error": "no k_window_gather events recorded"}
    us = sum(e.device_time * e.count for e in rows) / count
    return {"kernels": count, "mean_us": round(us, 2),
            "gb_per_s": round(batch_bytes(b) / (us * 1e-6) / 1e9, 1),
            "share_of_7p7_tb_s_data_sheet": round(batch_bytes(b) / (us * 1e-6) / HBM_PEAK, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="write the JSON result here")
    ap.add_argument("--batches", type=int, default=200, help="timed batches per loader and batch size")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--launches", type=int, default=400, help="gather calls per batch size in (c)")
    ap.add_argument("--datasets", default=",".join(DATASETS))
    ap.add_argument("--batch-sizes", default=",".join(map(str, BATCHES)))
    args = ap.parse_args()

    import torch
    from torch.utils.data import DataLoader

    from neurosync_trainer_lite_b200 import _native as nv
    from neurosync_trainer_lite_b200.dataset.dataset import AudioFacialDataset, DeviceWindowLoader, DeviceWindows
    if nv.lib.nsf_device_count() < 1:
        raise SystemExit("window_bench.py needs an sm_100 GPU")
    torch.cuda.set_device(0)
    result = {"card": card(), "window": WINDOW, "audio_cols": A_COLS, "facial_cols": F_COLS,
              "hbm_data_sheet_tb_s": HBM_PEAK / 1e12, "datasets": {}}
    rng = np.random.default_rng(7)
    for name in args.datasets.split(","):
        clips, rows = DATASETS[name]
        ds = make_dataset(clips, rows, seed=sorted(DATASETS).index(name))
        t0 = time.perf_counter()
        windows = DeviceWindows(ds, device=0)
        upload_s = time.perf_counter() - t0
        entry = {"clips": clips, "rows_per_clip": rows, "windows": len(ds),
                 "device_bytes": windows.audio.numel() * 4 + windows.facial.numel() * 4,
                 "upload_s": round(upload_s, 3), "batch_sizes": {}}
        for b in map(int, args.batch_sizes.split(",")):
            r = {"bytes_per_batch_read_plus_write": batch_bytes(b), "identical_batches": same_batches(ds, windows, b)}
            torch.manual_seed(0)
            host = DataLoader(ds, batch_size=b, shuffle=True, collate_fn=AudioFacialDataset.collate_fn)
            r["a_host_dataloader"] = stats(time_loader(host, args.batches, args.warmup, True))
            torch.manual_seed(0)
            dev = DeviceWindowLoader(ds, b, True, windows=windows)
            r["b_device_loader"] = stats(time_loader(dev, args.batches, args.warmup, False))
            r["speedup_median"] = round(r["a_host_dataloader"]["median_ms"] / r["b_device_loader"]["median_ms"], 1)
            r["c_gather_events"] = kernel_events(windows, b, args.launches, rng)
            r["c_kernel_profiler"] = kernel_profiler(windows, b, min(args.launches, 200), rng)
            entry["batch_sizes"][str(b)] = r
            print(json.dumps({"dataset": name, "batch": b, **r}), flush=True)
        result["datasets"][name] = entry
        del windows, ds
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()

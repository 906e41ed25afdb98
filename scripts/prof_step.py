#!/usr/bin/env python
"""One device-resident step of a bench workload, for profilers (ncu) and A/B timing.

    python scripts/prof_step.py [--workload c2] [--warmup 2] [--steps 1]

Prints the mean step time (CUDA events) and the library's per-stage times as one JSON line.  Environment switches
of the library (NSF_AC_LOOP, NSF_AC_KERNEL, ...) apply as usual.  Experiments only."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c2")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--steps", type=int, default=1)
    ap.add_argument("--sr", type=int, default=0, help="override: sample rate of an ad-hoc workload (with --seconds, --clips)")
    ap.add_argument("--seconds", type=float, default=0.0)
    ap.add_argument("--clips", type=int, default=0)
    args = ap.parse_args()
    import torch
    import bench
    from neurosync_trainer_lite_b200 import engine
    if args.sr:
        f_len, h_len = engine.frame_params(args.sr)
        bench.WORKLOADS["adhoc"] = dict(sr=args.sr, F=f_len, H=h_len, clips=args.clips, seconds=args.seconds, collect=None,
                                        desc=f"ad hoc: {args.clips} clips x {args.seconds} s @ {args.sr} Hz (F = {f_len})")
        args.workload = "adhoc"
    w = bench.WORKLOADS[args.workload]
    eng = engine.get_engine(w["sr"], w["F"], w["H"], device=0)
    packed, off, _base, _mine, _n = bench.make_inputs(args.workload, 0, 1, "weak")
    dev = torch.device("cuda", 0)
    pcm = torch.from_numpy(packed).to(dev)
    rows = int(eng.row_offsets(off)[-1])
    out = torch.empty((rows, 256), dtype=torch.float32, device=dev)
    ws = torch.empty(eng.workspace_bytes(len(packed), len(off) - 1), dtype=torch.uint8, device=dev)
    for _ in range(args.warmup):
        eng.extract_device(pcm, off, 0, out=out, workspace=ws)
    torch.cuda.synchronize()
    eng.set_profiling(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        eng.extract_device(pcm, off, 0, out=out, workspace=ws)
    e1.record()
    torch.cuda.synchronize()
    frames = sum(eng.plan.hop_frames(int(n)) for n in __import__("numpy").diff(off))
    print(json.dumps({"workload": args.workload, "F": w["F"], "hop_frames": frames, "env": {k: v for k, v in os.environ.items() if k.startswith("NSF_")},
                      "ms_per_step": e0.elapsed_time(e1) / args.steps, "stages_ms": eng.stage_times_ms(),
                      "checksum": float(out[::997].abs().sum().item())}))


if __name__ == "__main__":
    main()

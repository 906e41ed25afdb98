#!/usr/bin/env python
"""Measurements of the WAV conversion stage (nsf_convert_*), one GPU, one process tree.

    python scripts/convert_bench.py [--parent PATH_TO_PARENT_SO] [--out result.json]

1. device-resident conversion: 30 minutes of audio as 64 clips, once 48 kHz stereo int16 and once 44.1 kHz mono
   int24, converted to 88.2 kHz with convert_device (HQ filter); CUDA events after warm-up.  Reports audio-seconds/s,
   float64 FMAs/s (outputs x taps per output, from the filter shapes) and the share of the card's FP64 peak
   (37 TFLOP/s = 18.5 T FMA/s dense FP64, NVIDIA's HGX B200 data sheet divided by its 8 GPUs; a data-sheet figure).
2. A/B of nsf_resample_host against another build of the library (--parent, e.g. the parent commit's csrc built
   with scripts/build_variant.sh): per-clip calls on the same inputs for every rate pair of tests/test_resample.py,
   the two builds alternated, outputs compared byte for byte.
3. load_data on a 60-take tree of 48 kHz stereo int16 takes (30 s each): the batched conversion route against the
   per-take decode_for_path composition it replaced, alternated, 3 runs each, outputs compared.

The card's name and power limit are read in the same run and written beside the numbers.
"""
import argparse
import hashlib
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
RATES = [(44100, 88200), (48000, 88200), (88200, 16000), (16000, 88200), (22050, 88200), (88200, 44100)]
FP64_PEAK_FMA = 18.5e12


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def taps_per_output(nv, orig, target):
    import ctypes as C
    up = C.c_int32()
    n = nv.lib.nsf_resample_design_q(orig, target, nv.RESAMPLE_HQ, None, 0, C.byref(up), None, None, None)
    return -(-n // up.value)


def make_payload(nv, enc, channels, rate, clips, seconds, seed=0):
    rng = np.random.default_rng(seed)
    frames = int(round(seconds * rate))
    bps = {nv.ENC_I16: 2, nv.ENC_I24: 3}[enc]
    n = frames * channels
    v = np.clip(np.rint(rng.standard_normal(n * clips) * 0.2 * (1 << (8 * bps - 1))), -(1 << (8 * bps - 1)),
                (1 << (8 * bps - 1)) - 1).astype(np.int32)
    raw = v.astype("<u4").view(np.uint8).reshape(-1, 4)[:, :bps].reshape(-1)
    clip_bytes = n * bps
    stride = (clip_bytes + 7) // 8 * 8
    payload = np.zeros(stride * clips, dtype=np.uint8)
    src = np.zeros(clips, dtype=nv.PCM_SOURCE)
    for k in range(clips):
        payload[k * stride:k * stride + clip_bytes] = raw[k * clip_bytes:(k + 1) * clip_bytes]
        src[k] = (k * stride, frames, enc, channels, rate, 0)
    return payload, src


def device_conversion(eng, nv):
    import torch
    dev = torch.device("cuda", eng.device)
    res = {}
    for name, enc, ch, rate in (("48k_stereo_i16", nv.ENC_I16, 2, 48000), ("44k1_mono_i24", nv.ENC_I24, 1, 44100)):
        payload, src = make_payload(nv, enc, ch, rate, 64, 1800.0 / 64)
        p = torch.from_numpy(payload).to(dev)
        out, off = eng.convert_device(p, src, 88200)
        for _ in range(3):
            eng.convert_device(p, src, 88200, out=out)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        e0.record()
        for _ in range(reps):
            eng.convert_device(p, src, 88200, out=out)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        n_out = int(off[-1])
        fmas = n_out * taps_per_output(nv, rate, 88200)
        res[name] = {"clips": 64, "audio_seconds": 1800.0, "outputs": n_out, "taps_per_output": taps_per_output(nv, rate, 88200),
                     "fp64_fmas": fmas, "ms": round(ms, 3), "audio_seconds_per_s": round(1800.0 / (ms / 1e3), 1),
                     "fp64_fma_per_s": fmas / (ms / 1e3), "share_of_fp64_peak": round(fmas / (ms / 1e3) / FP64_PEAK_FMA, 4),
                     "input_bytes": int(payload.nbytes), "output_bytes": n_out * 4}
        del p, out
    return res


# ---- 2: nsf_resample_host A/B (child processes select the library with NSF_LIB_PATH) --------------------------
def ab_child(outdir):
    # the entry points both builds export, bound directly (the package binds every newer symbol at import)
    import ctypes as C
    lib = C.CDLL(os.environ.get("NSF_LIB_PATH") or os.path.join(ROOT, "neurosync_trainer_lite_b200", "_lib", "libnsf.so"))
    lib.nsf_plan_create.argtypes = [C.c_int32] * 6 + [C.POINTER(C.c_void_p)]
    lib.nsf_ctx_create.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p)]
    lib.nsf_resample_len.restype = C.c_int64
    lib.nsf_resample_len.argtypes = [C.c_int64, C.c_int32, C.c_int32]
    lib.nsf_resample_host.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_void_p,
                                      C.c_int64]
    plan, ctx = C.c_void_p(), C.c_void_p()
    assert lib.nsf_plan_create(88200, 1470, 735, 23, 128, 187, C.byref(plan)) == 0
    assert lib.nsf_ctx_create(plan, 0, C.byref(ctx)) == 0       # default quality: HQ, what the loaders use

    def resample(x, orig, target):
        out = np.empty(lib.nsf_resample_len(len(x), orig, target), dtype=np.float32)
        assert lib.nsf_resample_host(ctx, x.ctypes.data, 0, len(x), orig, target, out.ctypes.data, len(out)) == 0
        return out
    rng = np.random.default_rng(5)
    res = {}
    for orig, target in RATES:
        clips = [(rng.standard_normal(int(orig * s)) * 0.2).astype(np.float32) for s in (30.0, 12.5, 3.3)]
        for c in clips:
            resample(c, orig, target)                          # warm-up (and the filter upload)
        times, digest = [], hashlib.sha256()
        for _ in range(5):
            t0 = time.perf_counter()
            outs = [resample(c, orig, target) for c in clips]
            times.append(time.perf_counter() - t0)
        for o in outs:
            digest.update(o.tobytes())
        res[f"{orig}->{target}"] = {"s_median": float(np.median(times)), "sha256": digest.hexdigest()}
    with open(os.path.join(outdir, "ab.json"), "w") as fh:
        json.dump(res, fh)


def ab(parent_so, rounds=3):
    runs = {"new": [], "parent": []}
    tmp = tempfile.mkdtemp(prefix="convert_ab_")
    try:
        for r in range(rounds):
            for name in (("new", "parent") if r % 2 == 0 else ("parent", "new")):
                env = dict(os.environ)
                env.pop("NSF_LIB_PATH", None)
                if name == "parent":
                    env["NSF_LIB_PATH"] = parent_so
                subprocess.run([sys.executable, os.path.abspath(__file__), "--ab-child", tmp], env=env, check=True)
                with open(os.path.join(tmp, "ab.json")) as fh:
                    runs[name].append(json.load(fh))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    out = {}
    for pair in runs["new"][0]:
        new = [r[pair]["s_median"] for r in runs["new"]]
        old = [r[pair]["s_median"] for r in runs["parent"]]
        same = len({r[pair]["sha256"] for r in runs["new"] + runs["parent"]}) == 1
        out[pair] = {"new_ms": [round(x * 1e3, 3) for x in new], "parent_ms": [round(x * 1e3, 3) for x in old],
                     "speedup_median": round(float(np.median(old) / np.median(new)), 3), "outputs_identical": same}
    return out


# ---- 3: load_data on a 48 kHz stereo tree ----------------------------------------------------------------------
def make_tree(root, takes=60, seconds=30.0):
    import pandas as pd
    from neurosync_trainer_lite_b200 import synth
    cols = ["Timecode", "BlendshapeCount"] + [f"bs{i}" for i in range(61)]
    rows = int(seconds * 60)
    for k in range(takes):
        d = os.path.join(root, f"take_{k:03d}")
        os.makedirs(d)
        y = np.stack([synth.synth_clip(seconds, 48000, seed=k * 2 + c, kind="voiced") for c in range(2)], axis=1)
        data = np.clip(np.rint(y * 0.7 * 32767), -32768, 32767).astype("<i2").tobytes()
        import struct
        fmt = struct.pack("<HHIIHH", 1, 2, 48000, 48000 * 4, 4, 16)
        body = b"WAVE" + b"fmt " + struct.pack("<I", 16) + fmt + b"data" + struct.pack("<I", len(data)) + data
        with open(os.path.join(d, "audio.wav"), "wb") as fh:
            fh.write(b"RIFF" + struct.pack("<I", len(body)) + body)
        pd.DataFrame(np.hstack([np.zeros((rows, 2)), synth.synth_facial(rows, seed=k)]), columns=cols).to_csv(
            os.path.join(d, f"t{k}_iPhone_cal.csv"), index=False)


def old_route(root, sr):
    """The per-take route: decode_for_path on a thread pool, packed as float32, then load_data_batched's
    float32 device pass (fused extraction + augmentation)."""
    from concurrent.futures import ThreadPoolExecutor

    from neurosync_trainer_lite_b200 import _native as nv
    from neurosync_trainer_lite_b200 import engine
    from neurosync_trainer_lite_b200.dataset import data_processing as dp
    from neurosync_trainer_lite_b200.utils.audio.load_audio import decode_for_path
    from neurosync_trainer_lite_b200.utils.video.mov_extraction import find_files
    f, h = engine.frame_params(88200)
    eng = engine.get_engine(88200, f, h)
    takes = [find_files(os.path.join(root, d)) for d in os.listdir(root)]
    with ThreadPoolExecutor(min(32, len(os.sched_getaffinity(0)) or 1)) as pool:
        t0 = time.perf_counter()
        pcm = list(pool.map(lambda t: decode_for_path(t[2], sr)[0], takes))
        pcm = [p if p.dtype == np.float32 else p.astype(np.float32) / np.float32(32768) for p in pcm]
        off = np.concatenate([[0], np.cumsum([len(p) for p in pcm])]).astype(np.int64)
        packed = np.concatenate(pcm)
        t_audio = time.perf_counter() - t0
        facial = list(pool.map(lambda t: dp._facial_rows(t[3], np.float32), takes))
    f_off = np.concatenate([[0], np.cumsum([len(x) for x in facial])]).astype(np.int64)
    oa, of, o_off = eng.extract_collect_host(packed, off, np.concatenate(facial), f_off, nv.PEAK_NORMALIZE)
    out = []
    for k in range(len(takes)):
        fk = of[o_off[k]:o_off[k + 1]].copy()
        fk[:, :61] *= 100
        out.append((oa[o_off[k]:o_off[k + 1]], fk))
    return out, t_audio


def loader(root, sr, rounds=3):
    import contextlib
    import io

    from neurosync_trainer_lite_b200.dataset import data_processing as dp
    os.environ["NSF_FEATURE_CACHE"] = "npy"        # fast cache writes: the CSV writer would dominate both legs

    def clear():
        for d in os.listdir(root):
            for name in ("audio_features.npy", "audio_features.csv"):
                p = os.path.join(root, d, name)
                if os.path.exists(p):
                    os.remove(p)
    res = {"new_total_s": [], "new_audio_s": [], "old_total_s": [], "old_audio_s": []}
    equal = True
    for r in range(rounds + 1):                   # round 0 warms both legs up (filters, arenas, engines)
        for leg in (("new", "old") if r % 2 == 0 else ("old", "new")):
            clear()
            with contextlib.redirect_stdout(io.StringIO()):
                t0 = time.perf_counter()
                if leg == "new":
                    got = dp.load_data(root, sr, set())
                    t_audio = dp.last_timing["read_audio"]
                else:
                    want, t_audio = old_route(root, sr)
                dt = time.perf_counter() - t0
            if r > 0:
                res[f"{leg}_total_s"].append(round(dt, 3))
                res[f"{leg}_audio_s"].append(round(t_audio, 3))
        equal = equal and len(got) == len(want) and all(
            np.array_equal(ga, wa) and np.array_equal(gf, wf) for (ga, gf), (wa, wf) in zip(got, want))
    clear()
    res["outputs_identical"] = bool(equal)
    res["note"] = ("new_total_s is load_data end to end (scan, facial CSVs, conversion, extraction + augmentation, "
                   ".npy cache writes); old_total_s is the per-take composition without cache writes; the *_audio_s "
                   "columns are the audio stage alone (new: read + device conversion, old: decode_for_path + packing)")
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", help="library build to A/B nsf_resample_host against")
    ap.add_argument("--out", help="write the JSON result here")
    ap.add_argument("--ab-child", help=argparse.SUPPRESS)
    ap.add_argument("--takes", type=int, default=60)
    args = ap.parse_args()
    if args.ab_child:
        return ab_child(args.ab_child)
    from neurosync_trainer_lite_b200 import _native as nv
    from neurosync_trainer_lite_b200 import engine
    if nv.lib.nsf_device_count() < 1:
        raise SystemExit("convert_bench.py needs an sm_100 GPU")
    f, h = engine.frame_params(88200)
    eng = engine.get_engine(88200, f, h, device=0)
    result = {"card": card(), "fp64_peak_fma_per_s_datasheet": FP64_PEAK_FMA}
    result["device_conversion"] = device_conversion(eng, nv)
    print(json.dumps(result["device_conversion"]), flush=True)
    if args.parent:
        result["resample_host_ab"] = ab(os.path.abspath(args.parent))
        print(json.dumps(result["resample_host_ab"]), flush=True)
    tmp = tempfile.mkdtemp(prefix="convert_tree_")
    try:
        make_tree(tmp, takes=args.takes)
        result["load_data_48k_stereo"] = {"takes": args.takes, "seconds_per_take": 30.0, "sr": 88200,
                                          **loader(tmp, 88200)}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    print(json.dumps(result["load_data_48k_stereo"]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)
    ok = all(v["outputs_identical"] for v in result.get("resample_host_ab", {}).values())
    ok = ok and result["load_data_48k_stereo"]["outputs_identical"]
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())

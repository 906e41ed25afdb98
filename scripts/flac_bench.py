#!/usr/bin/env python
"""Speed of FLAC decode on the device (nsf_flac_decode_host), one GPU.

    python scripts/flac_bench.py [--out profiles/flac_r05.json] [--reps 5]

Two workloads of 60 takes x 30 s, each encoded once by the test oracle's encoder and repeated 60 times in one host
payload (page-locked): stereo 16-bit 44.1 kHz (mid/side, LPC order 8) and mono 16-bit 88.2 kHz (LPC order 8), in
4096-sample frames.  For each, nsf_flac_decode_host is timed against nsf_convert_host of the same samples as WAV
data-chunk bytes (decode + downmix to mono float32 at the file's rate, the step a WAV take costs): a host clock
around the synchronous calls after one warm-up call, median of --reps.  The decoded bytes are checked against the
samples.  The card's name and power limit are read in the same run and written beside the numbers.
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


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                                    # noqa: BLE001 - reported, not fatal
        return {"error": repr(e)}


def take(n, channels, seed):
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    cols = [np.round(8000 * np.sin(t * (0.02 + 0.004 * c)) + 300 * rng.standard_normal(n)) for c in range(channels)]
    return np.clip(np.stack(cols, 1), -32768, 32767).astype(np.int64)


def timed(fn, reps):
    fn()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    return float(np.median(times)), [float(t) for t in times]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "flac_r05.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--takes", type=int, default=60)
    args = ap.parse_args()
    from neurosync_trainer_lite_b200 import _native as nv
    from neurosync_trainer_lite_b200 import engine
    from neurosync_trainer_lite_b200.utils.audio import load_audio as la
    from oracle import flac_oracle as fo
    import io

    eng = engine.get_engine(88200, *engine.frame_params(88200))
    result = {"card": card(), "takes": args.takes, "seconds_per_take": 30, "reps": args.reps, "workloads": {}}
    for name, rate, channels, stereo in [("stereo16_44k1", 44100, 2, "mid_side"), ("mono16_88k2", 88200, 1, None)]:
        x = take(30 * rate, channels, seed=rate)
        one = fo.encode(x, rate, 16, block=4096, stereo=stereo or "independent", sub=fo.Sub("lpc", 8))
        lay = la.flac_layout(io.BytesIO(one))
        n = args.takes
        payload = engine.PinnedBuffer(len(one) * n).view(np.uint8, (len(one) * n,))
        payload[:] = np.frombuffer(one * n, np.uint8)
        src = np.array([(k * len(one) + lay.data_offset, lay.data_bytes, lay.frames, channels, 16, rate, lay.max_block)
                        for k in range(n)], dtype=nv.FLAC_SOURCE)
        pcm_bytes = x.astype("<i2").tobytes()
        wav_payload = engine.PinnedBuffer(len(pcm_bytes) * n).view(np.uint8, (len(pcm_bytes) * n,))
        wav_payload[:] = np.frombuffer(pcm_bytes * n, np.uint8)
        wsrc = [(k * len(pcm_bytes), len(x), nv.ENC_I16, channels, rate) for k in range(n)]
        out = {}

        def flac():
            out["pcm"], out["off"] = eng.flac_decode_host(payload, src)

        def wav():
            eng.convert_host(wav_payload, wsrc, rate)

        s_flac, t_flac = timed(flac, args.reps)
        s_wav, t_wav = timed(wav, args.reps)
        ok = all(out["pcm"][out["off"][k]:out["off"][k + 1]].tobytes() == pcm_bytes for k in range(n))
        audio_s = 30.0 * n
        result["workloads"][name] = {
            "flac_bytes": len(one) * n, "pcm_bytes": len(pcm_bytes) * n, "frames_per_take": -(-len(x) // 4096),
            "flac_decode_host_s": s_flac, "flac_decode_host_runs_s": t_flac,
            "flac_audio_s_per_s": audio_s / s_flac, "flac_compressed_MB_per_s": len(one) * n / s_flac / 1e6,
            "convert_host_wav_s": s_wav, "convert_host_wav_runs_s": t_wav,
            "decoded_bytes_match": bool(ok)}
        print(name, json.dumps(result["workloads"][name]), flush=True)
        if not ok:
            raise SystemExit(f"{name}: decoded bytes differ from the samples")
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()

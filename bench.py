#!/usr/bin/env python
"""Benchmark of the audio feature front-end (BASELINE.json metric: audio-seconds per second).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference]
                    [--workload c2|c3|c4|c5] [--scaling weak|strong] [--no-cpu-baseline] [--no-extras]
                    [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch of synthetic input.  Workloads (BASELINE.json `configs`):

* ``c2`` (default, configs[1])  30-minute single-actor dataset, 60 clips x 30 s @ 88.2 kHz, features only;
* ``c3`` (configs[2])  the same dataset + ``collect_features(include_fast, blend_boundaries, blend_frames=30)``;
* ``c4`` (configs[3])  8 voices x 30 min (480 clips) with fast + slow augmentation on 8 GPUs, rows gathered into ONE
  page-locked host array; every rank carries 60 clips, so N < 8 runs "N ranks' share" of the configuration;
* ``c5`` (configs[4])  10 000 clips x 2 s @ 16 kHz, batched small clips.

Scaling.  The path shards by clip with no collective.  ``weak`` = every rank processes the workload's per-rank
batch (c2: 60 clips per GPU), ``strong`` = the workload's clips are split over the ranks
(``shard.lpt_partition``), as configs[2] and configs[4] state.  The headline line runs ``c2`` weak (fixed
work per GPU, like the driver's scaling run expects); ``workloads`` in the same JSON line carries short passes
of c3 (strong), c4 (60 clips per rank; the full 480-clip configuration at N = 8) and c5 (strong), each with its
own kernel table and CPU baseline.

One JSON line on rank 0:

* ``value``    device-resident throughput (PCM already in HBM), CUDA events on the launch stream, max over ranks;
* ``e2e``      the same metric through the C ABI with HOST buffers, H2D and D2H inside the timed region.  Headline
               ``e2e`` = int16 PCM (what the takes' WAV files hold) + on-device peak normalisation, i.e. the
               arithmetic of ``extract_audio_features``; ``e2e_f32_pcm`` = float32 PCM through
               ``extract_and_combine_features`` semantics (twice the upload); both next to ``copy_ceiling``, the
               bare page-locked H2D + D2H of the same bytes at the same N;
* ``api_e2e``  a synthetic 60-take tree (int16 WAV + facial CSV per folder, ``.npy`` feature cache) through the
               reference-named ``dataset.data_processing.load_data`` (file reads and CSV parsing included);
* ``roofline`` / ``kernels``  per-kernel achieved vs MEASURED_PEAKS.json (live CUDA-event stage times);
* ``cpu_baseline``  the CPU oracle ("port" of the reference path; librosa itself is not installable) on the box's
               host cores, bounded sample, wall clock, BLAS pinned to one thread per worker process;
* ``clocks``   nvidia-smi samples taken during the timed region.

``--impl reference`` times the CPU oracle alone (all host cores, bounded sample per step) on the headline
workload's input format (int16 PCM -> decode -> peak normalise -> features).

``--dump-outputs DIR`` writes, after the timed steps, what the last timed device-resident step of the headline workload
computed on rank 0: ``features.npy`` (float32 feature rows) and, for c3 / c4, ``collect_audio.npy`` /
``collect_facial.npy`` (float32 augmented rows).  An output of more than DUMP_ROWS rows is a fixed, seeded sample of its
rows, in order; ``<name>_rows.npy`` (float64) holds their indices.  The inputs are synthesised from fixed seeds, so two
builds run with the same arguments can be compared array for array.
"""
import os

# One BLAS/OpenMP thread per process, decided BEFORE NumPy is imported anywhere: the CPU baseline runs one worker
# process per core (spawned children inherit the environment), so library threads would only oversubscribe.
for _k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
    os.environ[_k] = "1"

import argparse  # noqa: E402
import json  # noqa: E402
import shutil  # noqa: E402
import subprocess  # noqa: E402
import sys  # noqa: E402
import tempfile  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_MELS, N_MFCC, N_LAGS = 128, 23, 187
FACIAL_ROWS, FACIAL_COLS = 1800, 61                    # 30 s of 60 fps blendshape rows per clip
WORKLOADS = {
    # name: sr, F, H, clips (per rank when weak / in total when strong), seconds per clip, collect kwargs, description
    "c2": dict(sr=88200, F=1470, H=735, clips=60, seconds=30.0, collect=None,
               desc="C2: 30-min single-actor dataset, 60 clips x 30 s @ 88.2 kHz, features only"),
    "c3": dict(sr=88200, F=1470, H=735, clips=60, seconds=30.0,
               collect=dict(include_fast=True, include_slow=False, blend_boundaries=True, blend_frames=30),
               desc="C3: 30-min dataset + collect_features(include_fast, blend_boundaries, blend_frames=30)"),
    "c4": dict(sr=88200, F=1470, H=735, clips=60, seconds=30.0,
               collect=dict(include_fast=True, include_slow=True, blend_boundaries=True, blend_frames=30),
               desc="C4: 8 voices x 30 min (480 clips over 8 GPUs, 60 per rank) + collect_features(fast, slow, blend 30), "
                    "rows gathered into one page-locked host array"),
    "c5": dict(sr=16000, F=266, H=133, clips=10000, seconds=2.0, collect=None,
               desc="C5: 10000 clips x 2 s @ 16 kHz, batched small clips"),
}
DEFAULT_SCALING = {"c2": "weak", "c3": "strong", "c4": "weak", "c5": "strong"}
# --dump-outputs: rows kept per output array; the largest dump (c4: 256 + 256 + 61 float32 columns) stays under 64 MB
DUMP_ROWS = 16384
DUMP_LIMIT_BYTES = 64 << 20


def dump_row_index(n_rows):
    """Rows of an n_rows output that --dump-outputs keeps: all of them, or a fixed seeded sample in ascending order."""
    if n_rows <= DUMP_ROWS:
        return np.arange(n_rows, dtype=np.int64)
    return np.sort(np.random.default_rng(0).choice(n_rows, DUMP_ROWS, replace=False))


def sample_rows(name, rows):
    """{name: the kept rows of a (rows, cols) CUDA tensor as float32, name_rows: their indices as float64}."""
    import torch
    idx = dump_row_index(rows.shape[0])
    kept = rows.index_select(0, torch.from_numpy(idx).to(rows.device)).cpu().numpy()
    return {name: kept.astype(np.float32, copy=False), name + "_rows": idx.astype(np.float64)}


def write_outputs(directory, arrays):
    """One ``directory/<name>.npy`` per array: float32 / float64 only, DUMP_LIMIT_BYTES in all."""
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, total
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def algorithmic(sr, Fr, Hr, kp):
    """Algorithmic work per hop-frame (SURVEY.md section 8(d)); bytes are float32 in / float32 out."""
    bins = Fr // 2 + 1
    ac_flop = 2 * sum(Fr - l for l in range(N_LAGS + 1))
    return {
        # stage: (bound, units per hop-frame, unit)
        "fold": ("hbm", Hr * 4 + 8 * kp * 2, "B"),                     # signal hop in, fp16 hi/lo planes out
        "stft_gemm": ("tensor", 2 * Fr * 2 * bins, "FLOP"),            # DFT-as-GEMM, one pass
        "mel_db": ("hbm", bins * 4 + N_MELS * 4, "B"),                 # power in, dB out (unfused path only)
        "dct_stats": ("hbm", N_MELS * 4 + 2 * N_MFCC * 4 + N_MFCC * 4, "B"),
        "cmvn_delta_reduce": ("hbm", N_MFCC * 4 + 3 * N_MFCC * 4 / 2, "B"),
        "autocorr": ("tensor", ac_flop, "FLOP"),                       # one pass of the lag products
    }


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        return {"hbm": d["hbm_gbs"], "tensor": d["bf16_tflops_sustained"], "tensor_burst": d["bf16_tflops"],
                "sm_max_mhz": d.get("sm_max_mhz", 1965.0), "source": "measured"}
    return {"hbm": 6650.0, "tensor": 1400.0, "tensor_burst": 1590.0, "sm_max_mhz": 1965.0,
            "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            parts = [x.strip() for x in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        # the median over samples taken UNDER LOAD (idle samples sit at the idle clock)
        busy = [s for s in sm if s > 0.5 * max(mx)] if sm and mx else sm
        return {"sm_mhz": float(np.median(busy or sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---- CPU oracle timing ----------------------------------------------------------------------------
_CPU = {}        # per-worker state: base clips, facial CSV path, temp dir


def _cpu_init(specs, tmpdir):
    """Pool initializer (runs once in every worker): pins the math libraries to one thread, imports the oracle
    and synthesises the base clips, so that a timed task contains nothing but the reference arithmetic."""
    try:
        from threadpoolctl import threadpool_limits
        _CPU["limit"] = threadpool_limits(limits=1)
    except Exception:  # noqa: BLE001 - the environment variables set at the top already pin the libraries
        pass
    from neurosync_trainer_lite_b200 import synth
    from oracle import feature_oracle as fo
    _CPU["fo"] = fo
    _CPU["tmp"] = tmpdir
    kinds = ("voiced", "noise", "gated", "voiced")
    for name, (sr, seconds) in specs.items():
        clips = [synth.synth_clip(seconds, sr, seed=900 + i, kind=kinds[i % 4]) for i in range(4)]
        _CPU[name] = clips
        _CPU[name + "_i16"] = [synth.to_int16_pcm(0.8 * c) for c in clips]
    if any(WORKLOADS[n]["collect"] for n in specs):
        import pandas as pd
        facial = synth.synth_facial(FACIAL_ROWS, seed=0)
        cols = ["Timecode", "BlendshapeCount"] + [f"bs{i}" for i in range(FACIAL_COLS)]
        path = os.path.join(tmpdir, f"facial_{os.getpid()}_iPhone_cal.csv")
        pd.DataFrame(np.hstack([np.zeros((FACIAL_ROWS, 2)), facial]), columns=cols).to_csv(path, index=False)
        _CPU["facial_csv"] = path


def _cpu_task(args):
    """One clip through the reference arithmetic.  mode:
    'array'   extract_and_combine_features(y float32)                  (extract_features.py:26-46)
    'wav'     int16 PCM -> /32768 -> peak normalise -> features        (extract_audio_features :6-24, no file read)
    'collect' 'wav' + facial CSV read + collect_features augmentation, feature-cache CSV write patched out
    'collect_csv'  the same INCLUDING the audio_features.csv write     (data_processing.py:108-177)"""
    name, mode, idx = args
    w = WORKLOADS[name]
    fo = _CPU["fo"]
    t0 = time.perf_counter()
    if mode == "array":
        out = fo.extract_and_combine_features(_CPU[name][idx % 4], w["sr"], w["F"], w["H"])
    else:
        y = _CPU[name + "_i16"][idx % 4].astype(np.float32) / np.float32(32768)
        out, _ = fo.extract_audio_features_from_array(y, w["sr"])
        if mode.startswith("collect"):
            import pandas as pd
            if mode == "collect_csv":
                pd.DataFrame(out).to_csv(os.path.join(_CPU["tmp"], f"audio_features_{os.getpid()}.csv"), index=False)
            facial = pd.read_csv(_CPU["facial_csv"]).drop(columns=["Timecode", "BlendshapeCount"]).values
            out, _f = fo.collect_from_arrays(out, facial, **w["collect"])
    return time.perf_counter() - t0, out.shape[0]


class CpuOracle:
    """The CPU oracle on one worker process per host core (one clip per task); one pool for every workload."""

    def __init__(self, names, procs=None):
        import multiprocessing as mp
        self.cores = procs or len(os.sched_getaffinity(0)) or os.cpu_count() or 1
        self.tmp = tempfile.mkdtemp(prefix="nsf_cpu_")
        specs = {n: (WORKLOADS[n]["sr"], WORKLOADS[n]["seconds"]) for n in names}
        self.pool = mp.get_context("spawn").Pool(self.cores, initializer=_cpu_init, initargs=(specs, self.tmp))
        for n in names:                                                     # warm: imports, FFT plans, tables
            self.pool.map(_cpu_task, [(n, "wav", i) for i in range(self.cores)], chunksize=1)

    def clips_per_step(self, name):
        # one 30 s clip costs ~1.5 s of one core, one 2 s @ 16 kHz clip ~16 ms: bound the sample
        return self.cores * (2 if WORKLOADS[name]["seconds"] > 10 else 100)

    def step(self, name, mode="wav", clips=None):
        """-> dict(value = audio-s per WALL second with every worker busy, wall, busy-time figures)"""
        n = clips or self.clips_per_step(name)
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_task, [(name, mode, i) for i in range(n)], chunksize=1)
        wall = time.perf_counter() - t0
        busy = sum(r[0] for r in res)
        audio = n * WORKLOADS[name]["seconds"]
        return {"value": audio / wall, "wall_s": wall, "audio_s": audio, "clips": n,
                "value_busy_time": self.cores * audio / busy,       # excludes pool hand-off: all workers back to back
                "single_process_value": audio / busy}

    def describe(self, name, r, mode):
        return (f"{r['clips']} clips x {WORKLOADS[name]['seconds']:g} s ({r['audio_s']:g} audio-s) per step, mode "
                f"'{mode}', {self.cores} worker processes x 1 BLAS thread, wall {r['wall_s']:.2f} s")

    def baseline(self, name, mode="wav"):
        r = self.step(name, mode)
        return {"value": r["value"], "unit": "audio-s/s", "cores": self.cores, "kind": "port",
                "threads_per_worker": 1, "sample": self.describe(name, r, mode),
                "value_busy_time": r["value_busy_time"], "single_process_value": r["single_process_value"]}

    def close(self):
        self.pool.close()
        self.pool.join()
        shutil.rmtree(self.tmp, ignore_errors=True)


def run_reference(args, rank, world):
    """CPU oracle on all host cores; rank 0 only (the other ranks exit without work)."""
    if rank != 0:
        return
    name = args.workload
    mode = "collect" if WORKLOADS[name]["collect"] else "wav"
    cpu = CpuOracle([name])
    for _ in range(max(0, min(args.warmup, 1))):
        cpu.step(name, mode)
    res, t0 = [], time.perf_counter()
    for _ in range(args.steps):
        res.append(cpu.step(name, mode))
    total = time.perf_counter() - t0
    cpu.close()
    audio = sum(r["audio_s"] for r in res)
    value = audio / total                                            # wall clock over the whole timed region
    sample = cpu.describe(name, res[-1], mode)
    line = {
        "impl": "reference", "metric": "audio_seconds_per_second", "value": value, "unit": "audio-s/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total / max(args.steps, 1) * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOADS[name]["desc"], "sample": sample, "input": "int16 PCM (host)",
                   "note": "CPU oracle = NumPy restatement of the reference path pinned bit-exact to the "
                           "reference files (librosa itself is not installable here); value = audio-seconds of "
                           "the sample / wall seconds of the timed region"},
        "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": cpu.cores, "kind": "port",
                         "threads_per_worker": 1, "sample": sample,
                         "value_busy_time": float(np.mean([r["value_busy_time"] for r in res])),
                         "value_per_core": value / cpu.cores},
        "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa_node(index):
    """Pin this rank to the CPUs next to its GPU (NVML's ideal affinity) BEFORE any pinned buffer is
    allocated, so the staging memory of the host path is NUMA-local to the GPU's PCIe root."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = [64 * w + bit for w, word in enumerate(mask) for bit in range(64) if (word >> bit) & 1]
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return f"{len(allowed)} cpus ({allowed[0]}-{allowed[-1]})"
    except Exception as e:  # noqa: BLE001 - affinity is an optimisation, never a requirement
        return f"unavailable ({type(e).__name__})"
    return "unchanged"


# ---- native arm -------------------------------------------------------------------------------------
class Dist:
    """torch.distributed plumbing: barrier and max-over-ranks only (no collective on the data path)."""

    def __init__(self, world, local_rank):
        import torch
        self.torch, self.world, self.dist = torch, world, None
        self.dev = torch.device("cuda", local_rank)
        torch.cuda.set_device(self.dev)
        if world > 1:
            import torch.distributed as dist
            os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout for the one JSON line
            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max(self, x):
        if self.dist is None:
            return float(x)
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum(self, x):
        if self.dist is None:
            return float(x)
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


def make_inputs(name, rank, world, scaling):
    """This rank's clips of workload `name`: (packed float32 PCM, offsets, base clips, global clip indices)."""
    from neurosync_trainer_lite_b200 import engine, shard, synth
    w = WORKLOADS[name]
    n_base = 50 if name == "c5" else 6                # distinct signals; the rest are rotations of them
    kinds = ("voiced", "voiced", "noise", "voiced", "gated", "voiced")
    if scaling == "strong":
        # the workload's clips split over the ranks (BASELINE configs[2], [4]); clip i is the same signal
        # whatever N is, so every N computes the same dataset
        n_total = w["clips"]
        n_samples = int(round(w["seconds"] * w["sr"]))
        mine = shard.lpt_partition([n_samples] * n_total, world)[rank]
        seed0 = 0
    else:
        n_total = w["clips"] * world
        mine = list(range(rank * w["clips"], (rank + 1) * w["clips"]))
        seed0 = 100 * rank
    base = [synth.synth_clip(w["seconds"], w["sr"], seed=seed0 + s, kind=kinds[s % 6]) for s in range(n_base)]
    clips = []
    for i in (mine if scaling == "strong" else range(len(mine))):
        b = base[i % n_base]
        clips.append(b if i < n_base else np.roll(b, 997 * (i // n_base)))
    packed, off = engine.pack_clips(clips, dtype=np.float32)
    return packed, off, base, mine, n_total


def measure_workload(name, scaling, steps, warmup, D, rank, world, local_rank, detail, dump=False):
    """One workload on this rank's GPU: device-resident throughput, per-kernel stage times, end-to-end runs through
    the host entry points.  Returns a dict on every rank (timings are already max-over-ranks); with ``dump`` its
    ``_outputs`` holds the rows of the last timed step (see --dump-outputs)."""
    import torch
    from neurosync_trainer_lite_b200 import _native as nv
    from neurosync_trainer_lite_b200 import engine, synth
    w = WORKLOADS[name]
    sr, Fr, Hr, seconds, collect = w["sr"], w["F"], w["H"], w["seconds"], w["collect"]
    dev = D.dev
    eng = engine.get_engine(sr, Fr, Hr, device=local_rank)
    packed, off, base, mine, n_total = make_inputs(name, rank, world, scaling)
    n_clips = len(off) - 1
    total_audio = n_total * seconds                      # audio-seconds ALL ranks process per step
    rows = int(eng.row_offsets(off)[-1])
    frames = sum(eng.plan.hop_frames(int(n)) for n in np.diff(off))

    # ---- device-resident: PCM already in HBM -----------------------------------------------------
    pcm = torch.from_numpy(packed).to(dev)
    out = torch.empty((rows, 256), dtype=torch.float32, device=dev)
    ws = torch.empty(eng.workspace_bytes(len(packed), n_clips), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)
    col = None
    if collect:
        facial_h = np.concatenate([synth.synth_facial(FACIAL_ROWS, seed=int(i) % 6) for i in mine]).astype(np.float32)
        f_off = np.arange(n_clips + 1, dtype=np.int64) * FACIAL_ROWS
        a_off = eng.row_offsets(off)
        o_off = eng.collect_rows(a_off, f_off, **collect)
        col = {"facial_h": facial_h, "facial": torch.from_numpy(facial_h).to(dev), "f_off": f_off, "a_off": a_off,
               "o_off": o_off,
               "out_a": torch.empty((int(o_off[-1]), 256), dtype=torch.float32, device=dev),
               "out_f": torch.empty((int(o_off[-1]), FACIAL_COLS), dtype=torch.float32, device=dev)}

    def device_step():
        eng.extract_device(pcm, off, 0, out=out, workspace=ws)
        if col:
            eng.collect_device(out, col["a_off"], col["facial"], col["f_off"], out_audio=col["out_a"],
                               out_facial=col["out_f"], out_offsets=col["o_off"], **collect)

    for _ in range(max(warmup, 3)):
        device_step()
    D.barrier()
    launches0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        device_step()
    e1.record(stream)
    D.barrier()
    dev_ms = D.max(e0.elapsed_time(e1))
    launches = eng.launch_count() - launches0
    outputs = None
    if dump:                                           # read back after the timed region, before anything reuses `out`
        outputs = sample_rows("features", out)
        if col:
            outputs.update(sample_rows("collect_audio", col["out_a"]))
            outputs.update(sample_rows("collect_facial", col["out_f"]))

    # per-kernel stage times (CUDA events recorded by the library on the same stream)
    eng.set_profiling(True)
    acc = {}
    reps = max(3, min(steps, 10))
    for _ in range(reps):
        eng.extract_device(pcm, off, 0, out=out, workspace=ws)
        torch.cuda.synchronize(dev)
        for k, v in eng.stage_times_ms().items():
            acc[k] = acc.get(k, 0.0) + v / reps
    eng.set_profiling(False)
    if col:                                            # the augmentation kernel on its own (CUDA events, same stream)
        reps = 10
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        c0.record(stream)
        for _ in range(reps):
            eng.collect_device(out, col["a_off"], col["facial"], col["f_off"], out_audio=col["out_a"],
                               out_facial=col["out_f"], out_offsets=col["o_off"], **collect)
        c1.record(stream)
        torch.cuda.synchronize(dev)
        acc["collect"] = c0.elapsed_time(c1) / reps
    del pcm, out, ws
    torch.cuda.empty_cache()

    # ---- end to end through the C ABI with host buffers ------------------------------------------
    pcm16 = synth.to_int16_pcm(packed)
    pin16 = engine.PinnedBuffer(pcm16.nbytes)
    h16 = pin16.view(np.int16, pcm16.shape)
    h16[:] = pcm16
    del pcm16
    pin_in = engine.PinnedBuffer(packed.nbytes)
    h_in = pin_in.view(np.float32, packed.shape)
    h_in[:] = packed
    shared, gather_error = None, None
    if col:
        n_o = int(col["o_off"][-1])
        pin_f = engine.PinnedBuffer(col["facial_h"].nbytes)
        h_f = pin_f.view(np.float32, col["facial_h"].shape)
        h_f[:] = col["facial_h"]
        if name == "c4" and world > 1:
            # "features gathered to host": ONE (world * n_o, 256) float32 array in shared memory that every rank
            # page-locks (cudaHostRegister) and fills at its own row offset by DMA - no second host copy, no collective
            shared = SharedGather(f"nsf_c4_{os.environ.get('MASTER_PORT', '0')}", world * n_o, rank, D)
            if not shared.ok:                      # registration refused on this box: private buffers, and say so
                gather_error, shared = shared.error, None
        if shared is not None:
            h_oa, h_of = shared.audio[rank * n_o:(rank + 1) * n_o], shared.facial[rank * n_o:(rank + 1) * n_o]
        else:
            pin_oa = engine.PinnedBuffer(n_o * 256 * 4)
            pin_of = engine.PinnedBuffer(n_o * FACIAL_COLS * 4)
            h_oa, h_of = pin_oa.view(np.float32, (n_o, 256)), pin_of.view(np.float32, (n_o, FACIAL_COLS))
        d2h = n_o * (256 + FACIAL_COLS) * 4
    else:
        pin_out = engine.PinnedBuffer(rows * 256 * 4)
        h_out = pin_out.view(np.float32, (rows, 256))
        d2h = rows * 256 * 4

    def host_step(src, flags):
        if col:       # nsf_extract_collect_host: PCM and facial rows up, augmented rows back, features stay on the device
            eng.extract_collect_host(src, off, h_f, col["f_off"], flags, out_audio=h_oa, out_facial=h_of, **collect)
        else:
            eng.extract_host(src, off, flags, out=h_out)     # synchronous: returns when rows are on the host

    def timed_host(src, flags):
        for _ in range(max(warmup, 3)):
            host_step(src, flags)
        D.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            host_step(src, flags)
        torch.cuda.synchronize(dev)
        dt = D.max(time.perf_counter() - t0)
        D.barrier()
        return dt

    e2e16_s = timed_host(h16, nv.PEAK_NORMALIZE)
    first_rows16 = None if col else h_out[: int(eng.row_offsets(off)[1])].copy()
    e2e32_s = timed_host(h_in, 0)
    checksum = float(np.abs((h_oa if col else h_out)[::997]).sum())
    first_rows = None if col else h_out[: int(eng.row_offsets(off)[1])].copy()      # clip 0, float32-PCM path

    # ---- bare copy ceiling: the same bytes over the same links, nothing else -----------------------
    ceiling = copy_ceiling(D, h16.nbytes + (h_f.nbytes if col else 0), d2h, steps) if detail or world > 1 else None

    # parity spot check against the oracle (outside every timed region): clip 0 of rank 0
    parity = None
    if rank == 0 and not col:
        from oracle import feature_oracle as fo
        want = fo.extract_and_combine_features(base[0], sr, Fr, Hr)
        d = np.abs(first_rows - want)
        y16 = synth.to_int16_pcm(base[0]).astype(np.float32) / np.float32(32768)
        want16, _ = fo.extract_audio_features_from_array(y16, sr)
        d16 = np.abs(first_rows16 - want16)
        parity = {"clip": 0, "mfcc_max_abs": float(d[:, :23].max()), "delta_max_abs": float(d[:, 23:69].max()),
                  "autocorr_max_abs": float(d[:, 69:].max()),
                  "int16_path": {"mfcc_max_abs": float(d16[:, :23].max()), "delta_max_abs": float(d16[:, 23:69].max()),
                                 "autocorr_max_abs": float(d16[:, 69:].max())}}
    gathered = {"error": gather_error} if gather_error else None
    if shared is not None:
        gathered = shared.verify_and_close(h_oa, rank, world, n_o)

    pk = peaks()
    ms_per_step = dev_ms / steps
    alg = algorithmic(sr, Fr, Hr, eng.plan.fold_kp)
    fma_peak = 148 * 128 * 2 * pk["sm_max_mhz"] * 1e6 / 1e12     # fp32 FMA TFLOP/s at max clock
    if acc.get("mel_db", 0.0) < 0.02:
        # fused product path: the mel projection and dB run in the epilogue of the tcgen05 kernel, so the
        # "stft_gemm" stage is credited with the DFT and the mel GEMM FLOPs (SURVEY section 8(d))
        bins = Fr // 2 + 1
        alg["stft_gemm"] = ("tensor", alg["stft_gemm"][1] + 2 * bins * N_MELS, "FLOP")
        acc["stft_gemm"] = acc.get("stft_gemm", 0.0) + acc.pop("mel_db", 0.0)
        alg.pop("mel_db")
    if col:
        # rows in and rows out, 256 + 61 float32 columns each (SURVEY section 8(d), K5), expressed per hop-frame
        moved = (int(col["a_off"][-1]) + int(col["o_off"][-1])) * (256 + FACIAL_COLS) * 4
        alg["collect"] = ("hbm", moved / frames, "B")
    kernels = []
    for kname, (bound, units, unit) in alg.items():
        ms = acc.get(kname, 0.0)
        if ms <= 0:
            continue
        per_s = units * frames / (ms * 1e-3)
        if bound == "hbm":
            ach, peak, u = per_s / 1e9, pk["hbm"], "GB/s"
        else:
            ach, peak, u = per_s / 1e12, pk["tensor"], "TFLOP/s"
        kernels.append({"kernel": kname, "ms": round(ms, 4), "bound": bound, "achieved": round(ach, 2),
                        "peak": round(peak, 1), "unit": u, "frac": round(ach / peak, 4)})
    # executed (issued) tensor work where it differs from the algorithmic count: the split-fp16 products
    hmma_peak = 553.0                                   # mma.sync m16n8k16 f16, measured (profiles/ubench_mma_b200.txt)
    for k in kernels:
        ms = k["ms"] * 1e-3
        if k["kernel"] == "autocorr":
            nblk = (Fr + 15) // 16                      # K-blocks that hold samples (all-zero blocks are skipped)
            # MMAs the kernel issues per frame (nsf_autocorr_mma.cu, launch_autocorr_mma): the five-tile loop from 44
            # K-blocks up and at F = 266 (5 nblk - 12), the six-MMA loop otherwise (6 nblk minus the 12 zero-operand MMAs of
            # the first group)
            static_five = (Fr // 2 + 1 + 31) // 32 == 5 and nblk == 17          # F = 266: am_mma5_static<17>
            five = os.environ.get("NSF_AC_LOOP", "")[:1] == "f" or (os.environ.get("NSF_AC_LOOP", "")[:1] != "s"
                                                                   and (nblk >= 44 or static_five))
            mmas = max((5 if five else 6) * nblk - 12, nblk)
            ex = frames * mmas * 4096 / ms / 1e12
            # the lag products are a banded Toeplitz matrix-VECTOR product per frame (no operand shared between
            # frames), which only the warp-level HMMA pipe can fill: its measured peak is the relevant ceiling,
            # and the same FLOPs on the fp32 FMA pipe (the reference algorithm's pipe) are given for scale
            k.update(executed_tflops=round(ex, 1), executed_pipe=f"mma.sync (HMMA), split-fp16 products, {mmas} MMAs per frame",
                     executed_peak=hmma_peak, executed_frac=round(ex / hmma_peak, 4),
                     fp32_fma_peak=round(fma_peak, 1), frac_of_fp32_fma_peak=round(k["achieved"] / fma_peak, 4))
        elif k["kernel"] == "stft_gemm":
            kp = eng.plan.fold_kp
            npad = (eng.plan.fold_kp + 127) // 128 * 128          # bins per chain rounded to 128-wide tiles
            chains = eng.plan.chains
            ex = -(-frames // 128) * 128 * chains * 2 * 3 * 2.0 * kp * npad / ms / 1e12
            k.update(executed_tflops=round(ex, 1), executed_pipe="tcgen05 kind::f16, 3 split-fp16 products",
                     executed_peak=pk["tensor"], executed_frac=round(ex / pk["tensor"], 4))
    kernels.sort(key=lambda k: -k["ms"])

    h2d16 = int(h16.nbytes) + (int(h_f.nbytes) if col else 0)
    h2d32 = int(h_in.nbytes) + (int(h_f.nbytes) if col else 0)
    api = "nsf_extract_collect_host" if col else "nsf_extract_host"
    res = {
        "workload": w["desc"], "scaling": scaling, "value": total_audio / (ms_per_step * 1e-3), "unit": "audio-s/s",
        "ms_per_step": ms_per_step, "steps": steps, "clips_this_rank": n_clips, "clips_total": n_total,
        "audio_seconds_per_step": total_audio, "rows_this_rank": rows, "hop_frames_this_rank": frames,
        "collect_rows_this_rank": int(col["o_off"][-1]) if col else None,
        "e2e": {"value": total_audio * steps / e2e16_s, "unit": "audio-s/s", "h2d_bytes_per_step": h2d16,
                "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e16_s / steps * 1e3,
                "api": f"{api}(NSF_PCM_I16, NSF_PEAK_NORMALIZE), page-locked host buffers"},
        "e2e_f32_pcm": {"value": total_audio * steps / e2e32_s, "unit": "audio-s/s", "h2d_bytes_per_step": h2d32,
                        "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e32_s / steps * 1e3,
                        "api": f"{api}(NSF_PCM_F32), page-locked host buffers"},
        "gpu_launches": int(launches), "kernels": kernels, "parity": parity, "checksum": checksum,
        "gathered_host_array": gathered,
    }
    if ceiling:
        ceiling["e2e_frac_of_ceiling"] = round(ceiling["ms_per_step"] / res["e2e"]["ms_per_step"], 4)
        res["copy_ceiling"] = ceiling
    res["_frames"] = frames
    res["_outputs"] = outputs
    return res


class SharedGather:
    """One float32 array in /dev/shm shared by the ranks of the box, page-locked in every rank
    (nsf_host_register), into which each rank's rows arrive by DMA at the rank's row offset."""

    def __init__(self, tag, total_rows, rank, D):
        from neurosync_trainer_lite_b200 import _native as nv
        self.nv, self.D, self.rank = nv, D, rank
        base = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
        self.paths = [os.path.join(base, f"{tag}_{k}.f32") for k in ("audio", "facial")]
        shapes = [(total_rows, 256), (total_rows, FACIAL_COLS)]
        if rank == 0:
            for p, s in zip(self.paths, shapes):
                np.memmap(p, dtype=np.float32, mode="w+", shape=s).flush()
        D.barrier()
        self.audio, self.facial = (np.memmap(p, dtype=np.float32, mode="r+", shape=s) for p, s in zip(self.paths, shapes))
        t0 = time.perf_counter()
        self.error, done = None, []
        try:
            for a in (self.audio, self.facial):
                nv.check(nv.lib.nsf_host_register(nv.ptr(a), a.nbytes))
                done.append(a)
        except nv.NsfError as e:
            self.error = str(e)
        self.register_s = time.perf_counter() - t0
        self.ok = D.sum(0.0 if self.error else 1.0) == D.world      # every rank takes the same branch
        if not self.ok:
            self.error = self.error or "registration failed on another rank"
            for a in done:
                nv.lib.nsf_host_unregister(nv.ptr(a))
            del self.audio, self.facial
            D.barrier()
            if rank == 0:
                for p in self.paths:
                    if os.path.exists(p):
                        os.unlink(p)
            return
        D.barrier()

    def verify_and_close(self, my_rows, rank, world, n_o):
        """Every rank's slice must be visible to rank 0 in the ONE array (checksum per slice)."""
        self.D.barrier()
        mine = float(np.abs(my_rows[::997]).sum())
        ok = True
        sums = []
        if rank == 0:
            sums = [float(np.abs(self.audio[r * n_o:(r + 1) * n_o][::997]).sum()) for r in range(world)]
            ok = all(s > 0 for s in sums) and abs(sums[0] - mine) < 1e-6 * max(1.0, mine)
        info = {"shape": list(self.audio.shape), "bytes": int(self.audio.nbytes + self.facial.nbytes),
                "backing": "/dev/shm mapping page-locked with cudaHostRegister in every rank; each rank DMAs its "
                           "rows to its own offset", "register_seconds": round(self.register_s, 3),
                "all_slices_filled": bool(ok)}
        for a in (self.audio, self.facial):
            self.nv.lib.nsf_host_unregister(self.nv.ptr(a))
        self.D.barrier()
        del self.audio, self.facial
        if rank == 0:
            for p in self.paths:
                if os.path.exists(p):
                    os.unlink(p)
        return info


def copy_ceiling(D, h2d_bytes, d2h_bytes, steps):
    """Bare page-locked H2D + D2H of the e2e step's bytes on two streams (both directions at once), all ranks
    together: what the host link gives when nothing else happens.  torch is the allocator and copy engine here."""
    torch = D.torch
    dev = D.dev
    hin = torch.empty(h2d_bytes, dtype=torch.uint8, pin_memory=True)
    hout = torch.empty(d2h_bytes, dtype=torch.uint8, pin_memory=True)
    din = torch.empty(h2d_bytes, dtype=torch.uint8, device=dev)
    dout = torch.empty(d2h_bytes, dtype=torch.uint8, device=dev)
    s_up, s_down = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def go():
        with torch.cuda.stream(s_up):
            din.copy_(hin, non_blocking=True)
        with torch.cuda.stream(s_down):
            hout.copy_(dout, non_blocking=True)

    for _ in range(2):
        go()
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        go()
    torch.cuda.synchronize(dev)
    dt = D.max(time.perf_counter() - t0)
    D.barrier()
    # upload alone (the longer leg)
    t0 = time.perf_counter()
    for _ in range(steps):
        with torch.cuda.stream(s_up):
            din.copy_(hin, non_blocking=True)
    torch.cuda.synchronize(dev)
    up = D.max(time.perf_counter() - t0)
    D.barrier()
    ms = dt / steps * 1e3
    return {"ms_per_step": ms, "h2d_bytes": int(h2d_bytes), "d2h_bytes": int(d2h_bytes),
            "h2d_gbs_per_gpu": round(h2d_bytes / (up / steps) / 1e9, 2),
            "both_directions_gbs_per_gpu": round((h2d_bytes + d2h_bytes) / (dt / steps) / 1e9, 2),
            "what": "page-locked cudaMemcpyAsync of the same bytes, upload and download on separate streams, "
                    "all ranks at once, max over ranks"}


def api_e2e(D, rank, world, local_rank, steps):
    """The reference-named dataset builder end to end: a synthetic 60-take tree (audio.wav int16 @ 88.2 kHz +
    facial CSV per folder, binary feature cache) through dataset.data_processing.load_data -> examples."""
    import pandas as pd
    from neurosync_trainer_lite_b200 import synth
    from neurosync_trainer_lite_b200.dataset import data_processing as dp
    n_takes, seconds = 60, 30.0
    base = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    root = tempfile.mkdtemp(prefix=f"nsf_tree_r{rank}_", dir=base)
    try:
        kinds = ("voiced", "voiced", "noise", "voiced", "gated", "voiced")
        wavs = [synth.wav_bytes(synth.to_int16_pcm(0.8 * synth.synth_clip(seconds, 88200, seed=700 + s, kind=kinds[s])), 88200)
                for s in range(6)]
        cols = ["Timecode", "BlendshapeCount"] + [f"bs{i}" for i in range(FACIAL_COLS)]
        csvs = [pd.DataFrame(np.hstack([np.zeros((FACIAL_ROWS, 2)), synth.synth_facial(FACIAL_ROWS, seed=s)]),
                             columns=cols).to_csv(index=False) for s in range(6)]
        for k in range(n_takes):
            take = os.path.join(root, f"take_{k:03d}")
            os.makedirs(take)
            with open(os.path.join(take, "audio.wav"), "wb") as fh:
                fh.write(wavs[k % 6])
            with open(os.path.join(take, f"take{k:03d}_iPhone_cal.csv"), "w") as fh:
                fh.write(csvs[k % 6])
        os.environ["NSF_FEATURE_CACHE"] = "npy"
        os.environ["NSF_DEVICE"] = str(local_rank)

        def clear():
            for k in range(n_takes):
                p = os.path.join(root, f"take_{k:03d}", "audio_features.npy")
                if os.path.exists(p):
                    os.unlink(p)

        import contextlib
        import io
        times, phases = [], {}
        for it in range(steps + 1):                      # first pass = warm-up (arenas, page cache)
            clear()
            D.barrier()
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                ex = dp.load_data(root, 88200, set())
            dt = time.perf_counter() - t0
            assert len(ex) == n_takes and ex[0][0].shape == (2670, 256) and ex[0][1].shape == (2670, FACIAL_COLS)
            if it:
                times.append(dt)
                for k, v in dp.last_timing.items():
                    phases[k] = phases.get(k, 0.0) + v / steps
            del ex
        dt = D.max(float(np.mean(times)))
        return {"value": world * n_takes * seconds / dt, "unit": "audio-s/s", "ms_per_step": dt * 1e3,
                "api": "dataset.data_processing.load_data(root_dir, 88200, set()) on a 60-take tree per rank "
                       "(audio.wav int16 + *_iPhone_cal.csv, NSF_FEATURE_CACHE=npy), tree in /dev/shm",
                "phases_ms": {k: round(v * 1e3, 2) for k, v in phases.items()},
                "what_is_inside": "folder scan, WAV payloads read into page-locked memory by a thread pool, facial "
                                  "CSVs parsed by pandas (thread pool), fused extract + collect on the device, "
                                  "feature caches written (.npy), examples returned as float32 arrays"}
    finally:
        shutil.rmtree(root, ignore_errors=True)
        os.environ.pop("NSF_FEATURE_CACHE", None)


def run_single_process(args):
    """BASELINE configs[3] as SURVEY.md section 8(d) states it: ONE process, one library context and one host thread
    per GPU, every GPU downloading straight into its slice of ONE page-locked (rows, 256) host array.  End to end
    only (host int16 PCM in, gathered augmented rows out); wall clock around the whole call."""
    import __graft_entry__ as g
    g.build_library()
    import torch
    from neurosync_trainer_lite_b200 import engine, shard, synth
    n = args.gpus
    if torch.cuda.device_count() < n:
        raise RuntimeError(f"--single-process --gpus {n} needs {n} visible GPUs")
    name = args.workload
    w = WORKLOADS[name]
    if not w["collect"]:
        raise RuntimeError("--single-process runs the collect workloads (c3, c4)")
    parts = [make_inputs(name, r, n, "weak") for r in range(n)]
    packed = np.concatenate([p[0] for p in parts])
    lens = np.concatenate([np.diff(p[1]) for p in parts])
    off = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    n_clips = len(lens)
    pcm16 = synth.to_int16_pcm(packed)
    del packed, parts
    pin_in = engine.PinnedBuffer(pcm16.nbytes)
    h16 = pin_in.view(np.int16, pcm16.shape)
    h16[:] = pcm16
    del pcm16
    facial = np.concatenate([synth.synth_facial(FACIAL_ROWS, seed=i % 6) for i in range(n_clips)]).astype(np.float32)
    pin_f = engine.PinnedBuffer(facial.nbytes)
    h_f = pin_f.view(np.float32, facial.shape)
    h_f[:] = facial
    f_off = np.arange(n_clips + 1, dtype=np.int64) * FACIAL_ROWS
    from neurosync_trainer_lite_b200 import _native as nv
    devices = list(range(n))
    out_a = out_f = None
    times = []
    for it in range(max(args.warmup, 2) + args.steps):
        t0 = time.perf_counter()
        out_a, out_f, o_off = shard.extract_collect_multi_device(h16, off, h_f, f_off, devices, sr=w["sr"], flags=nv.PEAK_NORMALIZE,
                                                                 out_audio=out_a, out_facial=out_f, **w["collect"])
        if it >= max(args.warmup, 2):
            times.append(time.perf_counter() - t0)
    dt = float(np.mean(times))
    audio_s = n_clips * w["seconds"]
    filled = [bool(np.abs(out_a[o_off[c]:o_off[c] + 4]).sum() > 0) for c in range(0, n_clips, max(1, n_clips // (2 * n)))]
    line = {
        "metric": "audio_seconds_per_second", "value": audio_s / dt, "unit": "audio-s/s", "n_gpus": n, "steps": args.steps,
        "warmup": max(args.warmup, 2), "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "mode": "single-process, one thread + context per GPU",
        "config": {"workload": w["desc"], "clips_total": n_clips, "audio_seconds_per_step": audio_s,
                   "sharding": f"by clip, contiguous runs over {n} GPUs, no collective"},
        "e2e": {"value": audio_s / dt, "unit": "audio-s/s", "h2d_bytes_per_step": int(h16.nbytes + h_f.nbytes),
                "d2h_bytes_per_step": int(out_a.nbytes + out_f.nbytes), "ms_per_step": dt * 1e3,
                "api": "shard.extract_collect_multi_device -> nsf_extract_collect_host per device (int16 PCM, page-locked)"},
        "gathered_host_array": {"shape": list(out_a.shape), "bytes": int(out_a.nbytes + out_f.nbytes), "single_process": True,
                                "backing": "one cudaHostAlloc(portable) array; each device DMAs its rows to its own offset",
                                "all_slices_filled": all(filled)},
        "gpu_launches": int(sum(engine.get_engine(w["sr"], w["F"], w["H"], device=d).launch_count() for d in devices)),
    }
    print(json.dumps(line), flush=True)


def run_native(args, rank, world, local_rank):
    import __graft_entry__ as g
    g.build_library()
    from neurosync_trainer_lite_b200 import _native as nv
    if nv.lib.nsf_device_count() < 1:
        raise RuntimeError("bench.py needs an sm_100 GPU: the library has no CPU path")
    D = Dist(world, local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    name = args.workload
    scaling = args.scaling or ("weak" if name in ("c2", "c4") else DEFAULT_SCALING[name])
    warm = max(args.warmup, 3)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    main = measure_workload(name, scaling, args.steps, warm, D, rank, world, local_rank, detail=True,
                            dump=args.dump_outputs is not None and rank == 0)
    clocks = sampler.stop() if sampler else None
    outputs = main.pop("_outputs")
    if outputs:
        write_outputs(args.dump_outputs, outputs)

    extras = {}
    if not args.no_extras and name == "c2":
        for other in ("c3", "c4", "c5"):
            extras[other] = measure_workload(other, DEFAULT_SCALING[other], max(3, min(args.steps, 5)), 3, D, rank, world,
                                             local_rank, detail=False)
    api = api_e2e(D, rank, world, local_rank, max(2, min(args.steps, 3))) if not args.no_extras else None

    if rank != 0:
        D.close()
        return

    pk = peaks()
    # DRAM bytes per launch from the newest committed `ncu --set full` capture (scripts/ncu_extract.py)
    traffic = {}
    import glob
    for tp in sorted(glob.glob(os.path.join(ROOT, "profiles", "ncu_traffic_*.json")), reverse=True):
        with open(tp) as fh:
            cand = json.load(fh)
        if cand.get("workload") == name:                  # newest capture of THIS workload
            traffic = cand
            traffic["file"] = os.path.relpath(tp, ROOT)
            break
    top = main["kernels"][0]
    roofline = {"kernel": top["kernel"], "bound": top["bound"], "achieved": top["achieved"], "peak": top["peak"],
                "unit": top["unit"], "frac": top["frac"],
                "traffic": traffic.get(top["kernel"]) if traffic.get("workload") == name else None,
                "traffic_source": traffic.get("file") if traffic.get("workload") == name else None,
                "executed": {k: top[k] for k in top if k.startswith("executed_")},
                "peak_source": pk["source"] + (" (HBM copy)" if top["bound"] == "hbm" else " (bf16 dense, sustained)"),
                "ms_per_launch": top["ms"], "stage_ms_sum": round(sum(k["ms"] for k in main["kernels"]), 4)}

    cpu = None
    if not args.no_cpu_baseline and world == 1:        # rank 0 at N = 1 only
        names = [name] + list(extras)
        c = CpuOracle(names)
        mode = "collect" if WORKLOADS[name]["collect"] else "wav"
        cpu = c.baseline(name, mode)
        cpu["array_input"] = c.baseline(name, "array") if mode == "wav" else None    # extract_and_combine_features(y f32)
        for other, r in extras.items():
            if WORKLOADS[other]["collect"]:
                r["cpu_baseline"] = c.baseline(other, "collect")                       # BASELINE.md section 3 (ii)
                r["cpu_baseline"]["with_csv_cache_write"] = c.baseline(other, "collect_csv")   # (iii)
            else:
                r["cpu_baseline"] = c.baseline(other, "wav")
        c.close()
    for r in list(extras.values()) + [main]:
        r.pop("_frames", None)
        r.pop("_outputs", None)

    line = {
        "metric": "audio_seconds_per_second", "value": main["value"], "unit": "audio-s/s", "n_gpus": world,
        "steps": args.steps, "warmup": warm, "ms_per_step": main["ms_per_step"],
        "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": main["workload"], "clips_per_gpu": main["clips_this_rank"],
                   "clips_total": main["clips_total"], "audio_seconds_per_step": main["audio_seconds_per_step"],
                   "rows_per_gpu_step": main["rows_this_rank"], "hop_frames_per_gpu_step": main["hop_frames_this_rank"],
                   "collect_rows_per_gpu_step": main["collect_rows_this_rank"],
                   "sharding": f"by clip, {world} rank(s), no collective", "cpu_affinity": numa,
                   "l2": "inputs (635 MB of float32 PCM for c2) + intermediates exceed the 126 MB L2 every step"},
        "e2e": main["e2e"], "e2e_f32_pcm": main["e2e_f32_pcm"], "copy_ceiling": main.get("copy_ceiling"),
        "api_e2e": api,
        "gpu_launches": main["gpu_launches"],
        "roofline": roofline, "kernels": main["kernels"], "cpu_baseline": cpu, "clocks": clocks,
        "parity": main["parity"], "checksum": main["checksum"], "gathered_host_array": main["gathered_host_array"],
        "workloads": extras,
    }
    print(json.dumps(line), flush=True)
    D.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"],
                    help="weak: every rank runs the workload's per-rank batch; strong: the workload's clips are split "
                         "over the ranks.  Default: weak for c2 / c4, strong for c3 / c5")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the embedded c3 / c4 / c5 passes and the api_e2e leg")
    ap.add_argument("--single-process", action="store_true",
                    help="c3 / c4 end to end from ONE process driving --gpus N devices (one thread + context each) into one "
                         "page-locked host array; run without torchrun")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32 rows, "
                         "seeded row sample of large outputs, rank 0's share)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl == "reference" or args.single_process):
        ap.error("--dump-outputs writes the device-resident path's rows: not with --impl reference or --single-process")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.single_process:
        run_single_process(args)
    else:
        run_native(args, rank, world, local_rank)


if __name__ == "__main__":
    main()

"""The JSON line of bench.py against the driver's contract (keys, types, consistency), checked on the lines
committed under profiles/ - so a change of bench.py that drops a key shows up on the CPU box - plus the
argument parser and the workload table of bench.py itself (no GPU needed)."""
import glob
import json
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NATIVE = sorted(glob.glob(os.path.join(ROOT, "profiles", "bench_r01[fghi]_*.json")))
REQUIRED = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}


def _line(path):
    with open(path) as fh:
        return json.loads(fh.read().strip().splitlines()[-1])


@pytest.mark.parametrize("path", NATIVE, ids=[os.path.basename(p) for p in NATIVE])
def test_committed_bench_lines_follow_the_contract(path):
    d = _line(path)
    if d.get("impl") == "reference":
        assert d["cpu_baseline"]["kind"] == "port" and d["e2e"]["h2d_bytes_per_step"] == 0
        assert d["e2e"]["value"] == d["value"] == d["cpu_baseline"]["value"]
        return
    assert REQUIRED <= set(d), REQUIRED - set(d)
    assert d["metric"] == "audio_seconds_per_second" and d["unit"] == "audio-s/s" and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"] == "f32"
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["warmup"] >= 3 and d["gpu_launches"] > 0
    # value = audio of all ranks / device time of one step
    audio = d["config"]["audio_seconds_per_gpu_step"] * d["n_gpus"]
    assert d["value"] == pytest.approx(audio / (d["ms_per_step"] * 1e-3), rel=1e-9)
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and 0 < e["value"] < d["value"]
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["frac"] == pytest.approx(r["achieved"] / r["peak"], rel=2e-3)
    assert r["kernel"] == max(d["kernels"], key=lambda k: k["ms"])["kernel"]
    for k in d["kernels"]:
        assert k["bound"] in ("hbm", "tensor") and k["unit"] in ("GB/s", "TFLOP/s") and k["ms"] > 0
    if d["n_gpus"] == 1 and d.get("cpu_baseline"):
        c = d["cpu_baseline"]
        assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] > 0 and "sample" in c
    if d.get("clocks"):
        assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    p = d["parity"]
    assert p["mfcc_max_abs"] < 1e-3 and p["autocorr_max_abs"] < 2e-5


R02 = [os.path.join(ROOT, "profiles", f) for f in ("bench_r02k_n1.json", "bench_r02i_n2.json", "bench_r02l_n4.json",
                                                    "bench_r02l_n8.json", "bench_r02s_n1.json", "bench_r02s_n2.json")]


@pytest.mark.parametrize("path", R02, ids=[os.path.basename(p) for p in R02])
def test_round2_bench_lines_follow_the_contract(path):
    d = _line(path)
    assert REQUIRED <= set(d), REQUIRED - set(d)
    n = d["n_gpus"]
    assert d["metric"] == "audio_seconds_per_second" and d["unit"] == "audio-s/s" and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"] == "f32"
    assert "workload" in d["config"] and "model" not in d["config"] and d["warmup"] >= 3 and d["gpu_launches"] > 0
    assert d["config"]["clips_per_gpu"] == 60 and d["config"]["clips_total"] == 60 * n
    assert d["value"] == pytest.approx(d["config"]["audio_seconds_per_step"] / (d["ms_per_step"] * 1e-3), rel=1e-9)
    for key in ("e2e", "e2e_f32_pcm"):
        e = d[key]
        assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and 0 < e["value"] < d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] * 2 == d["e2e_f32_pcm"]["h2d_bytes_per_step"]        # int16 vs float32 PCM
    c = d["copy_ceiling"]
    assert c["h2d_bytes"] == d["e2e"]["h2d_bytes_per_step"] and c["ms_per_step"] > 0
    assert c["e2e_frac_of_ceiling"] == pytest.approx(c["ms_per_step"] / d["e2e"]["ms_per_step"], rel=2e-3)
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["frac"] == pytest.approx(r["achieved"] / r["peak"], rel=2e-3)
    assert r["kernel"] == max(d["kernels"], key=lambda k: k["ms"])["kernel"] and (r["traffic"] is None or r["traffic"] > 0)
    p = d["parity"]
    assert p["mfcc_max_abs"] < 1e-4 and p["delta_max_abs"] < 2e-5 and p["autocorr_max_abs"] < 2e-5
    assert d["api_e2e"]["value"] > 0 and "facial_csv_wait" in d["api_e2e"]["phases_ms"]
    # the other BASELINE configurations ride in the same line
    w = d["workloads"]
    assert set(w) == {"c3", "c4", "c5"}
    assert w["c3"]["scaling"] == "strong" and w["c3"]["clips_total"] == 60
    assert w["c5"]["scaling"] == "strong" and w["c5"]["clips_total"] == 10000
    assert w["c4"]["clips_this_rank"] == 60 and w["c4"]["clips_total"] == 60 * n
    for x in w.values():
        assert 0 < x["e2e"]["value"] < x["value"] and x["kernels"]
    if n == 1:
        cb = d["cpu_baseline"]
        assert cb["kind"] == "port" and cb["threads_per_worker"] == 1 and cb["cores"] >= 1 and cb["value"] > 0
        assert cb["value"] <= cb["value_busy_time"] * 1.05           # wall clock can only be slower than busy time
        for name in ("c3", "c4"):
            c3 = w[name]["cpu_baseline"]
            assert c3["with_csv_cache_write"]["value"] < c3["value"]  # the CSV write costs the reference time
        assert w["c5"]["cpu_baseline"]["value"] > 0
    else:
        g = w["c4"]["gathered_host_array"]
        assert g["all_slices_filled"] is True and g["shape"] == [n * w["c4"]["collect_rows_this_rank"], 256]
    if d.get("clocks"):
        assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


def test_round2_reference_arm_is_consistent_per_core():
    """The CPU oracle's per-core throughput must not depend on how bench.py was launched (round 1: 1.85x apart)."""
    per_core = []
    for f in ("bench_r02k_ref_n1.json", "bench_r02i_ref_n2.json", "bench_r02l_ref_n8.json", "bench_r02s_ref_n1.json",
              "bench_r02s_ref_n2.json"):
        d = _line(os.path.join(ROOT, "profiles", f))
        assert d["impl"] == "reference" and d["e2e"]["h2d_bytes_per_step"] == 0 and d["gpu_launches"] == 0
        assert d["value"] == d["e2e"]["value"] == d["cpu_baseline"]["value"]
        per_core.append(d["value"] / d["cpu_baseline"]["cores"])
    assert max(per_core) / min(per_core) < 1.10, per_core


def test_round2_scaling_lines():
    lines = {n: _line(os.path.join(ROOT, "profiles", f)) for n, f in
             ((1, "bench_r02k_n1.json"), (2, "bench_r02i_n2.json"), (4, "bench_r02l_n4.json"), (8, "bench_r02l_n8.json"))}
    for n, d in lines.items():
        assert d["n_gpus"] == n
        assert d["value"] > 0.95 * n * lines[1]["value"]                  # device-resident: linear by clip
        assert d["e2e"]["value"] >= lines[1]["e2e"]["value"]              # end to end: the shared host link
    sp = _line(os.path.join(ROOT, "profiles", "bench_r02l_single_process_c4_n8.json"))
    assert sp["gathered_host_array"]["single_process"] and sp["gathered_host_array"]["shape"] == [2994720, 256]
    assert sp["gathered_host_array"]["all_slices_filled"] is True


def test_final_build_lines():
    """Capture r02s (final build of round 2): two ranks double the device-resident value, the executed MMA count in the
    roofline follows the loop the autocorrelation kernel runs, and the 10 000-clip batch is no longer bound by the binding's
    per-clip row-count loop (the step is the sum of its kernels)."""
    one, two = (_line(os.path.join(ROOT, "profiles", f)) for f in ("bench_r02s_n1.json", "bench_r02s_n2.json"))
    assert two["n_gpus"] == 2 and two["value"] > 0.95 * 2 * one["value"] and two["e2e"]["value"] > one["e2e"]["value"]
    assert "448 MMAs per frame" in one["roofline"]["executed"]["executed_pipe"]          # 5 * 92 - 12 at F = 1470
    c5 = one["workloads"]["c5"]
    # (the C5 pass of this capture still counted the six-MMA loop's 90 MMAs per frame; the kernel ran the static
    # five-tile loop's 73 - bench.py was corrected after the capture, so the line's executed_frac for C5 is 23 % high)
    assert "MMAs per frame" in [k for k in c5["kernels"] if k["kernel"] == "autocorr"][0]["executed_pipe"]
    assert c5["ms_per_step"] < 1.03 * sum(k["ms"] for k in c5["kernels"])
    assert one["ms_per_step"] < 2.25 and c5["ms_per_step"] < 6.3


def test_pipelined_build_lines():
    """Capture r02t (software-pipelined autocorrelation kernel at F = 1470), 1 / 2 / 4 / 8 GPUs under torchrun: the
    device-resident value is linear in the ranks, every line follows the contract, the autocorrelation stage is faster
    than the symmetric kernel's 1.12 ms in every pass that is not the power-capped headline pass, and the 8-GPU line
    carries C4's rows gathered into one page-locked host array."""
    lines = {n: _line(os.path.join(ROOT, "profiles", f"bench_r02t_n{n}.json")) for n in (1, 2, 4, 8)}
    for n, d in lines.items():
        assert REQUIRED <= set(d), REQUIRED - set(d)
        assert d["n_gpus"] == n and d["scaling"] == "weak" and d["gpu_launches"] > 0
        assert d["value"] > 0.97 * n * lines[1]["value"]
        assert d["e2e"]["value"] > 0.9 * (lines[1]["e2e"]["value"] if n == 1 else 1.5 * lines[1]["e2e"]["value"])
        assert 0.9 <= d["copy_ceiling"]["e2e_frac_of_ceiling"] <= 1.25
        assert d["parity"]["autocorr_max_abs"] < 2e-5 and d["parity"]["mfcc_max_abs"] < 1e-4
    one = lines[1]
    assert one["ms_per_step"] < 2.12 and one["roofline"]["kernel"] == "autocorr" and one["roofline"]["ms_per_launch"] < 1.11
    assert "448 MMAs per frame" in one["roofline"]["executed"]["executed_pipe"]
    assert one["roofline"]["traffic_source"] == "profiles/ncu_traffic_r02s.json" or "r02" in one["roofline"]["traffic_source"]
    for w in ("c3", "c4"):
        ac = [k for k in one["workloads"][w]["kernels"] if k["kernel"] == "autocorr"][0]
        assert ac["ms"] < 1.08
    g = lines[8]["workloads"]["c4"]["gathered_host_array"]
    assert g["shape"] == [2994720, 256] and g["all_slices_filled"] is True
    ref = _line(os.path.join(ROOT, "profiles", "bench_r02t_ref_n1.json"))
    assert ref["impl"] == "reference" and ref["gpu_launches"] == 0 and ref["value"] == ref["cpu_baseline"]["value"]
    # capture r02u: the final build (incremental frame bookkeeping in the autocorrelation kernels)
    fin = _line(os.path.join(ROOT, "profiles", "bench_r02u_n1.json"))
    assert REQUIRED <= set(fin) and fin["n_gpus"] == 1 and fin["ms_per_step"] < 2.10 and fin["value"] > 8.5e5
    assert fin["roofline"]["traffic_source"].startswith("profiles/ncu_traffic_r02")
    assert fin["workloads"]["c5"]["ms_per_step"] < 6.0
    fref = _line(os.path.join(ROOT, "profiles", "bench_r02u_ref_n1.json"))
    assert fref["impl"] == "reference" and abs(fref["value"] / fin["cpu_baseline"]["value"] - 1.0) < 0.1


def test_weak_scaling_lines_are_consistent():
    lines = {n: _line(os.path.join(ROOT, "profiles", f"bench_r01g_n{n}.json")) for n in (1, 2, 4, 8)}
    for n, d in lines.items():
        assert d["n_gpus"] == n and d["config"]["clips_per_gpu"] == 60
        assert d["value"] > 0.95 * n * lines[1]["value"]                 # near-linear by clip, no collective


def test_bench_workload_table_and_algorithmic_counts():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    assert set(bench.WORKLOADS) == {"c2", "c3", "c4", "c5"}
    assert {n for n, w in bench.WORKLOADS.items() if w["collect"]} == {"c3", "c4"}
    # configs[2] and [4] are split over the ranks (strong), c2 / c4 carry a fixed batch per rank
    assert bench.DEFAULT_SCALING == {"c2": "weak", "c3": "strong", "c4": "weak", "c5": "strong"}
    # the math libraries are pinned before NumPy is imported by the module (children of the CPU pool inherit it)
    assert all(os.environ.get(k) == "1" for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"))
    alg = bench.algorithmic(88200, 1470, 735, 384)
    # SURVEY section 8(d): per hop-frame at 88.2 kHz
    assert alg["stft_gemm"][1] == 4327680 and alg["autocorr"][1] == 517564
    assert alg["stft_gemm"][0] == alg["autocorr"][0] == "tensor" and alg["fold"][0] == "hbm"


def _bench():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_dump_outputs_sample_is_fixed_and_bounded(tmp_path):
    """--dump-outputs keeps every row of a short output and the same seeded, ordered row sample of a long one, and the
    largest dump (C4: features + collected audio and facial rows, with their row indices) fits in 64 MB."""
    import numpy as np
    bench = _bench()
    assert np.array_equal(bench.dump_row_index(1000), np.arange(1000))
    big = bench.dump_row_index(60 * 6239)
    assert np.array_equal(big, bench.dump_row_index(60 * 6239)) and len(big) == bench.DUMP_ROWS
    assert np.all(np.diff(big) > 0) and big[-1] < 60 * 6239
    worst = bench.DUMP_ROWS * ((256 + 256 + 61) * 4 + 3 * 8)
    assert worst <= bench.DUMP_LIMIT_BYTES == 64 << 20
    bench.write_outputs(str(tmp_path / "d"), {"features": np.ones((3, 256), np.float32),
                                              "features_rows": np.arange(3.0)})
    assert sorted(os.listdir(tmp_path / "d")) == ["features.npy", "features_rows.npy"]
    with pytest.raises(AssertionError):
        bench.write_outputs(str(tmp_path / "e"), {"features_rows": np.arange(3)})          # int64: not a float dump


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_steps_rows(tmp_path):
    """bench.py --dump-outputs on C3 (features + collect_features): float arrays within 64 MB, and the sampled feature and
    collected rows are the rows a direct device call on the same synthetic inputs returns, bit for bit."""
    import subprocess
    import sys

    import numpy as np
    import torch
    out_dir = tmp_path / "dump"
    subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c3", "--steps", "2", "--warmup", "1",
                    "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                   check=True, cwd=str(tmp_path), timeout=1200, stdout=subprocess.DEVNULL)
    got = {f[:-len(".npy")]: np.load(out_dir / f) for f in os.listdir(out_dir)}
    assert set(got) == {p + s for p in ("features", "collect_audio", "collect_facial") for s in ("", "_rows")}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    bench = _bench()
    from neurosync_trainer_lite_b200 import engine, synth
    w = bench.WORKLOADS["c3"]
    packed, off, _, mine, _ = bench.make_inputs("c3", 0, 1, "strong")
    eng = engine.get_engine(w["sr"], w["F"], w["H"], device=0)
    dev = torch.device("cuda", 0)
    rows, _ = eng.extract_device(torch.from_numpy(packed).to(dev), off)
    facial = np.concatenate([synth.synth_facial(bench.FACIAL_ROWS, seed=int(i) % 6) for i in mine]).astype(np.float32)
    f_off = np.arange(len(mine) + 1, dtype=np.int64) * bench.FACIAL_ROWS
    col_a, col_f, _ = eng.collect_device(rows, eng.row_offsets(off), torch.from_numpy(facial).to(dev), f_off, **w["collect"])
    for name, full in (("features", rows), ("collect_audio", col_a), ("collect_facial", col_f)):
        idx = got[name + "_rows"].astype(np.int64)
        assert np.array_equal(idx, bench.dump_row_index(full.shape[0])), name
        np.testing.assert_array_equal(got[name], full[torch.from_numpy(idx).to(dev)].cpu().numpy(), err_msg=name)

"""The ``audio_features.csv`` feature cache formatted on the device (``nsf_format_csv_host``), against pandas.

CPU: the device's digit routine run on the host (``nsf_format_check``) equals Python's ``repr`` on random float64 bit
patterns, float32-exact doubles and edge cases; ``nsf_csv_bytes_bound`` covers the longest fields.
GPU: ``Engine.format_csv`` text equals ``pd.DataFrame(rows.astype(np.float64)).to_csv(index=False)`` byte for byte
(ragged file batches, both dtypes, pageable and page-locked buffers, many small groups), and the dataset builders
write exactly the files the pandas writer wrote, with the same examples and messages.
"""
import contextlib
import io
import os
import shutil
import subprocess
import sys

import numpy as np
import pandas as pd
import pytest

from neurosync_trainer_lite_b200 import synth


@pytest.fixture(scope="module")
def nv():
    import __graft_entry__ as g
    g.build_library()
    from neurosync_trainer_lite_b200 import _native
    return _native


def _check(nv, values):
    """nsf_format_check of float64 values -> list of str."""
    v = np.ascontiguousarray(values, dtype=np.float64)
    out = np.zeros(32 * max(len(v), 1), dtype=np.uint8)
    lengths = np.zeros(max(len(v), 1), dtype=np.int32)
    nv.check(nv.lib.nsf_format_check(v.ctypes.data_as(nv._f64p), len(v), nv.ptr(out), lengths.ctypes.data_as(nv._i32p)))
    rows = out.reshape(-1, 32)
    return [rows[i, :lengths[i]].tobytes().decode() for i in range(len(v))]


def _repr(x):
    return "" if x != x else repr(x)


def _assert_repr(nv, values):
    values = np.asarray(values, dtype=np.float64)
    got = _check(nv, values)
    bad = [(v, g) for v, g in zip(values.tolist(), got) if g != _repr(v)]
    assert not bad, bad[:10]


def _random_bits(n, seed):
    return np.random.default_rng(seed).integers(0, 2 ** 64, size=n, dtype=np.uint64).view(np.float64)


def _float32_exact(n, seed):
    bits = np.random.default_rng(seed).integers(0, 2 ** 32, size=n, dtype=np.uint64).astype(np.uint32)
    with np.errstate(invalid="ignore"):
        return bits.view(np.float32).astype(np.float64)


def _edge_values():
    v = [0.0, -0.0, 0.1, -0.1, 123.0, 0.00015, 1e-4, 1e-5, 1e16, -1e16, 9999999999999998.0, 5e-324, -5e-324,
         2.2250738585072014e-308, 2.225073858507201e-308, 1.7976931348623157e308, -1.2345678901234568e+17,
         float(np.float32(0.1)), 1.0, 0.5, 1e22, 1e23, 9007199254740993.0, np.inf, -np.inf, np.nan]
    v += [2.0 ** e for e in range(-1074, 1024)] + [-(2.0 ** e) for e in range(-1074, 1024, 7)]
    v += [float(f"1e{e}") for e in range(-323, 309)]
    v += [float(2 ** 53 + k) for k in range(-64, 65)] + [float(k) for k in range(-1000, 1000)]
    for edge in (1e-4, 1e16):       # both sides of the switch between positional and scientific notation
        x = edge
        for _ in range(20):
            x = np.nextafter(x, 0.0)
            v.append(x)
        x = edge
        for _ in range(20):
            x = np.nextafter(x, np.inf)
            v.append(x)
    return np.array(v, dtype=np.float64)


def test_digits_equal_repr_on_random_bit_patterns(nv):
    """Both signs, every exponent (NaN and inf patterns included), plus subnormals drawn on their own."""
    _assert_repr(nv, _random_bits(1_000_000, 1))
    sub = np.random.default_rng(2).integers(1, 2 ** 52, size=50_000, dtype=np.uint64)
    sub |= np.random.default_rng(3).integers(0, 2, size=sub.size, dtype=np.uint64) << np.uint64(63)
    _assert_repr(nv, sub.view(np.float64))


def test_digits_equal_repr_on_float32_exact_doubles(nv):
    _assert_repr(nv, _float32_exact(500_000, 4))
    _assert_repr(nv, np.random.default_rng(5).standard_normal(200_000).astype(np.float32).astype(np.float64))


def test_digits_equal_repr_on_edge_cases(nv):
    _assert_repr(nv, _edge_values())
    assert _check(nv, [1e-5, 1e16, 5e-324, -0.0, 9999999999999998.0, np.float32(0.1), np.nan, -np.inf]) == [
        "1e-05", "1e+16", "5e-324", "-0.0", "9999999999999998.0", "0.10000000149011612", "", "-inf"]


def _longest_field():
    """A double whose repr has the 24 characters of the widest field (sign, 17 digits, point, e-3xx)."""
    for v in _random_bits(10_000, 6):
        if np.isfinite(v) and len(repr(float(v))) == 24:
            return float(v)
    raise AssertionError("no 24-character value drawn")


def test_bytes_bound_covers_the_longest_fields(nv):
    v = _longest_field()
    for rows, cols in [(3, 1), (0, 256), (7, 256), (2, 1234)]:
        text = pd.DataFrame(np.full((rows, cols), v)).to_csv(index=False)
        assert nv.lib.nsf_csv_bytes_bound(rows, cols, 1) >= len(text)
    assert nv.lib.nsf_csv_bytes_bound(12, 1, 1) >= len(pd.DataFrame(np.full((12, 1), np.nan)).to_csv(index=False))
    assert nv.lib.nsf_csv_bytes_bound(3 + 7, 256, 2) >= sum(
        len(pd.DataFrame(np.full((r, 256), v)).to_csv(index=False)) for r in (3, 7))
    assert nv.lib.nsf_csv_bytes_bound(1, 0, 1) == -1 and nv.lib.nsf_csv_bytes_bound(-1, 4, 1) == -1
    assert nv.lib.nsf_csv_bytes_bound(1, 4, -1) == -1


def test_format_check_rejects_bad_arguments(nv):
    out = np.zeros(32, np.uint8)
    lengths = np.zeros(1, np.int32)
    v = np.zeros(1)
    assert nv.lib.nsf_format_check(None, 1, nv.ptr(out), lengths.ctypes.data_as(nv._i32p)) == nv.ERR_BAD_ARG
    assert nv.lib.nsf_format_check(v.ctypes.data_as(nv._f64p), -1, nv.ptr(out),
                                   lengths.ctypes.data_as(nv._i32p)) == nv.ERR_BAD_ARG


# ---- on the device ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng(nv):
    if nv.lib.nsf_device_count() < 1:
        pytest.fail("GPU tests need an sm_100 device (the library has no CPU path)")
    from neurosync_trainer_lite_b200 import engine
    return engine.get_engine(88200, *engine.frame_params(88200))


def _pandas_text(rows):
    return pd.DataFrame(np.asarray(rows).astype(np.float64)).to_csv(index=False).encode()


def _value_rows():
    """The random sets of the CPU tests (NaN / inf bit patterns included) as rows of 256, 7 and 1 columns."""
    v = np.concatenate([_random_bits(200_000, 11), _float32_exact(100_000, 12), _edge_values()])
    v = v[:len(v) // 256 * 256]
    return [v.reshape(-1, 256), v[:7 * 3000].reshape(-1, 7), v[:5000].reshape(-1, 1)]


@pytest.mark.gpu
def test_format_csv_equals_pandas(eng):
    for rows in _value_rows():
        text, off = eng.format_csv(rows)
        assert list(off) == [0, len(text)]
        assert text.tobytes() == _pandas_text(rows)
    one = np.array([[np.nan], [1.5], [np.nan], [-np.inf]])      # a lone NaN field is written ""
    assert eng.format_csv(one)[0].tobytes() == _pandas_text(one) == b'0\n""\n1.5\n""\n-inf\n'
    assert eng.format_csv(np.zeros((0, 3)))[0].tobytes() == b"0,1,2\n"


def _ragged(dtype, seed):
    rng = np.random.default_rng(seed)
    counts = [37, 0, 1801, 5, 0, 912, 1]
    rows = (rng.standard_normal((sum(counts), 256)) * 10.0 ** rng.integers(-7, 18, size=(sum(counts), 256)))
    rows[rng.random(rows.shape) < 1e-3] = np.nan
    rows[rng.random(rows.shape) < 1e-3] = -np.inf
    return rows.astype(dtype), np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)


def _assert_files(text, t_off, rows, r_off):
    assert t_off[0] == 0 and len(t_off) == len(r_off)
    for i in range(len(r_off) - 1):
        assert text[t_off[i]:t_off[i + 1]].tobytes() == _pandas_text(rows[r_off[i]:r_off[i + 1]]), i


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_ragged_batches_into_pageable_and_page_locked_text(eng, nv, dtype):
    from neurosync_trainer_lite_b200 import engine
    rows, r_off = _ragged(dtype, 21)
    text, t_off = eng.format_csv(rows, r_off)
    _assert_files(text, t_off, rows, r_off)
    # a sub-range of the files (row_offsets not starting at 0)
    sub, s_off = eng.format_csv(rows, r_off[2:6])
    _assert_files(sub, s_off, rows[r_off[2]:], r_off[2:6] - r_off[2])
    # page-locked rows and text through the C ABI
    bound = nv.lib.nsf_csv_bytes_bound(int(r_off[-1]), 256, len(r_off) - 1)
    rows_buf = engine.PinnedBuffer(rows.nbytes)
    pinned_rows = rows_buf.view(dtype, rows.shape)
    pinned_rows[...] = rows
    text_buf = engine.PinnedBuffer(bound)
    pinned_text = text_buf.view(np.uint8, (bound,))
    t_off2 = np.empty(len(r_off), np.int64)
    nv.check(nv.lib.nsf_format_csv_host(eng.handle, nv.F64 if dtype == np.float64 else nv.F32, nv.ptr(pinned_rows),
                                        256, r_off.ctypes.data_as(nv._i64p), len(r_off) - 1, nv.ptr(pinned_text),
                                        bound, t_off2.ctypes.data_as(nv._i64p)))
    assert np.array_equal(t_off2, t_off)
    assert pinned_text[:t_off[-1]].tobytes() == text.tobytes()


def _small_group_run():
    """Texts of the ragged batches (both dtypes) with a 1 Mi-value group budget: every file its own group or nearly."""
    from neurosync_trainer_lite_b200 import engine
    e = engine.get_engine(88200, *engine.frame_params(88200))
    out = {}
    for name, dtype in (("f32", np.float32), ("f64", np.float64)):
        rows, r_off = _ragged(dtype, 31)
        big = np.concatenate([rows] * 6)
        b_off = np.concatenate([r_off[:-1] + k * r_off[-1] for k in range(6)] + [[6 * r_off[-1]]])
        out[name], out[name + "_off"] = e.format_csv(big, b_off)
    return out


@pytest.mark.gpu
def test_results_do_not_depend_on_the_grouping(eng, tmp_path):
    """NSF_GROUP_MI=NSF_FIRST_MI=1 (read once per process, hence the child): about twenty groups over the three slots
    instead of two."""
    here = os.path.dirname(os.path.abspath(__file__))
    out = tmp_path / "small_groups.npz"
    code = ("import sys, numpy as np; sys.path[:0] = [%r, %r]\n"
            "import test_csv_cache as t\n"
            "np.savez(%r, **t._small_group_run())\n" % (os.path.dirname(here), here, str(out)))
    subprocess.run([sys.executable, "-c", code], check=True, timeout=900,
                   env=dict(os.environ, NSF_GROUP_MI="1", NSF_FIRST_MI="1"))
    small = np.load(out)
    default = _small_group_run()
    for name in ("f32", "f64"):
        assert np.array_equal(small[name + "_off"], default[name + "_off"])
        assert small[name].tobytes() == default[name].tobytes()
        rows, r_off = _ragged(np.float32 if name == "f32" else np.float64, 31)
        _assert_files(default[name][:default[name + "_off"][len(r_off) - 1]], default[name + "_off"][:len(r_off)],
                      rows, r_off)


@pytest.mark.gpu
def test_bad_arguments_raise_and_launch_nothing(eng, nv):
    rows = np.ones((4, 3))
    text = np.empty(1000, np.uint8)
    t_off = np.empty(3, np.int64)
    launches = eng.launch_count()

    def call(dtype=nv.F64, rows_p=nv.ptr(rows), cols=3, r_off=(0, 2, 4), n=2, text_p=nv.ptr(text), cap=1000):
        off = np.array(r_off, np.int64)
        return nv.lib.nsf_format_csv_host(eng.handle, dtype, rows_p, cols, off.ctypes.data_as(nv._i64p), n, text_p,
                                          cap, t_off.ctypes.data_as(nv._i64p))
    assert call() == nv.OK
    launches = eng.launch_count()
    assert call(dtype=7) == nv.ERR_BAD_ARG
    assert call(rows_p=None) == nv.ERR_BAD_ARG
    assert call(text_p=None) == nv.ERR_BAD_ARG
    assert call(cols=0) == nv.ERR_BAD_ARG
    assert call(r_off=(0, 3, 2)) == nv.ERR_BAD_ARG
    assert call(n=-1) == nv.ERR_BAD_ARG
    assert call(cap=nv.lib.nsf_csv_bytes_bound(4, 3, 2) - 1) == nv.ERR_BAD_ARG
    assert eng.launch_count() == launches
    with pytest.raises(ValueError):
        eng.format_csv(np.ones(5))
    with pytest.raises(ValueError):
        eng.format_csv(rows, [0, 5])
    with pytest.raises(nv.NsfError):
        eng.format_csv(rows, [0, 3, 2, 4])
    assert eng.launch_count() == launches


# ---- dataset builders ----------------------------------------------------------------------------------
def _pandas_writer(cache_csv, rows, cache_format, text=None):
    """The writer the builders used before the device formatter: the reference's to_csv (and the .npy)."""
    if cache_format in ("csv", "both"):
        pd.DataFrame(np.asarray(rows, dtype=np.float64)).to_csv(cache_csv, index=False)
        print(f"Audio features saved to {cache_csv}")
    if cache_format in ("npy", "both"):
        npy_path = os.path.splitext(cache_csv)[0] + ".npy"
        np.save(npy_path, np.asarray(rows, dtype=np.float32))
        print(f"Audio features saved to {npy_path}")


def _take_tree(root):
    cols = ["Timecode", "BlendshapeCount"] + [f"bs{i}" for i in range(61)]
    for k, (secs, rows) in enumerate([(2.0, 118), (3.1, 190), (1.4, 80), (4.2, 250)]):
        take = root / f"take_{k:03d}"
        take.mkdir(parents=True)
        y = synth.synth_clip(secs, 88200, seed=60 + k, kind=("voiced", "gated", "noise", "voiced")[k])
        (take / "audio.wav").write_bytes(synth.wav_bytes(synth.to_int16_pcm(0.8 * y), 88200))
        pd.DataFrame(np.hstack([np.zeros((rows, 2)), synth.synth_facial(rows, seed=k)]),
                     columns=cols).to_csv(take / f"t{k}_iPhone_cal.csv", index=False)


def _run(fn, root, *args, **kw):
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        result = fn(str(root), *args, **kw)
    return result, sorted(buf.getvalue().replace(str(root), "<root>").splitlines())


def _assert_examples(a, b):
    assert len(a) == len(b)
    for (xa, fa), (xb, fb) in zip(a, b):
        assert xa.dtype == xb.dtype and np.array_equal(xa, xb) and np.array_equal(fa, fb)


@pytest.mark.gpu
@pytest.mark.parametrize("cache_format", ["csv", "both"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_load_data_writes_the_pandas_csv(eng, tmp_path, monkeypatch, cache_format, dtype):
    from neurosync_trainer_lite_b200.dataset import data_processing as dp
    _take_tree(tmp_path / "src")
    shutil.copytree(tmp_path / "src", tmp_path / "dev")
    with monkeypatch.context() as m:
        m.setattr(dp, "_write_feature_cache", _pandas_writer)
        (want, want_idx), want_msgs = _run(dp.load_data_batched, tmp_path / "src", 88200, set(),
                                           cache_format=cache_format, dtype=dtype)
    (got, got_idx), got_msgs = _run(dp.load_data_batched, tmp_path / "dev", 88200, set(), cache_format=cache_format,
                                    dtype=dtype)
    assert got_idx == want_idx and got_msgs == want_msgs
    assert sum("Audio features saved to" in s and s.endswith(".csv") for s in got_msgs) == 4
    _assert_examples(got, want)
    for k in range(4):
        take = f"take_{k:03d}"
        csv = (tmp_path / "dev" / take / "audio_features.csv").read_bytes()
        assert csv == (tmp_path / "src" / take / "audio_features.csv").read_bytes(), take
        if cache_format == "both":
            assert csv == _pandas_text(np.load(tmp_path / "dev" / take / "audio_features.npy"))
    # a second load reads the caches and returns what it returns over the pandas-written tree
    (again, _), again_msgs = _run(dp.load_data_batched, tmp_path / "dev", 88200, set(), cache_format=cache_format,
                                  dtype=dtype)
    (again_ref, _), _ = _run(dp.load_data_batched, tmp_path / "src", 88200, set(), cache_format=cache_format,
                             dtype=dtype)
    assert sum(s.startswith("Loading audio features from") for s in again_msgs) == 4
    _assert_examples(again, again_ref)


@pytest.mark.gpu
def test_collect_features_writes_the_pandas_csv(eng, tmp_path, monkeypatch):
    from neurosync_trainer_lite_b200.dataset import data_processing as dp
    _take_tree(tmp_path / "src")
    shutil.copytree(tmp_path / "src", tmp_path / "dev")

    def collect(root):
        take = os.path.join(root, "take_001")
        return dp.collect_features(os.path.join(take, "audio.wav"), os.path.join(take, "audio_features.csv"),
                                   os.path.join(take, "t1_iPhone_cal.csv"), 88200)
    with monkeypatch.context() as m:
        m.setattr(dp, "_write_feature_cache", _pandas_writer)
        want, want_msgs = _run(collect, tmp_path / "src")
    got, got_msgs = _run(collect, tmp_path / "dev")
    assert got_msgs == want_msgs and "Audio features saved to <root>/take_001/audio_features.csv" in got_msgs
    _assert_examples([got], [want])
    csv = (tmp_path / "dev" / "take_001" / "audio_features.csv").read_bytes()
    assert csv == (tmp_path / "src" / "take_001" / "audio_features.csv").read_bytes()
    from neurosync_trainer_lite_b200.utils.audio.extraction.extract_features import extract_audio_features
    assert csv == _pandas_text(extract_audio_features(str(tmp_path / "dev" / "take_001" / "audio.wav"), 88200)[0])
    again, again_msgs = _run(collect, tmp_path / "dev")       # the cache is read back
    assert again_msgs == ["Loading audio features from <root>/take_001/audio_features.csv"]
    _assert_examples([again], [_run(collect, tmp_path / "src")[0]])

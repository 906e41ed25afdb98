"""CSV text parsed on the device (``nsf_csv_row_offsets`` / ``nsf_csv_parse``), against pandas.

CPU: the device's field routine run on the host (``nsf_parse_check``) gives, bit for bit, the double ``pd.read_csv``
reads for over a million generated strings, classifies integer literals as pandas types them, reads back every string
``nsf_format_check`` writes and rejects what lies outside its grammar.
GPU: ``Engine.parse_csv`` equals ``pd.read_csv(path).drop(columns=DROP).values`` cast to float32 / float64 on ragged
batches of LiveLink-shaped facial files, feature caches and edge-case files, reports unaccepted files with the right
status bit, and ``load_data_batched`` gives what the pandas readers give.
"""
import contextlib
import io
import shutil

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


def _check(nv, strings):
    """nsf_parse_check of str fields -> (values float64, kinds int32)."""
    raw = [s.encode() for s in strings]
    text = np.frombuffer(b"".join(raw) or b"\0", dtype=np.uint8)
    off = np.zeros(len(raw) + 1, dtype=np.int64)
    np.cumsum([len(b) for b in raw], out=off[1:])
    values = np.zeros(max(len(raw), 1), dtype=np.float64)
    kinds = np.zeros(max(len(raw), 1), dtype=np.int32)
    nv.check(nv.lib.nsf_parse_check(nv.ptr(text), off.ctypes.data_as(nv._i64p), len(raw),
                                    values.ctypes.data_as(nv._f64p), kinds.ctypes.data_as(nv._i32p)))
    return values[:len(raw)], kinds[:len(raw)]


def _pandas_floats(strings):
    """What pd.read_csv reads for each string in a float64 column (one that also holds 0.5)."""
    text = "x\n0.5\n" + "\n".join(strings) + "\n"
    col = pd.read_csv(io.StringIO(text))["x"]
    assert col.dtype == np.float64
    return col.values[1:]


def _assert_pandas(nv, strings, min_accepted=0.99):
    values, kinds = _check(nv, strings)
    ok = kinds != nv.CSV_KIND_BAD
    assert ok.mean() >= min_accepted, [s for s, k in zip(strings, ok) if not k][:10]
    acc = [s for s, k in zip(strings, ok) if k]
    want = _pandas_floats(acc)
    got = values[ok]
    bad = np.flatnonzero(got.view(np.uint64) != want.view(np.uint64))
    assert bad.size == 0, [(acc[i], got[i], want[i]) for i in bad[:10]]
    return int(ok.sum())


def _random_bits(n, seed):
    v = np.random.default_rng(seed).integers(0, 2 ** 64, size=n, dtype=np.uint64).view(np.float64)
    return v[np.isfinite(v)]


def _strings(seed):
    """About 1.05 M strings in the forms a CSV file hands pandas' float parser."""
    rng = np.random.default_rng(seed)
    out = [repr(float(x)) for x in _random_bits(300_000, seed)]                                   # repr of any double
    f32 = rng.integers(0, 2 ** 32, size=150_000, dtype=np.uint64).astype(np.uint32).view(np.float32)
    out += [repr(float(x)) for x in f32[np.isfinite(f32)]]                                         # widened float32
    mags = rng.standard_normal(300_000) * 10.0 ** rng.integers(-12, 14, size=300_000)
    prec = rng.integers(0, 21, size=300_000)
    out += ["%.*f" % (int(p), m) for p, m in zip(prec[:100_000], mags[:100_000])]
    out += ["%.*e" % (int(p), m) for p, m in zip(prec[100_000:200_000], mags[100_000:200_000])]
    out += ["%.17g" % m for m in mags[200_000:]]
    digits = rng.integers(0, 10, size=(100_000, 25))
    lens = rng.integers(18, 26, size=100_000)
    points = rng.integers(0, 26, size=100_000)
    exps = rng.integers(-330, 300, size=100_000)
    for d, n, p, e in zip(digits, lens, points, exps):                                            # 18-25 digit mantissas
        s = "".join(map(str, d[:n]))
        if p < n:
            s = s[:p] + "." + s[p:]
        out.append(s + ("e%d" % e if e % 3 else ""))
    small = rng.integers(0, 10 ** 6, size=100_000)
    for k, v in enumerate(small):                                                                 # leading zeros, 1., .5
        form = k % 5
        out.append(("000" + str(v)) if form == 0 else (str(v) + ".") if form == 1 else ("." + str(v)) if form == 2
                   else ("-00%d.%d" % (v, k)) if form == 3 else ("+%d.%de-%02d" % (v % 10, v, k % 40)))
    ex = rng.integers(1, 10, size=100_000)
    ee = rng.integers(-320, 309, size=100_000)
    out += ["%de%+03d" % (a, b) for a, b in zip(ex, ee)]                                            # 1e-05 style
    out += ["4.9e-324", "5e-324", "1e-320", "2.2250738585072014e-308", "2.225073858507201e-308",
            "1.7976931348623157e308", "1.7976931348623157e+308", "-1.7976931348623157e308", "1e308", "1e-308",
            "1e-616", "1e-700", "0.0000000000000000000000000001", "123456789012345678901234e-10", "-0.0", "0e5"]
    return out


def test_parse_check_equals_pandas_on_a_million_strings(nv):
    strings = _strings(5)
    accepted = 0
    for k in range(0, len(strings), 250_000):   # one chunk of pandas' reader per file
        accepted += _assert_pandas(nv, strings[k:k + 250_000], min_accepted=0.95)
    assert accepted >= 1_000_000


def test_parse_check_reads_back_what_format_check_writes(nv):
    from test_csv_cache import _check as format_check, _edge_values, _float32_exact
    vals = np.concatenate([_random_bits(200_000, 7), _float32_exact(100_000, 8), _edge_values()])
    vals = vals[np.isfinite(vals)]
    strings = format_check(nv, vals)
    assert _assert_pandas(nv, strings, min_accepted=1.0) == len(strings)
    values, kinds = _check(nv, ["inf", "-inf", ""])
    assert list(kinds) == [nv.CSV_KIND_INF, nv.CSV_KIND_INF, nv.CSV_KIND_EMPTY]
    assert values[0] == np.inf and values[1] == -np.inf and np.isnan(values[2])


def test_integer_literals_are_classified_as_pandas_types_them(nv):
    literals = ["0", "-0", "+5", "000123", "123456789012345", "-999999999999999", "7"]
    others = ["1.", ".5", "1e5", "1.0", "-0.0", "0e0"]
    _, kinds = _check(nv, literals + others)
    assert list(kinds) == [nv.CSV_KIND_INTEGER] * len(literals) + [nv.CSV_KIND_NUMBER] * len(others)
    for s, k in zip(literals + others, kinds):
        col = pd.read_csv(io.StringIO(f"x\n{s}\n{s}\n"))["x"]
        assert (col.dtype == np.int64) == (k == nv.CSV_KIND_INTEGER), s
    # -0: +0 in an all-integer column, -0.0 in a column that also holds a non-integer (within one chunk)
    assert not np.signbit(pd.read_csv(io.StringIO("x\n-0\n1\n")).values.astype(np.float64)[0, 0])
    assert np.signbit(pd.read_csv(io.StringIO("x\n-0\n0.5\n")).values[0, 0])
    values, _ = _check(nv, ["-0"])
    assert np.signbit(values[0])   # the field routine's double; the integer-column rule is the kernels'


def test_fixed_list_is_unaccepted(nv):
    bad = [" 1.5", "1.5 ", "NaN", "nan", "NA", "null", "1e", "1e+", "1e400", "0e309", "\"1\"", "-", ".", "+", "e5",
           "1234567890123456", "-0000000000000001", "1.5\r", "1,5", "1..5", "0x10", "Infinity", "+inf", "1" * 41,
           "1é", "1_0"]
    _, kinds = _check(nv, bad)
    assert all(k == nv.CSV_KIND_BAD for k in kinds), [(s, k) for s, k in zip(bad, kinds) if k != nv.CSV_KIND_BAD]


def test_parse_check_rejects_bad_arguments(nv):
    text = np.frombuffer(b"1.5", dtype=np.uint8)
    off = np.array([0, 3], np.int64)
    v = np.zeros(1)
    k = np.zeros(1, np.int32)
    args = [nv.ptr(text), off.ctypes.data_as(nv._i64p), 1, v.ctypes.data_as(nv._f64p), k.ctypes.data_as(nv._i32p)]
    assert nv.lib.nsf_parse_check(*args) == nv.OK and v[0] == 1.5 and k[0] == nv.CSV_KIND_NUMBER
    for i in (0, 1, 3, 4):
        a = list(args)
        a[i] = None
        assert nv.lib.nsf_parse_check(*a) == nv.ERR_BAD_ARG
    assert nv.lib.nsf_parse_check(*args[:2], -1, *args[3:]) == nv.ERR_BAD_ARG
    dec = np.array([2, 1], np.int64)
    assert nv.lib.nsf_parse_check(args[0], dec.ctypes.data_as(nv._i64p), 1, *args[3:]) == nv.ERR_BAD_ARG


# ---- on the device ---------------------------------------------------------------------------------------
DROP = ["Timecode", "BlendshapeCount"]


@pytest.fixture(scope="module")
def eng(nv):
    if nv.lib.nsf_device_count() < 1:
        pytest.fail("GPU tests need an sm_100 device (the library has no CPU path)")
    from neurosync_trainer_lite_b200 import engine
    return engine.get_engine(88200, *engine.frame_params(88200))


def _livelink(rows, seed, crlf=False, final_newline=True):
    """A LiveLink Face-shaped facial CSV: Timecode strings, an integer BlendshapeCount, 61 columns of decimals."""
    rng = np.random.default_rng(seed)
    names = ["Timecode", "BlendshapeCount"] + [f"Blend{i}" for i in range(61)]
    vals = rng.uniform(-0.2, 1.0, size=(rows, 61)) * (rng.random((rows, 61)) < 0.95)
    prec = rng.integers(6, 9, size=(rows, 61))
    lines = [",".join(names)]
    for r in range(rows):
        tc = "10:%02d:%02d:%02d.%03d" % (r // 3600 % 60, r // 60 % 60, r % 60, r % 1000)
        lines.append(",".join([tc, "61"] + ["%.*f" % (int(p), v) if v else "0" for p, v in zip(prec[r], vals[r])]))
    nl = "\r\n" if crlf else "\n"
    return (nl.join(lines) + (nl if final_newline else "")).encode()


def _pack(files):
    off = np.zeros(len(files) + 1, dtype=np.int64)
    np.cumsum([len(f) for f in files], out=off[1:])
    return np.frombuffer(b"".join(files) or b"\0", dtype=np.uint8)[:int(off[-1])], off


def _want(data, drop, dtype):
    return np.ascontiguousarray(pd.read_csv(io.BytesIO(data)).drop(columns=drop).values, dtype=dtype)


def _parse(eng, files, drop, dtype):
    names = files[0].split(b"\n", 1)[0].rstrip(b"\r").decode().split(",")
    kept = [n for n in names if n not in drop]
    out_col = [-1 if n in drop else kept.index(n) for n in names]
    text, off = _pack(files)
    return eng.parse_csv(text, off, len(names), out_col, dtype)


def _assert_equal(rows, r_off, status, files, drop, dtype, skip=()):
    for i, f in enumerate(files):
        if i in skip:
            continue
        assert status[i] == 0, (i, status[i])
        want = _want(f, drop, dtype)
        got = rows[r_off[i]:r_off[i + 1]]
        assert got.shape == want.shape, (i, got.shape, want.shape)
        iv = np.uint64 if dtype == np.float64 else np.uint32
        assert np.array_equal(got.view(iv), want.view(iv)), i


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_facial_batches_equal_pandas(eng, dtype):
    files = [_livelink(n, seed=k, crlf=k % 3 == 1, final_newline=k % 4 != 2)
             for k, n in enumerate([1800, 7, 0, 1, 930, 2400, 64])]
    rows, r_off, status = _parse(eng, files, DROP, dtype)
    assert rows.dtype == dtype and rows.shape[1] == 61
    _assert_equal(rows, r_off, status, files, DROP, dtype)


def _cache_rows(seed, n):
    rng = np.random.default_rng(seed)
    rows = rng.standard_normal((n, 256)) * 10.0 ** rng.integers(-9, 12, size=(n, 256))
    rows[rng.random(rows.shape) < 2e-3] = np.nan
    rows[rng.random(rows.shape) < 1e-3] = np.inf
    rows[rng.random(rows.shape) < 1e-3] = -np.inf
    rows[rng.random(rows.shape) < 1e-3] = -0.0
    return rows


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_feature_caches_equal_pandas(eng, dtype):
    files = []
    for k, (n, src) in enumerate([(1800, np.float64), (3, np.float32), (0, np.float64), (2500, np.float32)]):
        text, _ = eng.format_csv(_cache_rows(k, n).astype(src))
        files.append(text.tobytes())
    rows, r_off, status = _parse(eng, files, [], dtype)
    _assert_equal(rows, r_off, status, files, [], dtype)


_EDGE = [
    b"a,b,c\r\n1.5,-0,2\r\n\r\n-3,-0,4\r\n",               # CRLF, a blank line, an all-integer column with -0
    b"a,b,c\n1,2,3\n\n\n4,5,6",                          # blank lines, no final newline
    b"a,b,c\n",                                          # header only
    b"a,b,c",                                            # header only, no newline
    b"a,b,c\n,,\n1e-05,.5,1.\n-inf,inf,\n",              # empty fields, spellings of the writer
    b"a,b,c\n000000000000000012.5,1e-400,4.9e-324\n",
]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_edge_files_equal_pandas(eng, dtype):
    rows, r_off, status = _parse(eng, _EDGE, [], dtype)
    _assert_equal(rows, r_off, status, _EDGE, [], dtype)
    assert not np.signbit(rows[r_off[0]:r_off[1], 1]).any()


_BAD = [
    (b'a,b\n1,"2"\n', 0x4),           # quoted field
    (b"a,b\n1,2\r3,4\n", 0x4),        # bare \r
    (b"a,b\n1,2,3\n", 0x2),           # extra field
    (b"a,b\n1\n", 0x2),               # missing field
    (b"a,b\n1,NaN\n", 0x1),           # NA spelling
    (b"a,b\n1,1234567890123456\n", 0x8),   # 16-digit integer
    (b"a,b\n-0,1\n0.5,2\n", 0x8),     # -0 in a mixed column
]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_unaccepted_files_are_reported(eng, nv, dtype):
    good = [b"a,b\n1.25,-2\n3,4.5\n", b"a,b\n7,8\n"]
    files = [good[0]] + [f for f, _ in _BAD] + [good[1]]
    rows, r_off, status = _parse(eng, files, [], dtype)
    for k, (_, bit) in enumerate(_BAD):
        assert status[k + 1] & bit, (k, status[k + 1])
    _assert_equal(rows, r_off, status, files, [], dtype, skip=range(1, len(_BAD) + 1))
    # a dropped column is not parsed, but a quote in it still changes the tokenisation
    d_rows, _, d_status = _parse(eng, [b"a,b\nx y,1\n", b'a,b\n"x",1\n'], ["a"], dtype)
    assert d_status[0] == 0 and d_rows[0, 0] == 1 and d_status[1] & nv.CSV_BAD_LINE


@pytest.mark.gpu
def test_bad_arguments_launch_nothing(eng, nv):
    import torch
    text = torch.zeros(64, dtype=torch.uint8, device="cuda")
    text[:8] = torch.tensor(list(b"a,b\n1,2\n"), dtype=torch.uint8)
    out = torch.empty((4, 2), dtype=torch.float64, device="cuda")
    st = torch.empty(4, dtype=torch.int32, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    import ctypes as C
    launches = eng.launch_count()

    def parse(dtype=nv.F64, text_p=text.data_ptr(), t_off=(0, 8), cols=2, out_col=(0, 1), out_cols=2,
              r_off=(0, 1), out_ld=2, status=st.data_ptr(), n=None):
        t = np.array(t_off, np.int64)
        oc = np.array(out_col, np.int32)
        r = np.array(r_off, np.int64)
        return nv.lib.nsf_csv_parse(eng.handle, C.c_void_p(s), dtype, C.c_void_p(text_p), t.ctypes.data_as(nv._i64p),
                                    len(t) - 1 if n is None else n, cols, oc.ctypes.data_as(nv._i32p), out_cols,
                                    r.ctypes.data_as(nv._i64p), C.c_void_p(out.data_ptr()), out_ld,
                                    C.c_void_p(status))
    assert parse(dtype=7) == nv.ERR_BAD_ARG
    assert parse(text_p=0) == nv.ERR_BAD_ARG
    assert parse(text_p=text.data_ptr() + 1) == nv.ERR_BAD_ARG
    assert parse(t_off=(0, 8, 4)) == nv.ERR_BAD_ARG
    assert parse(n=-1) == nv.ERR_BAD_ARG
    assert parse(cols=0, out_col=()) == nv.ERR_BAD_ARG
    assert parse(out_col=(0, 2)) == nv.ERR_BAD_ARG
    assert parse(out_col=(1, 1)) == nv.ERR_BAD_ARG
    assert parse(out_col=(-2, 1)) == nv.ERR_BAD_ARG
    assert parse(out_ld=1) == nv.ERR_BAD_ARG
    assert parse(r_off=(1, 2)) == nv.ERR_BAD_ARG
    assert parse(status=0) == nv.ERR_BAD_ARG
    assert parse(t_off=(0,), r_off=(0,)) == nv.OK           # n_files == 0
    t = np.array([0], np.int64)
    r = np.zeros(1, np.int64)
    assert nv.lib.nsf_csv_row_offsets(eng.handle, C.c_void_p(s), C.c_void_p(text.data_ptr()),
                                      t.ctypes.data_as(nv._i64p), 0, r.ctypes.data_as(nv._i64p)) == nv.OK
    assert nv.lib.nsf_csv_row_offsets(eng.handle, C.c_void_p(s), C.c_void_p(text.data_ptr()),
                                      t.ctypes.data_as(nv._i64p), -1, r.ctypes.data_as(nv._i64p)) == nv.ERR_BAD_ARG
    assert eng.launch_count() == launches
    assert parse() == nv.OK
    torch.cuda.synchronize()
    assert out[0].tolist() == [1.0, 2.0] and st[0].item() == 0
    with pytest.raises(ValueError):
        eng.parse_csv(np.zeros(4, np.uint8), [0, 5], 1, [0])
    with pytest.raises(ValueError):
        eng.parse_csv(np.zeros(4, np.uint8), [0, 4], 2, [0])


# ---- dataset builder ----------------------------------------------------------------------------------
def _pandas_parse(eng, pool, paths, text, off, drop, dtype):
    """The readers before the device parser: pandas, one file at a time."""
    from neurosync_trainer_lite_b200.dataset import data_processing as dp
    return [dp._pandas_rows(p, drop, dtype) for p in paths]


def _take_tree(root, bad_take=1):
    for k, (secs, rows) in enumerate([(2.0, 118), (3.1, 190), (1.4, 80), (4.2, 250)]):
        take = root / f"take_{k:03d}"
        take.mkdir(parents=True)
        y = synth.synth_clip(secs, 88200, seed=80 + k, kind=("voiced", "gated", "noise", "voiced")[k])
        (take / "audio.wav").write_bytes(synth.wav_bytes(synth.to_int16_pcm(0.8 * y), 88200))
        data = _livelink(rows, seed=k, crlf=k == 2)
        if k == bad_take:   # outside the device grammar: a quoted Timecode, which pandas reads
            data = data.replace(b"\n10:00:00:00.000,", b'\n"10:00:00:00.000",', 1)
        (take / f"t{k}_iPhone_cal.csv").write_bytes(data)


def _run(fn, root, *args, **kw):
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        result = fn(str(root), *args, **kw)
    return result, sorted(buf.getvalue().replace(str(root), "<root>").splitlines())


def _assert_examples(a, b):
    assert len(a) == len(b)
    for (xa, fa), (xb, fb) in zip(a, b):
        assert xa.dtype == xb.dtype and np.array_equal(xa, xb) and np.array_equal(fa, fb)
        assert np.array_equal(xa.view(np.uint8), xb.view(np.uint8)) and np.array_equal(fa.view(np.uint8), fb.view(np.uint8))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_load_data_equals_the_pandas_readers(eng, tmp_path, monkeypatch, dtype):
    from neurosync_trainer_lite_b200.dataset import data_processing as dp
    _take_tree(tmp_path / "src")
    assert pd.read_csv(tmp_path / "src" / "take_001" / "t1_iPhone_cal.csv")["Timecode"][0] == "10:00:00:00.000"
    shutil.copytree(tmp_path / "src", tmp_path / "dev")
    for second in (False, True):   # first load: facial CSVs; second: the audio_features.csv caches too
        with monkeypatch.context() as m:
            m.setattr(dp, "_parse_csvs", _pandas_parse)
            (want, want_idx), want_msgs = _run(dp.load_data_batched, tmp_path / "src", 88200, set(), dtype=dtype)
        (got, got_idx), got_msgs = _run(dp.load_data_batched, tmp_path / "dev", 88200, set(), dtype=dtype)
        assert "parse_csv" in dp.last_timing and "facial_csv_wait" in dp.last_timing
        assert got_idx == want_idx == [0, 1, 2, 3] and got_msgs == want_msgs
        assert sum(s.startswith("Loading audio features from") for s in got_msgs) == (4 if second else 0)
        _assert_examples(got, want)


@pytest.mark.gpu
def test_missing_timecode_raises_the_pandas_key_error(eng, tmp_path, monkeypatch):
    from neurosync_trainer_lite_b200.dataset import data_processing as dp
    _take_tree(tmp_path, bad_take=-1)
    f = tmp_path / "take_002" / "t2_iPhone_cal.csv"
    df = pd.read_csv(f)
    df.drop(columns=["Timecode"]).to_csv(f, index=False)
    with pytest.raises(KeyError) as got:
        _run(dp.load_data_batched, tmp_path, 88200, set())
    with monkeypatch.context() as m:
        m.setattr(dp, "_parse_csvs", _pandas_parse)
        with pytest.raises(KeyError) as want:
            _run(dp.load_data_batched, tmp_path, 88200, set())
    assert str(got.value) == str(want.value)

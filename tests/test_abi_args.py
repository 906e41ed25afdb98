"""Argument rejection of the older C ABI entries: a bad argument returns its status before anything is queued.

Every case calls the entry directly and checks three things: the status code, that no kernel was launched
(``nsf_launch_count`` is unchanged), and that the outputs, filled with a sentinel, are untouched.  Each entry is also
called once with good arguments, so that a rejection is due to the one argument the case changes.
"""
import ctypes as C

import numpy as np
import pytest


@pytest.fixture(scope="module")
def nv():
    import __graft_entry__ as g
    g.build_library()
    from neurosync_trainer_lite_b200 import _native
    return _native


@pytest.fixture(scope="module")
def eng(nv):
    if nv.lib.nsf_device_count() < 1:
        pytest.fail("GPU tests need an sm_100 device (the library has no CPU path)")
    from neurosync_trainer_lite_b200 import engine
    return engine.get_engine(88200, *engine.frame_params(88200))


SENTINEL = 7.25


def _snapshot(outputs):
    return [o.copy() if isinstance(o, np.ndarray) else o.cpu().clone() for o in outputs]


def _rejects(nv, eng, status, call, *outputs):
    """call() returns `status`, launches nothing and leaves every output (host array or CUDA tensor) as it was."""
    import torch
    before = _snapshot(outputs)
    launches = eng.launch_count()
    got = call()
    torch.cuda.synchronize()
    assert got == status, (got, status, nv.last_error())
    assert eng.launch_count() == launches
    for after, b in zip(_snapshot(outputs), before):
        assert np.array_equal(after, b), "a rejected call wrote into an output"


def _i64(values):
    return np.ascontiguousarray(values, dtype=np.int64)


def _p64(arr):
    return arr.ctypes.data_as(C.POINTER(C.c_int64))


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _pcm(n=88200, seed=0):
    return (np.random.default_rng(seed).standard_normal(n) * 0.1).astype(np.float32)


CLIPS = (0, 44100, 88200)
TOO_SHORT = (0, 44100, 44200)                 # 100 samples: fewer than the 9 hop-frames the deltas need


# ---- nsf_extract_batch ----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_extract_batch_rejects(nv, eng):
    import torch
    pcm = torch.from_numpy(_pcm()).cuda()
    cols = eng.plan.feature_cols(0)
    rows = int(eng.row_offsets(CLIPS)[-1])
    out = torch.full((rows + 64, cols), SENTINEL, device="cuda")
    need = eng.workspace_bytes(88200, 2, 0)
    ws = torch.zeros(2 * need, dtype=torch.uint8, device="cuda")

    def call(fmt=nv.PCM_F32, off=CLIPS, flags=0, out_ld=cols, ws_bytes=2 * need, row_off=None):
        o = _i64(off)
        r = None if row_off is None else _p64(_i64(row_off))
        return nv.lib.nsf_extract_batch(eng.handle, _stream(), C.c_void_p(pcm.data_ptr()), fmt, _p64(o), len(o) - 1,
                                        flags, C.c_void_p(out.data_ptr()), out_ld, r, None, C.c_void_p(ws.data_ptr()),
                                        ws_bytes)
    assert call() == nv.OK
    torch.cuda.synchronize()
    out.fill_(SENTINEL)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(fmt=7), out)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(out_ld=cols - 1), out)
    _rejects(nv, eng, nv.ERR_WORKSPACE, lambda: call(ws_bytes=need // 4), out)
    _rejects(nv, eng, nv.ERR_WORKSPACE, lambda: call(ws_bytes=0), out)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(off=(0, 44100, 30000)), out)
    _rejects(nv, eng, nv.ERR_TOO_SHORT, lambda: call(off=TOO_SHORT), out)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(row_off=(0, 5, rows)), out)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(flags=nv.NO_MFCC | nv.NO_AUTOCORR), out)
    _rejects(nv, eng, nv.ERR_UNSUPPORTED, lambda: call(flags=nv.AC_NO_PAD), out)


# ---- nsf_extract_host / nsf_extract_collect_host ---------------------------------------------------------------
@pytest.mark.gpu
def test_extract_host_rejects(nv, eng):
    pcm = _pcm()
    cols = eng.plan.feature_cols(0)
    rows = int(eng.row_offsets(CLIPS)[-1])
    out = np.full((rows + 64, cols), SENTINEL, np.float32)
    y = np.full(88200, SENTINEL, np.float32)

    def call(fmt=nv.PCM_F32, off=CLIPS, flags=0):
        o = _i64(off)
        return nv.lib.nsf_extract_host(eng.handle, nv.ptr(pcm), fmt, _p64(o), len(o) - 1, flags, nv.ptr(out), cols,
                                       nv.ptr(y))
    assert call() == nv.OK
    out.fill(SENTINEL)
    y.fill(SENTINEL)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(fmt=7), out, y)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(off=(0, 44100, 30000)), out, y)
    _rejects(nv, eng, nv.ERR_TOO_SHORT, lambda: call(off=TOO_SHORT), out, y)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(flags=nv.NO_MFCC | nv.NO_AUTOCORR), out, y)
    _rejects(nv, eng, nv.ERR_UNSUPPORTED, lambda: call(flags=nv.AC_NO_PAD), out, y)


@pytest.mark.gpu
def test_extract_collect_host_rejects(nv, eng):
    pcm = _pcm()
    cols = eng.plan.feature_cols(0)
    r_off = eng.row_offsets(CLIPS)
    facial = np.random.default_rng(1).standard_normal((int(r_off[-1]) + 8, 61)).astype(np.float32)
    f_off = (0, int(r_off[1]) + 4, int(r_off[-1]) + 8)
    cflags = nv.COLLECT_FAST | nv.COLLECT_BLEND
    n_out = int(eng.collect_rows(r_off, f_off, True, False, True, 30)[-1])
    out_a = np.full((n_out + 64, cols), SENTINEL, np.float32)
    out_f = np.full((n_out + 64, 61), SENTINEL, np.float32)
    feats = np.full((int(r_off[-1]) + 64, cols), SENTINEL, np.float32)

    def call(fmt=nv.PCM_F32, off=CLIPS, fo=f_off, flags=0):
        o, f = _i64(off), _i64(fo)
        return nv.lib.nsf_extract_collect_host(eng.handle, nv.ptr(pcm), fmt, _p64(o), len(o) - 1, flags, nv.ptr(facial),
                                               61, _p64(f), cflags, 30, nv.ptr(out_a), nv.ptr(out_f), nv.ptr(feats))
    assert call() == nv.OK
    for a in (out_a, out_f, feats):
        a.fill(SENTINEL)
    outs = (out_a, out_f, feats)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(fmt=7), *outs)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(off=(0, 44100, 30000)), *outs)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(fo=(0, 40, 20)), *outs)
    _rejects(nv, eng, nv.ERR_TOO_SHORT, lambda: call(off=TOO_SHORT), *outs)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(flags=nv.NO_MFCC | nv.NO_AUTOCORR), *outs)
    _rejects(nv, eng, nv.ERR_UNSUPPORTED, lambda: call(flags=nv.AC_NO_PAD), *outs)


# ---- nsf_normalize_host -------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_normalize_host_rejects(nv, eng):
    pcm = _pcm()
    y = np.full(88200, SENTINEL, np.float32)
    peaks = np.full(2, SENTINEL, np.float32)

    def call(fmt=nv.PCM_F32, off=CLIPS, y_p=nv.ptr(y)):
        o = _i64(off)
        return nv.lib.nsf_normalize_host(eng.handle, nv.ptr(pcm), fmt, _p64(o), len(o) - 1, y_p, nv.ptr(peaks))
    assert call() == nv.OK
    y.fill(SENTINEL)
    peaks.fill(SENTINEL)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(fmt=7), y, peaks)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(off=(0, 44100, 30000)), y, peaks)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(y_p=None), y, peaks)


# ---- nsf_collect_batch / nsf_collect_host -------------------------------------------------------------------------
A_OFF, F_OFF = (0, 40, 100), (0, 45, 100)
CFLAGS = 0x1 | 0x2 | 0x4          # fast, slow, blend


def _collect_inputs(eng):
    audio = np.random.default_rng(2).standard_normal((100, 256))
    facial = np.random.default_rng(3).standard_normal((100, 61))
    o_off = eng.collect_rows(A_OFF, F_OFF, True, True, True, 30)
    return audio, facial, o_off


@pytest.mark.gpu
def test_collect_batch_rejects(nv, eng):
    import torch
    audio, facial, o_off = _collect_inputs(eng)
    d_a, d_f = torch.from_numpy(audio).cuda(), torch.from_numpy(facial).cuda()
    n_out = int(o_off[-1])
    out_a = torch.full((n_out, 256), SENTINEL, dtype=torch.float64, device="cuda")
    out_f = torch.full((n_out, 61), SENTINEL, dtype=torch.float64, device="cuda")

    def call(dtype=nv.F64, a_cols=256, f_cols=61, ao=A_OFF, fo=F_OFF, oo=tuple(o_off)):
        a, f, o = _i64(ao), _i64(fo), _i64(oo)
        return nv.lib.nsf_collect_batch(eng.handle, _stream(), dtype, C.c_void_p(d_a.data_ptr()), a_cols, _p64(a),
                                        C.c_void_p(d_f.data_ptr()), f_cols, _p64(f), len(a) - 1, CFLAGS, 30,
                                        C.c_void_p(out_a.data_ptr()), C.c_void_p(out_f.data_ptr()), _p64(o))
    assert call() == nv.OK
    torch.cuda.synchronize()
    out_a.fill_(SENTINEL)
    out_f.fill_(SENTINEL)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(dtype=7), out_a, out_f)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(a_cols=0), out_a, out_f)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(f_cols=0), out_a, out_f)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(ao=(0, 40, 30)), out_a, out_f)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(fo=(0, 45, 44)), out_a, out_f)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(oo=(0, int(o_off[1]) + 1, n_out)), out_a, out_f)


@pytest.mark.gpu
def test_collect_host_rejects(nv, eng):
    audio, facial, o_off = _collect_inputs(eng)
    n_out = int(o_off[-1])
    out_a = np.full((n_out, 256), SENTINEL)
    out_f = np.full((n_out, 61), SENTINEL)

    def call(dtype=nv.F64, a_cols=256, f_cols=61, ao=A_OFF, fo=F_OFF):
        a, f = _i64(ao), _i64(fo)
        return nv.lib.nsf_collect_host(eng.handle, dtype, nv.ptr(audio), a_cols, _p64(a), nv.ptr(facial), f_cols,
                                       _p64(f), len(a) - 1, CFLAGS, 30, nv.ptr(out_a), nv.ptr(out_f))
    assert call() == nv.OK
    out_a.fill(SENTINEL)
    out_f.fill(SENTINEL)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(dtype=7), out_a, out_f)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(a_cols=0), out_a, out_f)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(f_cols=0), out_a, out_f)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(ao=(0, 40, 30)), out_a, out_f)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(fo=(0, 45, 44)), out_a, out_f)


# ---- nsf_rows_host / nsf_post_host / nsf_resample_host ------------------------------------------------------------
@pytest.mark.gpu
def test_rows_host_rejects(nv, eng):
    a = np.random.default_rng(4).standard_normal((50, 61))
    b = np.random.default_rng(5).standard_normal((40, 61))
    out = np.full((100, 61), SENTINEL)

    def call(op=nv.ROWS_BLEND_STACK, dtype=nv.F64, b_p=nv.ptr(b)):
        return nv.lib.nsf_rows_host(eng.handle, op, dtype, nv.ptr(a), 50, b_p, 40, 61, 30, nv.ptr(out))
    assert call() == nv.OK
    out.fill(SENTINEL)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(op=9), out)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(dtype=7), out)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(b_p=None), out)


@pytest.mark.gpu
def test_post_host_rejects(nv, eng):
    x = np.random.default_rng(6).standard_normal((20, 23)).astype(np.float32)
    out = np.full((20, 69), SENTINEL, np.float32)
    pf = nv.POST_EDGEFIX | nv.POST_CMVN | nv.POST_DELTAS

    def call(t=20):
        return nv.lib.nsf_post_host(eng.handle, x.ctypes.data_as(C.POINTER(C.c_float)), t, 23, pf, nv.ptr(out))
    assert call() == nv.OK
    out.fill(SENTINEL)
    _rejects(nv, eng, nv.ERR_TOO_SHORT, lambda: call(t=8), out)


@pytest.mark.gpu
def test_resample_host_rejects(nv, eng):
    pcm = _pcm(48000)
    n_out = int(nv.lib.nsf_resample_len(48000, 48000, 88200))
    out = np.full(n_out, SENTINEL, np.float32)

    def call(cap=n_out, fmt=nv.PCM_F32):
        return nv.lib.nsf_resample_host(eng.handle, nv.ptr(pcm), fmt, 48000, 48000, 88200, nv.ptr(out), cap)
    assert call() == nv.OK
    out.fill(SENTINEL)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(cap=n_out - 1), out)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(fmt=7), out)


# ---- nsf_convert_batch ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_convert_batch_rejects(nv, eng):
    import torch
    payload = torch.from_numpy((np.random.default_rng(7).standard_normal(3000) * 1000).astype(np.int16)).cuda()
    src = nv.pcm_sources([(0, 1000, nv.ENC_I16, 1, 88200), (2000, 1000, nv.ENC_I16, 2, 44100)])
    off = nv.convert_offsets(src, 88200, payload.numel() * 2)
    out = torch.full((int(off[-1]) + 16,), SENTINEL, device="cuda")

    def call(oo=tuple(off)):
        o = _i64(oo)
        return nv.lib.nsf_convert_batch(eng.handle, _stream(), C.c_void_p(payload.data_ptr()), payload.numel() * 2,
                                        nv.ptr(src), len(src), 88200, C.c_void_p(out.data_ptr()), _p64(o))
    assert call() == nv.OK
    torch.cuda.synchronize()
    out.fill_(SENTINEL)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: call(oo=(0, int(off[1]) + 1, int(off[2]) + 1)), out)


# ---- nsf_chunk_gather / nsf_chunk_blend -----------------------------------------------------------------------------
@pytest.mark.gpu
def test_chunk_calls_reject_bad_geometry(nv, eng):
    import torch
    rows = torch.randn(300, 256, device="cuda")
    chunks = torch.full((8, 64, 256), SENTINEL, device="cuda")
    blended = torch.full((300, 61), SENTINEL, device="cuda")
    decoded = torch.randn(8, 64, 61, device="cuda")

    def gather(n_rows=300, cols=256, ld=256, frame=64, overlap=16):
        return nv.lib.nsf_chunk_gather(eng.handle, _stream(), C.c_void_p(rows.data_ptr()), n_rows, cols, ld, frame,
                                       overlap, C.c_void_p(chunks.data_ptr()))

    def blend(n_rows=300, frame=64, overlap=16, scale_cols=10, divisor=100.0):
        return nv.lib.nsf_chunk_blend(eng.handle, _stream(), C.c_void_p(decoded.data_ptr()), n_rows, 61, frame, overlap,
                                      scale_cols, divisor, C.c_void_p(blended.data_ptr()))
    assert nv.lib.nsf_chunk_count(300, 64, 16) <= 8
    assert gather() == nv.OK and blend() == nv.OK
    torch.cuda.synchronize()
    chunks.fill_(SENTINEL)
    blended.fill_(SENTINEL)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: gather(overlap=64), chunks)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: gather(overlap=-1), chunks)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: gather(n_rows=0), chunks)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: gather(ld=255), chunks)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: blend(overlap=64), blended)
    _rejects(nv, eng, nv.ERR_BAD_ARG, lambda: blend(divisor=0.0), blended)
    _rejects(nv, eng, nv.ERR_UNSUPPORTED, lambda: blend(overlap=40), blended)

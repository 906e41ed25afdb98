"""The host-buffer pipeline behind nsf_extract_host, nsf_convert_host and nsf_extract_collect_host: clip groups
rotating over three slots, pageable buffers staged through pinned arenas, pitched downloads.

The results must not depend on how the clips are grouped, on whether the caller's buffers are page-locked, or on
the row pitch of the output.  The one allowed difference is in columns 0-68 (MFCC and deltas) of feature rows: at
most one float32 ulp, from the order of the float64 atomicAdds that accumulate the per-clip CMVN moments."""
import os
import subprocess
import sys

import numpy as np
import pytest

from neurosync_trainer_lite_b200 import synth

pytestmark = pytest.mark.gpu

SR = 88200
MFCC_COLS = 69
# 157 s at 88.2 kHz, 13.2 Mi samples: three groups by default (6 / 6 / 8 Mi), sixteen at NSF_GROUP_MI=NSF_FIRST_MI=1
SECONDS = [4.5, 17.0, 0.6, 12.0, 9.5, 15.5, 2.0, 13.0, 7.0, 16.0, 3.5, 11.0, 8.0, 14.5, 1.2, 10.0, 5.5, 6.0]
FACIAL_COLS = 61
# WAV takes of the conversion batch: (encoding, channels, rate, seconds); 156 s of output at 88.2 kHz
TAKES = [("i16", 2, 48000, 9.0), ("i24", 1, 44100, 12.5), ("f32", 2, 88200, 6.0), ("u8", 1, 22050, 10.0),
         ("i16", 1, 16000, 14.0), ("f32", 1, 48000, 8.0), ("i24", 2, 88200, 11.0), ("i16", 1, 44100, 7.5)] * 2


@pytest.fixture(scope="module")
def nv():
    import __graft_entry__ as g
    g.build_library()
    from neurosync_trainer_lite_b200 import _native
    if _native.lib.nsf_device_count() < 1:
        pytest.fail("GPU tests need an sm_100 device (the library has no CPU path)")
    return _native


@pytest.fixture(scope="module")
def engine(nv):
    from neurosync_trainer_lite_b200 import engine
    return engine


def _take_bytes(enc, n, seed):
    rng = np.random.default_rng(seed)
    if enc == "u8":
        return rng.integers(0, 256, n, dtype=np.uint8).tobytes()
    if enc == "i16":
        return rng.integers(-32768, 32768, n, dtype=np.int16).astype("<i2").tobytes()
    if enc == "i24":
        v = rng.integers(-(1 << 23), 1 << 23, n, dtype=np.int32).astype("<u4").view(np.uint8).reshape(-1, 4)
        return np.ascontiguousarray(v[:, :3]).tobytes()
    return rng.uniform(-1.0, 1.0, n).astype("<f4").tobytes()


def _inputs():
    """The batches every test here runs (deterministic, so a child process rebuilds the same ones)."""
    from neurosync_trainer_lite_b200 import _native as nv
    from neurosync_trainer_lite_b200 import engine
    kinds = ("voiced", "noise", "gated")
    clips = [synth.synth_clip(s, SR, seed=300 + i, kind=kinds[i % 3]) for i, s in enumerate(SECONDS)]
    y, off = engine.pack_clips(clips)
    plan = engine.get_plan(SR, *engine.frame_params(SR))
    rng = np.random.default_rng(17)
    f_rows = [int(plan.feature_rows(len(c))) + (i % 5) - 2 for i, c in enumerate(clips)]
    facial = rng.uniform(0.0, 1.0, (sum(f_rows), FACIAL_COLS)).astype(np.float32)
    f_off = np.concatenate([[0], np.cumsum(f_rows)]).astype(np.int64)
    enc = {"u8": nv.ENC_U8, "i16": nv.ENC_I16, "i24": nv.ENC_I24, "f32": nv.ENC_F32}
    payload, srcs = bytearray(), []
    for k, (e, ch, rate, s) in enumerate(TAKES):
        n = int(s * rate)
        payload += b"\x00" * (-len(payload) % 8)
        srcs.append((len(payload), n, enc[e], ch, rate))
        payload += _take_bytes(e, n * ch, seed=500 + k)
    return dict(y=y.astype(np.float32), pcm16=synth.to_int16_pcm(y), off=off, facial=facial, f_off=f_off,
                payload=np.frombuffer(bytes(payload), dtype=np.uint8).copy(), srcs=nv.pcm_sources(srcs))


def _run_all(d):
    """Every pipelined host call over the batches of _inputs(), into pageable NumPy arrays."""
    from neurosync_trainer_lite_b200 import _native as nv
    from neurosync_trainer_lite_b200 import engine
    eng = engine.get_engine(SR, *engine.frame_params(SR))
    r = {"extract_f32": eng.extract_host(d["y"], d["off"])}
    r["extract_i16"], r["y_i16"] = eng.extract_host(d["pcm16"], d["off"], nv.PEAK_NORMALIZE, want_y=True)
    r["convert"], _ = eng.convert_host(d["payload"], d["srcs"], SR)
    features = np.empty((int(eng.row_offsets(d["off"])[-1]), eng.plan.feature_cols()), np.float32)
    r["collect_audio"], r["collect_facial"], _ = eng.extract_collect_host(
        d["pcm16"], d["off"], d["facial"], d["f_off"], nv.PEAK_NORMALIZE, include_slow=True, features_out=features)
    r["features"] = features
    return r


FEATURE_ROWS = ("extract_f32", "extract_i16", "collect_audio", "features")


def _assert_same(a, b, name):
    """Bit for bit; feature rows may differ by one float32 ulp in their MFCC columns.  Returns whether they did."""
    assert a.shape == b.shape and a.dtype == b.dtype, name
    if name not in FEATURE_ROWS:
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), name
        return False
    assert np.array_equal(a[:, MFCC_COLS:].view(np.uint32), b[:, MFCC_COLS:].view(np.uint32)), name
    x, z = a[:, :MFCC_COLS], b[:, :MFCC_COLS]
    assert np.all(np.abs(x - z) <= np.spacing(np.maximum(np.abs(x), np.abs(z)))), name
    return not np.array_equal(x.view(np.uint32), z.view(np.uint32))


def test_results_do_not_depend_on_the_grouping(engine, tmp_path):
    """NSF_GROUP_MI=NSF_FIRST_MI=1 (read once per process, hence the child) splits the batches into many small groups,
    so every slot takes several groups in turn; the default budgets give three groups."""
    here = os.path.dirname(os.path.abspath(__file__))
    out = tmp_path / "small_groups.npz"
    code = ("import sys, numpy as np; sys.path[:0] = [%r, %r]\n"
            "import test_host_pipeline as t\n"
            "np.savez(%r, **t._run_all(t._inputs()))\n" % (os.path.dirname(here), here, str(out)))
    subprocess.run([sys.executable, "-c", code], check=True, timeout=900,
                   env=dict(os.environ, NSF_GROUP_MI="1", NSF_FIRST_MI="1"))
    small = np.load(out)
    default = _run_all(_inputs())
    assert sorted(small.files) == sorted(default)
    ulp = [k for k in sorted(default) if _assert_same(small[k], default[k], k)]
    print("one-ulp MFCC differences in:", ulp or "none")


def test_pitched_output(engine, nv):
    """nsf_extract_host with out_ld > cols writes each row's cols floats and leaves the rest of the row alone, into
    pageable memory (row-by-row copy-out) and page-locked memory (pitched device-to-host copy)."""
    d = _inputs()
    eng = engine.get_engine(SR, *engine.frame_params(SR))
    cols = eng.plan.feature_cols()
    want = eng.extract_host(d["y"], d["off"])
    off, off_p = nv.i64_array(d["off"])
    sentinel = np.float32(-1234.5)
    pinned = engine.PinnedBuffer(want.shape[0] * (cols + 7) * 4)
    for out in (np.empty((want.shape[0], cols + 7), np.float32), pinned.view(np.float32, (want.shape[0], cols + 7))):
        out[:] = sentinel
        nv.check(nv.lib.nsf_extract_host(eng.handle, nv.ptr(d["y"]), nv.PCM_F32, off_p, len(off) - 1, 0, nv.ptr(out),
                                         cols + 7, None))
        _assert_same(out[:, :cols].copy(), want, "extract_f32")
        assert np.all(out[:, cols:] == sentinel)


def test_pageable_and_page_locked_buffers_agree(engine, nv):
    """convert_host and extract_collect_host (every host buffer) read and write page-locked memory with the copy
    engines and pageable memory through the pinned stages: the same results."""
    d = _inputs()
    eng = engine.get_engine(SR, *engine.frame_params(SR))
    keep = []

    def pinned(shape, dtype, fill=None):
        buf = engine.PinnedBuffer(int(np.prod(shape)) * np.dtype(dtype).itemsize)
        keep.append(buf)
        arr = buf.view(dtype, shape)
        if fill is not None:
            arr[:] = fill
        return arr

    want, off = eng.convert_host(d["payload"], d["srcs"], SR)
    got, _ = eng.convert_host(pinned(d["payload"].shape, np.uint8, d["payload"]), d["srcs"], SR,
                              out=pinned((int(off[-1]),), np.float32))
    _assert_same(got, want, "convert")

    cols = eng.plan.feature_cols()
    n_rows = int(eng.row_offsets(d["off"])[-1])
    features = np.empty((n_rows, cols), np.float32)
    wa, wf, wo = eng.extract_collect_host(d["pcm16"], d["off"], d["facial"], d["f_off"], nv.PEAK_NORMALIZE,
                                          include_slow=True, features_out=features)
    pin_features = pinned((n_rows, cols), np.float32)
    ga, gf, go = eng.extract_collect_host(pinned(d["pcm16"].shape, np.int16, d["pcm16"]), d["off"],
                                          pinned(d["facial"].shape, np.float32, d["facial"]), d["f_off"],
                                          nv.PEAK_NORMALIZE, include_slow=True, out_audio=pinned(wa.shape, np.float32),
                                          out_facial=pinned(wf.shape, np.float32), features_out=pin_features)
    assert np.array_equal(go, wo)
    _assert_same(ga, wa, "collect_audio")
    _assert_same(gf, wf, "collect_facial")
    _assert_same(pin_features, features, "features")


def test_collect_on_two_streams(engine):
    """Two stream-ordered collect calls with different geometries, the first queued behind device work on its stream
    and the second issued before that work ends: each call reads its own offsets."""
    import torch
    eng = engine.get_engine(SR, *engine.frame_params(SR))
    dev = torch.device("cuda", eng.device)
    rng = np.random.default_rng(23)

    def batch(sizes, a_cols, f_cols):
        a_off = np.concatenate([[0], np.cumsum([na for na, _ in sizes])]).astype(np.int64)
        f_off = np.concatenate([[0], np.cumsum([nf for _, nf in sizes])]).astype(np.int64)
        return (rng.standard_normal((int(a_off[-1]), a_cols)).astype(np.float32), a_off,
                rng.uniform(0, 1, (int(f_off[-1]), f_cols)).astype(np.float32), f_off)

    calls = [batch([(1801, 1800), (300, 305), (64, 64)], 256, 61),
             batch([(40, 33), (500, 512), (2, 2), (97, 90), (1200, 1190)], 128, 52)]
    inputs = [(torch.from_numpy(a).to(dev), torch.from_numpy(f).to(dev)) for a, _, f, _ in calls]
    streams = [torch.cuda.Stream(dev), torch.cuda.Stream(dev)]
    torch.cuda.synchronize(dev)
    with torch.cuda.stream(streams[0]):
        torch.cuda._sleep(20_000_000)          # about 10 ms of device time ahead of the first call
    got = [eng.collect_device(ta, c[1], tf, c[3], include_slow=True, stream=s)
           for (ta, tf), c, s in zip(inputs, calls, streams)]
    torch.cuda.synchronize(dev)
    for (ga, gf, go), (a, a_off, f, f_off) in zip(got, calls):
        wa, wf, wo = eng.collect_host(a, a_off, f, f_off, include_slow=True)
        assert np.array_equal(go, wo)
        assert np.array_equal(ga.cpu().numpy(), wa) and np.array_equal(gf.cpu().numpy(), wf)

"""Batched WAV conversion (decode + downmix + resample, include/nsf.h nsf_convert_*).

The host statement of the conversion is decode_wav followed by Engine.resample_host per clip
(utils/audio/load_audio.py); the device route must reproduce it bit for bit, and the dataset builder's batched
route must give exactly what the per-take decode_for_path route gave."""
import ctypes as C
import os
import struct
from pathlib import Path

import numpy as np
import pytest

from oracle import resample_oracle as ro

ENC_BITS = {"u8": (1, 8), "i16": (1, 16), "i24": (1, 24), "i32": (1, 32), "f32": (3, 32), "f64": (3, 64)}
ENC_BYTES = {"u8": 1, "i16": 2, "i24": 3, "i32": 4, "f32": 4, "f64": 8}


@pytest.fixture(scope="module")
def nv():
    from neurosync_trainer_lite_b200 import _native
    return _native


def enc_id(nv, name):
    return {"u8": nv.ENC_U8, "i16": nv.ENC_I16, "i24": nv.ENC_I24, "i32": nv.ENC_I32, "f32": nv.ENC_F32,
            "f64": nv.ENC_F64}[name]


def samples(enc, n, seed):
    """n interleaved samples of `enc` as little-endian bytes (float ones with signed zeros and large values)."""
    rng = np.random.default_rng(seed)
    if enc == "u8":
        return rng.integers(0, 256, n, dtype=np.uint8).tobytes()
    if enc == "i16":
        return rng.integers(-32768, 32768, n, dtype=np.int16).astype("<i2").tobytes()
    if enc == "i24":
        v = rng.integers(-(1 << 23), 1 << 23, n, dtype=np.int32)
        u = v.astype("<u4").view(np.uint8).reshape(-1, 4)[:, :3]
        return np.ascontiguousarray(u).tobytes()
    if enc == "i32":
        return rng.integers(-(1 << 31), 1 << 31, n, dtype=np.int64).astype("<i4").tobytes()
    x = rng.standard_normal(n) * 0.3
    x[rng.random(n) < 0.05] = -0.0
    x[rng.random(n) < 0.01] *= 1e5
    return x.astype("<f4" if enc == "f32" else "<f8").tobytes()


def wav_file(data, enc, channels, rate, extensible=False, odd_chunk=False, declared=None):
    """RIFF/WAVE bytes: a fmt chunk (plain or WAVE_FORMAT_EXTENSIBLE), optionally an odd-sized chunk before the data
    chunk, and a data chunk whose header may declare more bytes than follow (a truncated file)."""
    code, bits = ENC_BITS[enc]
    block = channels * bits // 8
    fmt = struct.pack("<HHIIHH", 0xFFFE if extensible else code, channels, rate, rate * block, block, bits)
    if extensible:
        guid = struct.pack("<H", code) + b"\x00\x00\x00\x00\x10\x00\x80\x00\x00\xaa\x00\x38\x9b\x71"
        fmt += struct.pack("<HHI", 22, bits, 0) + guid
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt
    if odd_chunk:
        body += b"LIST" + struct.pack("<I", 5) + b"abcde" + b"\x00"
    body += b"data" + struct.pack("<I", len(data) if declared is None else declared) + data
    return b"RIFF" + struct.pack("<I", len(body)) + body


# ---- CPU ---------------------------------------------------------------------------------------------
def test_offsets_match_decode_wav_lengths(nv):
    from neurosync_trainer_lite_b200.utils.audio.load_audio import decode_wav
    clips, payload = [], b""
    rates = [44100, 48000, 88200, 16000, 22050, 8000]
    for k, enc in enumerate(ENC_BITS):
        for ch in (1, 2, 3, 6, 8, 12):
            n = 1 + (k * 37 + ch * 101) % 900
            data = samples(enc, n * ch, seed=k * 13 + ch)
            rate = rates[(k + ch) % len(rates)]
            pcm, sr = decode_wav(wav_file(data, enc, ch, rate))
            payload += b"\x00" * (-len(payload) % 8)
            clips.append(((len(payload), n, enc_id(nv, enc), ch, rate), len(pcm), sr))
            payload += data
    for target in (88200, 44100, 16000):
        off = nv.convert_offsets([c for c, _, _ in clips], target, len(payload))
        want = [n if sr == target else nv.lib.nsf_resample_len(n, sr, target) for _, n, sr in clips]
        assert list(np.diff(off)) == want and off[0] == 0


@pytest.mark.parametrize("src,payload,why", [
    ((0, 10, 6, 1, 44100), 100, "unknown encoding"),
    ((0, 10, 1, 0, 44100), 100, "channels"),
    ((0, -1, 1, 1, 44100), 100, "negative"),
    ((0, 10, 1, 1, 0), 100, "sample_rate"),
    ((0, 10, 1, 1, -5), 100, "sample_rate"),
    ((0, 51, 1, 1, 44100), 100, "past payload"),
    ((96, 1, 5, 1, 44100), 100, "past payload"),
    ((1, 10, 1, 1, 44100), 100, "aligned"),          # i16 at an odd byte
    ((2, 10, 3, 1, 44100), 100, "aligned"),          # i32 at 2 mod 4
    ((2, 2, 4, 2, 44100), 100, "aligned"),           # f32 at 2 mod 4
    ((4, 2, 5, 1, 44100), 100, "aligned"),           # f64 at 4 mod 8
])
def test_bad_descriptors_are_rejected_without_a_gpu(nv, src, payload, why):
    good = (0, 4, nv.ENC_U8, 1, 22050)
    with pytest.raises(nv.NsfError) as e:
        nv.convert_offsets([good, src], 88200, payload)
    assert e.value.status == nv.ERR_BAD_ARG and why in str(e.value) and "source 1" in str(e.value)
    out = np.empty(3, dtype=np.int64)
    arr = nv.pcm_sources([good, src])
    assert nv.lib.nsf_convert_offsets(nv.ptr(arr), 2, 88200, payload, out.ctypes.data_as(C.POINTER(C.c_int64))) == \
        nv.ERR_BAD_ARG
    with pytest.raises(nv.NsfError):
        nv.convert_offsets([good], 0, payload)
    # 8- and 24-bit samples may start anywhere
    assert list(nv.convert_offsets([(3, 5, nv.ENC_U8, 1, 88200), (5, 3, nv.ENC_I24, 2, 88200)], 88200, 100)) == \
        [0, 5, 8]


@pytest.mark.parametrize("enc", list(ENC_BITS))
@pytest.mark.parametrize("shape", ["plain", "extensible8", "odd_chunk", "truncated"])
def test_wav_source_agrees_with_decode_wav(tmp_path, enc, shape):
    from neurosync_trainer_lite_b200.dataset.data_processing import _ENC_BYTES, _wav_source
    from neurosync_trainer_lite_b200.utils.audio.load_audio import decode_wav
    ch = 8 if shape == "extensible8" else 2
    n = 301
    data = samples(enc, n * ch, seed=len(enc) + ch)
    declared = len(data) + 1000 if shape == "truncated" else None
    blob = wav_file(data, enc, ch, 48000, extensible=shape == "extensible8", odd_chunk=shape == "odd_chunk",
                    declared=declared)
    path = tmp_path / "a.wav"
    path.write_bytes(blob)
    off, nbytes, e, channels, rate = _wav_source(str(path))
    pcm, sr = decode_wav(blob)
    assert rate == sr == 48000 and channels == ch and nbytes == len(data) and blob[off:off + nbytes] == data
    assert nbytes // (_ENC_BYTES[e] * channels) == len(pcm)
    # the raw bytes decode to what decode_wav returns (host restatement of the device decode)
    assert decode_wav(wav_file(blob[off:off + nbytes], enc, ch, 48000))[0].tobytes() == pcm.tobytes()


def test_wav_source_rejects_what_decode_wav_rejects(tmp_path):
    from neurosync_trainer_lite_b200.dataset.data_processing import _wav_source
    from neurosync_trainer_lite_b200.utils.audio.load_audio import decode_wav
    blob = wav_file(b"\x00" * 12, "i16", 1, 44100).replace(struct.pack("<HHIIHH", 1, 1, 44100, 88200, 2, 16),
                                                           struct.pack("<HHIIHH", 1, 1, 44100, 88200, 2, 12))
    for b in (blob, b"RIFX" + blob[4:], blob.replace(b"data", b"date")):
        p = tmp_path / "x.wav"
        p.write_bytes(b)
        with pytest.raises(ValueError) as e1:
            decode_wav(b)
        with pytest.raises(ValueError) as e2:
            _wav_source(str(p))
        assert str(e1.value) == str(e2.value)


# ---- the dataset builder's audio route (host planning, no GPU) --------------------------------------------
PCM16_TAKES = [("i16", 1, 88200, n, False) for n in (1000, 777, 4001)]


def _wav_tree(root, specs):
    """One take folder per (enc, channels, rate, frames, extensible) holding its audio.wav; returns the paths."""
    paths = []
    for k, (enc, ch, rate, n, ext) in enumerate(specs):
        take = root / f"take_{k:03d}"
        take.mkdir(parents=True)
        (take / "audio.wav").write_bytes(wav_file(samples(enc, n * max(ch, 1), seed=k), enc, ch, rate, extensible=ext))
        paths.append(str(take / "audio.wav"))
    return paths


def _plan(paths, sr):
    from neurosync_trainer_lite_b200.dataset import data_processing as dp
    return dp._plan_audio([dp._wav_source(p) for p in paths], sr)


@pytest.mark.parametrize("extensible", [False, True])
def test_mono_pcm16_takes_at_88200_take_the_int16_route(tmp_path, nv, extensible):
    from neurosync_trainer_lite_b200.dataset import data_processing as dp
    specs = list(PCM16_TAKES)
    specs[1] = specs[1][:4] + (extensible,)
    paths = _wav_tree(tmp_path, specs)
    plan = _plan(paths, 88200)
    data_bytes = [dp._wav_source(p)[1] for p in paths]
    assert plan.int16 and plan.mid is None
    assert list(plan.lengths) == [b // 2 for b in data_bytes] == [1000, 777, 4001]
    assert list(plan.sources["byte_offset"]) == [0, 2000, 3554] and plan.nbytes == sum(data_bytes)
    assert set(plan.sources["encoding"]) == {nv.ENC_I16} and set(plan.sources["channels"]) == {1}


@pytest.mark.parametrize("enc,ch,rate", [("i16", 0, 88200), ("i16", 2, 88200), ("i16", 1, 48000), ("i24", 1, 88200),
                                         ("f32", 1, 88200), ("u8", 1, 88200)])
def test_any_other_take_sends_every_take_through_the_conversion(tmp_path, nv, enc, ch, rate):
    from neurosync_trainer_lite_b200.utils.audio.load_audio import decode_wav
    paths = _wav_tree(tmp_path, PCM16_TAKES + [(enc, ch, rate, 999, False)])
    plan = _plan(paths, 88200)
    assert not plan.int16 and plan.rate == 88200 and plan.mid is None
    assert all(plan.sources["byte_offset"] % 8 == 0) and plan.sources[-1]["channels"] == max(ch, 1)
    assert [len(decode_wav(Path(p).read_bytes())[0]) for p in paths] == list(plan.sources["frames"])
    assert list(plan.lengths) == list(np.diff(nv.convert_offsets(plan.sources, 88200, plan.nbytes)))
    # the int16 route also needs sr == 88200 (sr=None keeps the native rate in decode())
    for sr in (None, 44100):
        assert not _plan(paths[:3], sr).int16


def test_a_rate_below_88200_converts_in_two_stages(tmp_path, nv):
    paths = _wav_tree(tmp_path, PCM16_TAKES + [("i24", 2, 48000, 999, False)])
    plan = _plan(paths, 44100)
    first = nv.convert_offsets(plan.sources, 44100, plan.nbytes)
    mid = nv.pcm_sources([(int(first[k]) * 4, int(first[k + 1] - first[k]), nv.ENC_F32, 1, 44100)
                          for k in range(len(paths))])
    assert not plan.int16 and plan.rate == 44100 and np.array_equal(plan.mid, mid)
    assert list(plan.lengths) == list(np.diff(nv.convert_offsets(mid, 88200, int(first[-1]) * 4)))


def test_unsupported_encoding_is_rejected_before_anything_is_read(tmp_path):
    from concurrent.futures import ThreadPoolExecutor

    from neurosync_trainer_lite_b200.dataset import data_processing as dp
    from neurosync_trainer_lite_b200.utils.audio.load_audio import decode_wav
    paths = _wav_tree(tmp_path, PCM16_TAKES + [("i16", 1, 88200, 6, False)])
    blob = Path(paths[-1]).read_bytes().replace(struct.pack("<HHIIHH", 1, 1, 88200, 176400, 2, 16),
                                                struct.pack("<HHIIHH", 1, 1, 88200, 176400, 2, 12))
    Path(paths[-1]).write_bytes(blob)
    with pytest.raises(ValueError) as want:
        decode_wav(blob)
    queued = []
    # no engine: the header pass must fail before the length check, the reads and the jobs queued behind them
    with ThreadPoolExecutor(4) as pool, pytest.raises(ValueError) as got:
        dp._read_audio(None, pool, paths, 88200, then=lambda: queued.append(1))
    assert str(got.value) == str(want.value) and not queued


# ---- GPU ---------------------------------------------------------------------------------------------
def _engine():
    from neurosync_trainer_lite_b200 import engine
    f, h = engine.frame_params(88200)
    return engine.get_engine(88200, f, h)


def _reference(eng, blob, target, quality):
    """decode_wav + Engine.resample_host: the host route the conversion restates."""
    from neurosync_trainer_lite_b200.utils.audio.load_audio import decode_wav
    pcm, sr = decode_wav(blob)
    if sr != target:
        return eng.resample_host(pcm, sr, target, quality=quality) if len(pcm) else np.zeros(0, np.float32), pcm
    return (pcm if pcm.dtype == np.float32 else pcm.astype(np.float32) / np.float32(32768)), pcm


def _batch(nv, specs):
    """specs: (enc, channels, rate, frames, misalign) -> (payload, sources, wav blobs)."""
    payload, srcs, blobs = bytearray(), [], []
    for k, (enc, ch, rate, n, odd) in enumerate(specs):
        data = samples(enc, n * ch, seed=1000 + k)
        payload += b"\x00" * (-len(payload) % 8 + (1 if odd else 0))
        srcs.append((len(payload), n, enc_id(nv, enc), ch, rate))
        payload += data
        blobs.append(wav_file(data, enc, ch, rate))
    return np.frombuffer(bytes(payload), dtype=np.uint8), srcs, blobs


RATE_CASES = [(88200, 88200), (44100, 88200), (48000, 88200), (16000, 88200), (22050, 88200), (88200, 16000)]


@pytest.mark.gpu
@pytest.mark.parametrize("quality", ["hq", "poly"])
@pytest.mark.parametrize("orig,target", RATE_CASES)
def test_convert_host_equals_decode_then_resample(nv, quality, orig, target):
    eng = _engine()
    specs = []
    for k, enc in enumerate(ENC_BITS):
        for j, ch in enumerate((1, 2, 3, 6, 8, 12)):
            n = (1, 17, 250, 4001, 20000, 77)[(k + j) % 6]
            specs.append((enc, ch, orig, n, enc in ("u8", "i24") and j % 2 == 1))
    specs.append(("i16", 2, orig, 1 << 20, False))                 # about 1 M frames
    specs.append(("i24", 1, orig, 300001, True))
    payload, srcs, blobs = _batch(nv, specs)
    got, off = eng.convert_host(payload, srcs, target, quality=quality)
    assert got.dtype == np.float32 and len(got) == off[-1]
    for i, blob in enumerate(blobs):
        want, dec = _reference(eng, blob, target, quality)
        g = got[off[i]:off[i + 1]]
        assert np.array_equal(g.view(np.uint32), want.view(np.uint32)), (i, specs[i])
        if orig != target and len(dec) <= 50000:
            x = dec.astype(np.float32) / np.float32(32768) if dec.dtype == np.int16 else dec
            if np.all(np.isfinite(x)) and np.abs(x).max() <= 1.0:
                np.testing.assert_allclose(g, ro.resample(x.astype(np.float64), orig, target, quality=quality),
                                           rtol=0, atol=1.5e-7)


@pytest.mark.gpu
def test_convert_device_equals_host_and_feeds_extract_device(nv):
    import torch
    eng = _engine()
    specs = [("i16", 2, 48000, 40000, False), ("i24", 1, 44100, 33333, True), ("f32", 6, 88200, 30000, False),
             ("u8", 1, 22050, 12000, True), ("f64", 3, 16000, 9000, False)]
    payload, srcs, _ = _batch(nv, specs)
    want, off = eng.convert_host(payload, srcs, 88200)
    dev = torch.device("cuda", eng.device)
    got, off_d = eng.convert_device(torch.from_numpy(payload.copy()).to(dev), srcs, 88200)
    torch.cuda.synchronize()
    assert np.array_equal(off, off_d)
    assert np.array_equal(got.cpu().numpy().view(np.uint32), want.view(np.uint32))
    rows_d, _ = eng.extract_device(got, off, nv.PEAK_NORMALIZE)
    torch.cuda.synchronize()
    rows_h = eng.extract_host(want, off, nv.PEAK_NORMALIZE)
    assert np.array_equal(rows_d.cpu().numpy(), rows_h)
    # a misaligned device base is rejected on the host, before any launch
    with pytest.raises(nv.NsfError) as e:
        eng.convert_device(torch.zeros(64, dtype=torch.uint8, device=dev)[1:], [(0, 4, nv.ENC_I16, 1, 48000)], 88200)
    assert e.value.status == nv.ERR_BAD_ARG


# ---- the dataset builder on a mixed-format tree ------------------------------------------------------
MIXED = [("i16", 1, 88200, 2.1), ("i16", 2, 48000, 1.7), ("i24", 1, 44100, 2.4), ("f32", 6, 88200, 1.2),
         ("u8", 1, 22050, 1.9), ("i24x", 2, 44100, 1.5)]


def _mixed_tree(root, specs=MIXED, facial_rows=140):
    import pandas as pd
    from neurosync_trainer_lite_b200 import synth
    cols = ["Timecode", "BlendshapeCount"] + [f"bs{i}" for i in range(61)]
    for k, (enc, ch, rate, secs) in enumerate(specs):
        take = root / f"take_{k:03d}"
        take.mkdir(parents=True)
        y = np.stack([synth.synth_clip(secs, rate, seed=70 + k + c, kind=("voiced", "gated", "noise")[(k + c) % 3])
                      for c in range(ch)], axis=1) * 0.7
        e = enc.rstrip("x")
        if e == "u8":
            data = np.clip(np.rint(y * 127 + 128), 0, 255).astype(np.uint8).tobytes()
        elif e == "i16":
            data = np.clip(np.rint(y * 32767), -32768, 32767).astype("<i2").tobytes()
        elif e == "i24":
            v = np.clip(np.rint(y * 8388607), -(1 << 23), (1 << 23) - 1).astype(np.int32).reshape(-1)
            data = np.ascontiguousarray(v.astype("<u4").view(np.uint8).reshape(-1, 4)[:, :3]).tobytes()
        else:
            data = y.astype("<f4").tobytes()
        (take / "audio.wav").write_bytes(wav_file(data, e, ch, rate, extensible=enc.endswith("x")))
        pd.DataFrame(np.hstack([np.zeros((facial_rows, 2)), np.random.default_rng(k).uniform(0, 1, (facial_rows, 61))]),
                     columns=cols).to_csv(take / f"t{k}_iPhone_cal.csv", index=False)


def _old_route(root, sr, dtype):
    """The per-take route the batched builder replaced: decode_for_path per take, packed as float32, then the same
    extraction / augmentation calls load_data_batched makes."""
    from neurosync_trainer_lite_b200 import _native as nv_
    from neurosync_trainer_lite_b200.dataset import data_processing as dp
    from neurosync_trainer_lite_b200.utils.audio.load_audio import decode_for_path
    from neurosync_trainer_lite_b200.utils.video.mov_extraction import find_files
    eng = _engine()
    takes = []
    for folder in os.listdir(root):
        _, _, wav, facial_csv, _, _ = find_files(os.path.join(root, folder))
        takes.append((wav, facial_csv))
    pcm = [decode_for_path(w, sr)[0] for w, _ in takes]
    pcm = [p if p.dtype == np.float32 else p.astype(np.float32) / np.float32(32768) for p in pcm]
    off = np.concatenate([[0], np.cumsum([len(p) for p in pcm])]).astype(np.int64)
    packed = np.concatenate(pcm).astype(np.float32)
    facial = [dp._facial_rows(f, dtype) for _, f in takes]
    f_off = np.concatenate([[0], np.cumsum([len(f) for f in facial])]).astype(np.int64)
    roff = eng.row_offsets(off)
    out = []
    if dtype == np.float32:
        oa, of, o_off = eng.extract_collect_host(packed, off, np.concatenate(facial), f_off, nv_.PEAK_NORMALIZE)
        for k in range(len(takes)):
            out.append((oa[o_off[k]:o_off[k + 1]], of[o_off[k]:o_off[k + 1]].copy()))
    else:
        rows = eng.extract_host(packed, off, nv_.PEAK_NORMALIZE).astype(np.float64)
        oa, of, o_off = eng.collect_host(rows, roff, np.concatenate(facial), f_off)
        for k in range(len(takes)):
            out.append((oa[o_off[k]:o_off[k + 1]], of[o_off[k]:o_off[k + 1]].copy()))
    for _, f in out:
        f[:, :61] *= 100
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("sr", [88200, 44100])
def test_mixed_format_dataset_equals_the_per_take_route(tmp_path, sr):
    from neurosync_trainer_lite_b200.dataset import data_processing as dp
    for name, dtype in (("a", np.float32), ("b", np.float64)):
        root = tmp_path / name
        _mixed_tree(root)
        want = _old_route(str(root), sr, dtype)
        if dtype == np.float32:
            got = dp.load_data(str(root), sr, set())
        else:
            got, _ = dp.load_data_batched(str(root), sr, set(), dtype=np.float64)
        assert len(got) == len(want) == len(MIXED)
        for (ga, gf), (wa, wf) in zip(got, want):
            assert ga.dtype == wa.dtype == dtype
            assert np.array_equal(ga, wa) and np.array_equal(gf, wf)
        assert all((root / f"take_{k:03d}" / "audio_features.csv").exists() for k in range(len(MIXED)))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_extensible_pcm16_dataset_equals_the_plain_one(tmp_path, dtype):
    """WAVE_FORMAT_EXTENSIBLE mono PCM16 takes at 88.2 kHz go the int16 route like plain ones: same examples, same
    cache files, bit for bit."""
    from neurosync_trainer_lite_b200.dataset import data_processing as dp
    out = []
    for enc in ("i16", "i16x"):
        root = tmp_path / enc
        _mixed_tree(root, [(enc, 1, 88200, secs) for secs in (2.1, 1.3, 1.8)])
        got, _ = dp.load_data_batched(str(root), 88200, set(), cache_format="both", dtype=dtype)
        caches = [(root / take / name).read_bytes() for take in sorted(os.listdir(root))
                  for name in ("audio_features.csv", "audio_features.npy")]
        out.append((got, caches))
    (want, want_caches), (got, got_caches) = out
    assert len(got) == len(want) == 3 and got_caches == want_caches
    for (ga, gf), (wa, wf) in zip(got, want):
        assert ga.dtype == wa.dtype == dtype
        assert ga.tobytes() == wa.tobytes() and gf.tobytes() == wf.tobytes()


@pytest.mark.gpu
def test_mixed_format_dataset_errors(tmp_path):
    import pandas as pd
    from neurosync_trainer_lite_b200.dataset import data_processing as dp
    cols = ["Timecode", "BlendshapeCount"] + [f"bs{i}" for i in range(61)]
    bad = tmp_path / "bad" / "take_000"
    bad.mkdir(parents=True)
    blob = wav_file(b"\x00" * 4000, "i16", 2, 48000).replace(struct.pack("<HHIIHH", 1, 2, 48000, 192000, 4, 16),
                                                             struct.pack("<HHIIHH", 3, 2, 48000, 192000, 4, 16))
    (bad / "audio.wav").write_bytes(blob)                                   # IEEE float, 16 bit: unsupported
    pd.DataFrame(np.zeros((10, 63)), columns=cols).to_csv(bad / "s_iPhone_cal.csv", index=False)
    with pytest.raises(ValueError):
        dp.load_data(str(tmp_path / "bad"), 88200, set())
    short = tmp_path / "short" / "take_000"
    short.mkdir(parents=True)
    (short / "audio.wav").write_bytes(wav_file(samples("i16", 2 * 2000, 1), "i16", 2, 44100))
    pd.DataFrame(np.zeros((10, 63)), columns=cols).to_csv(short / "s_iPhone_cal.csv", index=False)
    with pytest.raises(TypeError):
        dp.load_data(str(tmp_path / "short"), 88200, set())

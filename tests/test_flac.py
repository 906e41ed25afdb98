"""FLAC input (include/nsf.h nsf_flac_*, utils/audio/load_audio.py decode_flac / flac_layout).

Decoding is lossless, so the contract is exact: a FLAC stream decodes to what decode_wav returns for the WAV file
holding the same samples.  The CPU tests pin the frame decoder through nsf_flac_check (the device code compiled for
the host) against the oracle's independent Python decoder, over streams the oracle's encoder writes with every
coding feature forced; the GPU tests run the device route end to end."""
import ctypes as C
import io
import mmap

import numpy as np
import pytest

from oracle import flac_oracle as fo

RIFF_MESSAGE = "not a RIFF/WAVE stream (only WAV decoding is built in)"


@pytest.fixture(scope="module")
def nv():
    from neurosync_trainer_lite_b200 import _native
    return _native


@pytest.fixture(scope="module")
def la():
    from neurosync_trainer_lite_b200.utils.audio import load_audio
    return load_audio


def signal(n, channels, bits, seed, wasted=0):
    """Band-limited noise plus a tone, full scale of `bits` bits, multiples of 2^wasted."""
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    top = (1 << (bits - 1)) - 1
    cols = []
    for c in range(channels):
        x = 0.6 * np.sin(t * (0.01 + 0.003 * c)) + 0.2 * np.convolve(rng.standard_normal(n), np.ones(5) / 5, "same")
        cols.append(np.clip(np.round(x * top), -top - 1, top).astype(np.int64))
    x = np.stack(cols, axis=1)
    return (x >> wasted) << wasted


# every coding feature: (name, encode kwargs, channels, bits, wasted)
FEATURES = [
    ("verbatim", dict(sub=fo.Sub("verbatim")), 1, 16, 0),
    ("constant", dict(sub=fo.Sub("constant")), 1, 16, 0),
    ("fixed0", dict(sub=fo.Sub("fixed", 0)), 1, 16, 0),
    ("fixed1", dict(sub=fo.Sub("fixed", 1)), 2, 8, 0),
    ("fixed2", dict(sub=fo.Sub("fixed", 2)), 2, 16, 0),
    ("fixed3", dict(sub=fo.Sub("fixed", 3)), 1, 24, 0),
    ("fixed4", dict(sub=fo.Sub("fixed", 4)), 3, 16, 0),
    ("lpc1", dict(sub=fo.Sub("lpc", 1)), 1, 16, 0),
    ("lpc8_p15", dict(sub=fo.Sub("lpc", 8, precision=15)), 2, 24, 0),
    ("lpc32", dict(sub=fo.Sub("lpc", 32, precision=12)), 1, 16, 0),
    ("lpc12_shift0", dict(sub=fo.Sub("lpc", 12, precision=5, shift=0)), 1, 16, 0),
    ("rice5_po4", dict(sub=fo.Sub("fixed", 2, method=1, porder=4)), 1, 24, 0),
    ("rice4_po0", dict(sub=fo.Sub("lpc", 4, porder=0)), 1, 16, 0),
    ("escape", dict(sub=fo.Sub("fixed", 2, porder=3, escape=(0, 3, 5))), 1, 16, 0),
    ("escape_w0", dict(sub=fo.Sub("fixed", 1, porder=1, escape=(0, 1))), 1, 8, 0),
    ("escape_w31", dict(sub=fo.Sub("fixed", 1, method=1, porder=2, escape=(1,), escape_width=31)), 1, 24, 0),
    ("wasted3", dict(sub=fo.Sub("lpc", 6, wasted=3)), 2, 16, 3),
    ("wasted_verbatim", dict(sub=fo.Sub("verbatim", wasted=7)), 1, 24, 7),
    ("left_side", dict(stereo="left_side", sub=fo.Sub("lpc", 8)), 2, 16, 0),
    ("side_right", dict(stereo="side_right", sub=fo.Sub("fixed", 2)), 2, 24, 0),
    ("mid_side", dict(stereo="mid_side", sub=fo.Sub("lpc", 10)), 2, 16, 0),
    ("mid_side_8bit", dict(stereo="mid_side", sub=fo.Sub("verbatim")), 2, 8, 0),
    ("variable", dict(variable=True, blocks=[1, 200, 4608, 17, 3000, 1],
                      sub=lambda i: fo.Sub("fixed", 2) if i in (1, 2, 4) else fo.Sub("verbatim")), 2, 16, 0),
    ("odd_blocks", dict(blocks=[192, 576, 255, 256, 4097, 65535, 100]), 1, 16, 0),
    ("eight_channels", dict(block=1152), 8, 16, 0),
    ("explicit_rate_khz", dict(header=dict(rate_code=12)), 1, 16, 0),
    ("streaminfo_codes", dict(header=dict(rate_code=0, size_code=0)), 1, 16, 0),
    ("metadata", dict(metadata=[(1, bytes(100)), (2, b"appl" + bytes(9)), (3, bytes(18 * 2)),
                                (4, bytes(40)), (5, bytes(396 + 36)), (6, bytes(32))]), 1, 16, 0),
]
RATES = {"explicit_rate_khz": 32000}


def feature_stream(name):
    kw, ch, bits, wasted = next((k, c, b, w) for n, k, c, b, w in FEATURES if n == name)
    kw = dict(kw)
    n = sum(kw["blocks"]) if "blocks" in kw else 3 * 4096 + 512      # a last block forced partition orders divide
    x = signal(n, ch, bits, seed=len(name), wasted=wasted)
    if name in ("constant", "escape_w0"):
        x = np.full((n, ch), x[0, 0], np.int64)
    rate = RATES.get(name, 44100)
    if "block" not in kw and "blocks" not in kw:
        kw["block"] = 4096
    return x, rate, bits, fo.encode(x, rate, bits, **kw)


def source(nv, data, pos, end, ch, bits, rate, max_block=65535):
    return np.array([(pos, end - pos, 1, ch, bits, rate, max_block)], dtype=nv.FLAC_SOURCE)


# ---- CPU -----------------------------------------------------------------------------------------------------
def test_crc_check_values():
    assert fo.crc8(b"123456789") == 0xF4        # CRC-8/SMBUS
    assert fo.crc16(b"123456789") == 0xFEE8     # CRC-16/UMTS


@pytest.mark.parametrize("name", [f[0] for f in FEATURES])
def test_oracle_round_trip(name):
    x, rate, bits, data = feature_stream(name)
    y, r, b, _ = fo.decode(data)
    assert r == rate and b == bits
    np.testing.assert_array_equal(y, x)


@pytest.mark.parametrize("name", [f[0] for f in FEATURES])
def test_flac_check_agrees_with_the_oracle_frame_by_frame(nv, la, name):
    x, rate, bits, data = feature_stream(name)
    lay = la.flac_layout(io.BytesIO(data))
    assert (lay.channels, lay.rate, lay.bits, lay.frames) == (x.shape[1], rate, bits, len(x))
    _, _, _, frames = fo.decode(data)
    end = len(data)
    for start, f in frames:
        rec, samples = nv.flac_check(data, source(nv, data, start, end, lay.channels, bits, rate, lay.max_block))
        assert int(rec["status"]) == nv.FLAC_OK, (start, int(rec["status"]))
        assert (int(rec["end"]), int(rec["number"]), int(rec["block"]), int(rec["assignment"]), int(rec["channels"]),
                int(rec["variable"]), int(rec["bits"]), int(rec["sample_rate"])) == \
            (f["end"], f["number"], f["block"], f["assignment"], f["channels"], f["variable"], f["bits"], f["rate"])
        assert rec["crc8_ok"] == 1 and rec["crc16_ok"] == 1
        np.testing.assert_array_equal(samples.T, f["samples"])


def guarded(data):
    """data placed so that its last byte is the last readable byte before a PROT_NONE page: a read past the end
    of the data faults instead of passing unnoticed.  Returns (keep-alive, address of the data)."""
    page = mmap.PAGESIZE
    size = (len(data) + page - 1) // page * page
    mm = mmap.mmap(-1, size + page)
    base = C.addressof(C.c_char.from_buffer(mm))
    libc = C.CDLL(None, use_errno=True)
    libc.mprotect.argtypes = [C.c_void_p, C.c_size_t, C.c_int]
    assert libc.mprotect(C.c_void_p(base + size), page, 0) == 0
    mm[size - len(data):size] = data
    return mm, base + size - len(data)


@pytest.mark.parametrize("name", ["verbatim", "fixed2", "lpc32", "rice5_po4", "escape", "wasted3", "mid_side",
                                  "variable", "odd_blocks", "eight_channels", "streaminfo_codes"])
def test_flac_check_reports_corruption_without_reading_out_of_range(nv, la, name):
    x, rate, bits, data = feature_stream(name)
    lay = la.flac_layout(io.BytesIO(data))
    _, _, _, frames = fo.decode(data)
    rng = np.random.default_rng(7)
    frame_out = np.zeros(1, dtype=nv.FLAC_FRAME)
    samples = np.zeros(lay.channels * 65536, np.int32)
    for start, f in frames[:3]:
        whole = data[start:f["end"]]
        cases = [whole[:n] for n in sorted(set(rng.integers(0, len(whole), 12).tolist()))]   # truncations
        for pos in rng.integers(0, len(whole), 24).tolist():                                    # byte flips
            b = bytearray(whole)
            b[pos] ^= int(rng.integers(1, 256))
            cases.append(bytes(b))
        for i, case in enumerate(cases):
            if not case:
                continue
            keep, addr = guarded(case)
            src = source(nv, case, 0, len(case), lay.channels, bits, rate, lay.max_block)
            nv.check(nv.lib.nsf_flac_check(C.c_void_p(addr), nv.ptr(src), nv.ptr(frame_out),
                                           samples.ctypes.data_as(nv._i32p), samples.size))
            status = int(frame_out[0]["status"])
            # a truncated frame, or any one corrupted byte (the CRC-16 catches every burst of up to 16 bits)
            assert status != nv.FLAC_OK, (start, i)
            del keep


def test_flac_layout_accepts_metadata_arrangements(la):
    x = signal(3000, 2, 16, 1)
    for meta in ([], [(1, bytes(0))], [(4, b"x" * 70), (1, bytes(8192))], [(6, bytes(300000)), (3, bytes(18))],
                 [(2, b"abcd"), (5, bytes(432)), (126, b"??")]):
        data = fo.encode(x, 48000, 16, block=1024, metadata=meta)
        lay = la.flac_layout(io.BytesIO(data))
        assert (lay.channels, lay.rate, lay.bits, lay.frames, lay.max_block) == (2, 48000, 16, 3000, 1024)
        assert lay.data_offset + lay.data_bytes == len(data)
        assert data[lay.data_offset:lay.data_offset + 2] == b"\xff\xf8"


def _with_streaminfo(data, **fields):
    """data with its STREAMINFO re-written (fields of fo.streaminfo)."""
    info = int.from_bytes(data[8:26], "big")
    si = dict(min_block=info >> 128, max_block=(info >> 112) & 0xFFFF, rate=(info >> 44) & 0xFFFFF,
              channels=((info >> 41) & 7) + 1, bits=((info >> 36) & 31) + 1, total=info & ((1 << 36) - 1))
    si.update(fields)
    return data[:8] + fo.streaminfo(si["rate"], si["channels"], si["bits"], si["total"], si["min_block"],
                                     si["max_block"]) + data[42:]


@pytest.mark.parametrize("case, message", [
    ("bps12", "bits per sample 12"), ("bps20", "bits per sample 20"), ("bps32", "bits per sample 32"),
    ("total0", "total samples is 0"), ("no_streaminfo", "STREAMINFO is not the first"),
    ("streaminfo_second", "STREAMINFO is not the first"), ("two_streaminfo", "more than one STREAMINFO"),
    ("ogg", "Ogg"), ("id3", "ID3v2"), ("not_flac", "not a FLAC stream"), ("type127", "type 127"),
    ("truncated_block", "truncated FLAC metadata block"), ("no_frames", "no frame data"),
])
def test_flac_layout_rejects(la, case, message):
    x = signal(2000, 1, 16, 2)
    good = fo.encode(x, 44100, 16, block=1024)
    si_block = good[4:42]
    data = {
        "bps12": _with_streaminfo(good, bits=12), "bps20": _with_streaminfo(good, bits=20),
        "bps32": _with_streaminfo(good, bits=32), "total0": _with_streaminfo(good, total=0),
        "no_streaminfo": b"fLaC" + fo.metadata_block(1, bytes(4), True) + good[42:],
        "streaminfo_second": b"fLaC" + fo.metadata_block(1, bytes(4), False) + si_block + good[42:],
        "two_streaminfo": b"fLaC" + bytes([0]) + si_block[1:] + si_block + good[42:],
        "ogg": b"OggS" + good, "id3": b"ID3\x04\x00\x00\x00\x00\x00\x00" + good, "not_flac": b"RIFF" + good[4:],
        "type127": b"fLaC" + bytes([0]) + si_block[1:] + fo.metadata_block(127, b"", True) + good[42:],
        "truncated_block": good[:30], "no_frames": good[:42],
    }[case]
    with pytest.raises(ValueError, match=message):
        la.flac_layout(io.BytesIO(data))


@pytest.mark.parametrize("data", [b"", b"RIFX....", b"ID3\x04" + bytes(40), b"OggS" + bytes(40), b"fLa", b"fLaX"])
def test_decode_of_non_flac_bytes_raises_the_wav_message(la, data):
    with pytest.raises(ValueError) as e:
        la.decode(data, None)
    assert str(e.value) == RIFF_MESSAGE


# ---- GPU -----------------------------------------------------------------------------------------------------
def same_decode(la, flac, wav):
    a, sr_a = la.decode(flac, None)
    b, sr_b = la.decode(wav, None)
    assert sr_a == sr_b and a.dtype == b.dtype and a.shape == b.shape
    assert a.tobytes() == b.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("bits", [8, 16, 24])
@pytest.mark.parametrize("channels", range(1, 9))
def test_decode_flac_equals_decode_wav(la, bits, channels):
    x = signal(20000 + 37 * channels, channels, bits, seed=bits * 10 + channels)
    sub = (lambda i: [fo.Sub("verbatim"), fo.Sub("fixed", 3), fo.Sub("lpc", 12)][i % 3])
    data = fo.encode(x, 22050, bits, block=4608, sub=sub)
    same_decode(la, data, fo.wav_bytes(x, 22050, bits))


@pytest.mark.gpu
@pytest.mark.parametrize("bits", [8, 16, 24])
@pytest.mark.parametrize("stereo", list(fo.STEREO))
def test_decode_flac_stereo_modes(la, bits, stereo):
    x = signal(30000, 2, bits, seed=bits)
    x[:, 1] = np.clip(-x[:, 0] + x[:, 1] // 4, -(1 << (bits - 1)), (1 << (bits - 1)) - 1)   # wide side channel
    data = fo.encode(x, 48000, bits, block=4096, stereo=stereo, sub=lambda i: fo.Sub("lpc", 1 + 7 * i % 32))
    same_decode(la, data, fo.wav_bytes(x, 48000, bits))


@pytest.mark.gpu
@pytest.mark.parametrize("name", [f[0] for f in FEATURES])
def test_decode_flac_every_feature(la, name):
    x, rate, bits, data = feature_stream(name)
    same_decode(la, data, fo.wav_bytes(x, rate, bits))


@pytest.mark.gpu
@pytest.mark.parametrize("rate", [88200, 44100])
def test_extract_audio_features_flac_equals_wav(tmp_path, rate):
    from neurosync_trainer_lite_b200.utils.audio.extraction.extract_features import extract_audio_features
    x = signal(rate * 2, 2, 16, seed=rate)
    flac = fo.encode(x, rate, 16, stereo="mid_side", sub=fo.Sub("lpc", 8))
    wav = fo.wav_bytes(x, rate, 16)
    (tmp_path / "take.flac").write_bytes(flac)
    (tmp_path / "take.wav").write_bytes(wav)
    for a, b in [(extract_audio_features(str(tmp_path / "take.flac")), extract_audio_features(str(tmp_path / "take.wav"))),
                 (extract_audio_features(flac, from_bytes=True), extract_audio_features(wav, from_bytes=True))]:
        assert a[0].tobytes() == b[0].tobytes() and a[1].tobytes() == b[1].tobytes()


def planted(copies):
    """A mono 16-bit stream whose middle VERBATIM frame holds `copies` complete valid frames (header CRC-8 and frame
    CRC-16 right) as sample bytes: false syncs that parse cleanly and must stay off the frame chain."""
    fake = fo.encode_frame(np.full((16, 1), 1234, np.int64), 16, 44100, 1)
    fake += bytes(len(fake) & 1)
    vals = np.frombuffer(fake * copies, dtype=">i2").astype(np.int64)
    x = signal(3 * 4096, 1, 16, seed=3)
    x[4096:4096 + len(vals), 0] = vals
    sub = lambda i: fo.Sub("verbatim") if i == 1 else fo.Sub("lpc", 8)
    return x, fo.encode(x, 44100, 16, block=4096, sub=sub)


@pytest.mark.gpu
@pytest.mark.parametrize("copies", [1, 64])
def test_planted_false_sync_is_skipped(la, copies):
    x, data = planted(copies)            # 64 copies outgrow the first candidate table: the scan runs again
    same_decode(la, data, fo.wav_bytes(x, 44100, 16))


@pytest.mark.gpu
def test_corrupt_streams_raise_naming_the_frame(la):
    x = signal(4 * 4096, 2, 16, seed=5)
    good = fo.encode(x, 44100, 16, block=4096, sub=fo.Sub("lpc", 8))
    _, _, _, frames = fo.decode(good)
    start2, f2 = frames[2]
    bad = bytearray(good)
    bad[f2["end"] - 1] ^= 0x10           # the stored CRC-16 itself: the frame parses, its checksum disagrees
    with pytest.raises(ValueError, match=f"frame at byte {start2}: frame CRC-16 mismatch"):
        la.decode(bytes(bad), None)
    with pytest.raises(ValueError, match=f"frame at byte {frames[3][0]}: truncated frame"):
        la.decode(good[:frames[3][0] + 100], None)
    with pytest.raises(ValueError, match=f"frame at byte {frames[0][0]}: bits per sample disagree with STREAMINFO"):
        la.decode(_with_streaminfo(good, bits=24), None)
    with pytest.raises(ValueError, match=f"frame at byte {frames[0][0]}: channel count disagrees with STREAMINFO"):
        la.decode(_with_streaminfo(good, channels=1), None)
    with pytest.raises(ValueError, match=f"frame at byte {frames[3][0]}: frame runs past the STREAMINFO total"):
        la.decode(_with_streaminfo(good, total=3 * 4096 + 5), None)
    with pytest.raises(ValueError, match=f"frame at byte {f2['end']}: header CRC-8 mismatch"):
        b = bytearray(good)
        b[f2["end"] + 2] ^= 0x01
        la.decode(bytes(b), None)


@pytest.mark.gpu
def test_batch_spans_pipeline_groups():
    from neurosync_trainer_lite_b200 import _native as nv
    from neurosync_trainer_lite_b200 import engine
    from neurosync_trainer_lite_b200.utils.audio import load_audio as la
    x = signal(30 * 44100, 2, 16, seed=11)
    one = fo.encode(x, 44100, 16, stereo="left_side", sub=fo.Sub("fixed", 2))
    lay = la.flac_layout(io.BytesIO(one))
    payload = np.frombuffer(one * 60, dtype=np.uint8)
    src = np.array([(k * len(one) + lay.data_offset, lay.data_bytes, lay.frames, 2, 16, 44100, lay.max_block)
                    for k in range(60)], dtype=nv.FLAC_SOURCE)
    eng = engine.get_engine(88200, *engine.frame_params(88200))
    launches = nv.lib.nsf_launch_count(eng.handle)
    pcm, off = eng.flac_decode_host(payload, src)
    # 60 x 2.6 M samples: far more than one group of the pipeline, and six launches per group
    assert nv.lib.nsf_launch_count(eng.handle) - launches >= 2 * 6
    expect = x.astype("<i2").tobytes()
    assert off[-1] == 60 * len(expect)
    for k in range(60):
        assert pcm[off[k]:off[k + 1]].tobytes() == expect, k

"""Audio loaders with the reference's names and return conventions (``utils/audio/load_audio.py``).

Division of labour
* **decode** (container -> PCM).  The reference decodes through ``librosa.load`` -> soundfile (libsndfile); neither
  is installable in this image, so ``decode`` dispatches on the stream's first bytes:
  - RIFF/WAVE: a small RIFF reader on the host (container parsing, not arithmetic; SURVEY.md section 8(f)-2) does
    soundfile's conversions (int16 / 32768, int24 / 2**23, int32 / 2**31, uint8 (v - 128) / 128, float32 as is,
    channels averaged);
  - FLAC (``fLaC``): ``flac_layout`` reads the metadata blocks on the host and the frames (Rice codes and linear
    prediction over every sample) are decoded on the GPU through ``nsf_flac_decode_host``, which writes the WAV data
    chunk of the decoded samples; the same host tail as for WAV turns it into the array, so a FLAC file gives exactly
    what the WAV holding its samples gives.  Bits per sample 8, 16 and 24; each frame's CRC-8 and CRC-16 are
    checked, the STREAMINFO MD5 is not;
  - anything else (MP3, Ogg, ...) raises ``ValueError``.
* **peak normalisation** ``y / max|y|`` (reference ``load_audio.py:12-14``) runs on the GPU through
  ``nsf_normalize_host`` - or, on the feature path, fused into ``nsf_extract_host`` via
  ``NSF_PEAK_NORMALIZE`` so the PCM crosses PCIe once, as int16 when the file is int16.
* **resampling** (only when the file's rate differs from the requested one) runs on the GPU through
  ``nsf_resample_host``: a rational polyphase filter with the arithmetic of
  ``scipy.signal.resample_poly`` (Kaiser-windowed sinc), checked against a float64 NumPy oracle.
* ``decode_wav`` + resampling is also the host statement of the batched device conversion
  (``nsf_convert_*``, ``Engine.convert_host``) that ``load_data`` uses for every take that is not mono PCM16 at
  88.2 kHz; that route reproduces these functions bit for bit.  The
  reference uses ``soxr_hq``, whose filter is not reproducible here, so this step is *not*
  parity-pinned against the reference; the synthetic benchmark configurations never resample.
"""
import io
import struct
from collections import namedtuple

import numpy as np

from ... import _native as nv
from ... import engine as _engine

REFERENCE_RATE = 88200  # load_audio.py:8-10: file-path mode always ends at 88.2 kHz

# (format tag, bits per sample) -> nsf_pcm_source encoding: every encoding decode_wav reads
WAV_ENCODINGS = {(1, 8): nv.ENC_U8, (1, 16): nv.ENC_I16, (1, 24): nv.ENC_I24, (1, 32): nv.ENC_I32,
                 (3, 32): nv.ENC_F32, (3, 64): nv.ENC_F64}

WavLayout = namedtuple("WavLayout", "tag channels rate bits data_offset data_bytes")
FlacLayout = namedtuple("FlacLayout", "channels rate bits frames max_block data_offset data_bytes")
FLAC_BITS = (8, 16, 24)


def wav_layout(fh):
    """``WavLayout`` of the seekable binary RIFF/WAVE stream ``fh``, read from its headers.  ``tag`` is the format tag
    (WAVE_FORMAT_EXTENSIBLE's from its sub-format GUID), ``channels`` as declared (0 included).  Odd-sized chunks are
    padded; the first ``data`` chunk ends the walk, truncated at the end of the stream.  ``ValueError`` for every
    stream ``decode_wav`` cannot decode."""
    size = fh.seek(0, io.SEEK_END)
    fh.seek(0)
    head = fh.read(12)
    if len(head) < 12 or head[:4] != b"RIFF" or head[8:12] != b"WAVE":
        raise ValueError("not a RIFF/WAVE stream (only WAV decoding is built in)")
    pos, fmt, data = 12, None, None
    while pos + 8 <= size:
        fh.seek(pos)
        tag, n = struct.unpack("<4sI", fh.read(8))
        if tag == b"fmt ":
            body = fh.read(n)
            fmt = struct.unpack_from("<HHIIHH", body, 0)
            if fmt[0] == 0xFFFE and len(body) >= 26:       # WAVE_FORMAT_EXTENSIBLE: real tag in GUID
                fmt = (struct.unpack_from("<H", body, 24)[0],) + fmt[1:]
        elif tag == b"data":
            data = (pos + 8, min(n, size - (pos + 8)))
            break
        pos += 8 + n + (n & 1)
    if fmt is None or data is None:
        raise ValueError("WAV stream lacks a fmt or data chunk")
    code, channels, rate, _, _, bits = fmt
    if (code, bits) not in WAV_ENCODINGS:
        raise ValueError(f"unsupported WAV encoding (format {code}, {bits} bit)")
    return WavLayout(code, channels, rate, bits, *data)


def decode_wav(data):
    """RIFF/WAVE bytes -> (pcm, native_sr).  pcm is int16 (mono PCM16 files, kept as is so it can
    be uploaded at 2 bytes/sample) or float32 in [-1, 1) (everything else, soundfile scaling)."""
    code, channels, sr, bits, off, n = wav_layout(io.BytesIO(data))
    return _samples(code, channels, bits, data[off:off + n]), sr


def _samples(code, channels, bits, payload):
    """The samples of a WAV data chunk as ``decode_wav`` returns them: int16 for mono PCM16, else float32 in
    [-1, 1) with soundfile's scaling, channels averaged."""
    if code == 1 and bits == 16:
        pcm = np.frombuffer(payload, dtype="<i2", count=len(payload) // 2)
        if channels == 1:
            return pcm.copy()
        x = pcm.astype(np.float32) / np.float32(32768)
    elif code == 1 and bits == 8:
        x = (np.frombuffer(payload, dtype=np.uint8).astype(np.float32) - 128) / np.float32(128)
    elif code == 1 and bits == 24:
        raw = np.frombuffer(payload, dtype=np.uint8, count=len(payload) // 3 * 3).reshape(-1, 3)
        v = (raw[:, 0].astype(np.int32) | (raw[:, 1].astype(np.int32) << 8) |
             (raw[:, 2].astype(np.int8).astype(np.int32) << 16))
        x = (v.astype(np.float64) / float(1 << 23)).astype(np.float32)
    elif code == 1 and bits == 32:
        v = np.frombuffer(payload, dtype="<i4", count=len(payload) // 4)
        x = (v.astype(np.float64) / float(1 << 31)).astype(np.float32)
    elif code == 3 and bits == 32:
        x = np.frombuffer(payload, dtype="<f4", count=len(payload) // 4).copy()
    else:                                                   # (3, 64): wav_layout rejected every other encoding
        x = np.frombuffer(payload, dtype="<f8", count=len(payload) // 8).astype(np.float32)
    if channels > 1:
        x = x[: len(x) // channels * channels].reshape(-1, channels).mean(axis=1, dtype=np.float32)
    return np.ascontiguousarray(x, dtype=np.float32)


def flac_layout(fh):
    """``FlacLayout`` of the seekable binary FLAC stream ``fh``, read from its metadata blocks: STREAMINFO's
    channels, rate, bits per sample, total samples per channel and maximum block size, and the byte range of the
    frames (everything after the last metadata block).  Blocks after STREAMINFO (padding, seek table, tags,
    pictures, ...) are skipped.  ``ValueError`` for every stream ``decode_flac`` does not decode: no ``fLaC``
    marker (an ID3v2 tag or an Ogg page in front included), a missing, misplaced or repeated STREAMINFO, an
    invalid block type, a truncated block, no frame data, 12-, 20- or 32-bit samples, an unknown length (total
    samples 0)."""
    size = fh.seek(0, io.SEEK_END)
    fh.seek(0)
    magic = fh.read(4)
    if magic != b"fLaC":
        if magic[:3] == b"ID3":
            raise ValueError("FLAC stream behind an ID3v2 tag is not supported")
        if magic == b"OggS":
            raise ValueError("Ogg-encapsulated FLAC is not supported")
        raise ValueError("not a FLAC stream (no fLaC marker)")
    pos, info, last = 4, None, False
    while not last:
        head = fh.read(4)
        if len(head) < 4:
            raise ValueError(f"truncated FLAC metadata block header at byte {pos}")
        last, kind, n = head[0] >> 7, head[0] & 0x7F, int.from_bytes(head[1:4], "big")
        if kind == 127:
            raise ValueError(f"invalid FLAC metadata block type 127 at byte {pos}")
        if pos + 4 + n > size:
            raise ValueError(f"truncated FLAC metadata block at byte {pos}")
        if (kind == 0) != (info is None):
            raise ValueError("STREAMINFO is not the first FLAC metadata block" if info is None
                             else "more than one STREAMINFO block")
        if kind == 0:
            if n != 34:
                raise ValueError(f"STREAMINFO block of {n} bytes (34 expected)")
            info = int.from_bytes(fh.read(34)[:18], "big")
        else:
            fh.seek(n, io.SEEK_CUR)
        pos += 4 + n
    max_block = (info >> 112) & 0xFFFF
    rate = (info >> 44) & 0xFFFFF
    channels = ((info >> 41) & 7) + 1
    bits = ((info >> 36) & 31) + 1
    frames = info & ((1 << 36) - 1)
    if bits not in FLAC_BITS:
        raise ValueError(f"unsupported FLAC bits per sample {bits} (8, 16 and 24 are decoded)")
    if frames == 0:
        raise ValueError("FLAC STREAMINFO total samples is 0 (unknown length)")
    if rate == 0:
        raise ValueError("FLAC STREAMINFO sample rate is 0")
    if max_block == 0:
        raise ValueError("FLAC STREAMINFO maximum block size is 0")
    if pos >= size:
        raise ValueError("truncated FLAC stream: no frame data")
    return FlacLayout(channels, rate, bits, frames, max_block, pos, size - pos)


def decode_flac(data):
    """FLAC bytes -> (pcm, native_sr): what ``decode_wav`` returns for the WAV holding the same samples.  The frames
    are decoded on the GPU into the WAV data chunk (u8 v + 128, i16, packed i24); ``ValueError`` for a stream
    ``flac_layout`` rejects and for a corrupt frame (naming its byte offset and the reason)."""
    lay = flac_layout(io.BytesIO(data))
    src = np.array([(lay.data_offset, lay.data_bytes, lay.frames, lay.channels, lay.bits, lay.rate, lay.max_block)],
                   dtype=nv.FLAC_SOURCE)
    f, h = _engine.frame_params(REFERENCE_RATE)
    try:
        pcm, _ = _engine.get_engine(REFERENCE_RATE, f, h).flac_decode_host(np.frombuffer(data, dtype=np.uint8), src)
    except nv.NsfError as e:
        if e.status != nv.ERR_BAD_ARG:
            raise
        raise ValueError(nv.last_error() or str(e)) from None
    return _samples(1, lay.channels, lay.bits, pcm), lay.rate


def _resample(y, orig_sr, target_sr):
    """``librosa.resample`` stand-in on the device (not parity-pinned against soxr_hq, see above)."""
    f, h = _engine.frame_params(int(target_sr))
    return _engine.get_engine(int(target_sr), f, h).resample_host(np.asarray(y), orig_sr, target_sr)


def _read(source):
    if isinstance(source, (bytes, bytearray, memoryview)):
        return bytes(source)
    if isinstance(source, io.IOBase) or hasattr(source, "read"):
        return source.read()
    with open(source, "rb") as fh:
        return fh.read()


def decode(source, sr):
    """``librosa.load(source, sr=sr)`` without the normalisation: (pcm int16|float32, sr)."""
    data = _read(source)
    pcm, native = decode_flac(data) if data[:4] == b"fLaC" else decode_wav(data)
    if sr is not None and native != sr:
        pcm = _resample(pcm, native, sr)
        native = sr
    return pcm, native


def _as_float(pcm):
    return pcm if pcm.dtype == np.float32 else pcm.astype(np.float32) / np.float32(32768)


def _normalize(pcm, sr):
    """Peak normalisation on the device; geometry of the engine follows ``sr`` like the features do."""
    f, h = _engine.frame_params(sr)
    return _engine.get_engine(sr, f, h).normalize_host(pcm)


def load_audio(audio_path, sr=88200):
    """reference load_audio.py:18-21 -- decode (+ resample to ``sr``), no normalisation."""
    pcm, sr = decode(audio_path, sr)
    print(f"Loaded audio file '{audio_path}' with sample rate {sr}")
    return _as_float(pcm), sr


def decode_for_path(audio_path, sr=88200):
    """Decode half of ``load_and_preprocess_audio``: PCM at 88.2 kHz, not yet normalised."""
    pcm, sr = decode(audio_path, sr)
    print(f"Loaded audio file '{audio_path}' with sample rate {sr}")
    if sr != REFERENCE_RATE:                                     # load_audio.py:8-10
        pcm = _resample(pcm, sr, REFERENCE_RATE)
        sr = REFERENCE_RATE
    return pcm, sr


def load_and_preprocess_audio(audio_path, sr=88200):
    """reference load_audio.py:6-16 -- decode, force 88.2 kHz, peak-normalise (on the GPU)."""
    pcm, sr = decode_for_path(audio_path, sr)
    return _normalize(pcm, sr), sr


def load_audio_from_bytes(audio_bytes, sr=88200):
    """reference load_audio.py:23-32 -- decode at ``sr`` (no forced 88.2 kHz), peak-normalise."""
    pcm, sr = decode(io.BytesIO(audio_bytes), sr)
    return _normalize(pcm, sr), sr


def load_audio_file_from_memory(audio_bytes, sr=88200):
    """reference load_audio.py:34-44."""
    pcm, sr = decode(io.BytesIO(audio_bytes), sr)
    print(f"Loaded audio data with sample rate {sr}")
    return _normalize(pcm, sr), sr

"""Audio loaders with the reference's names and return conventions (``utils/audio/load_audio.py``).

Division of labour
* **decode** (RIFF/WAV container -> PCM) stays on the host: it is container parsing, not arithmetic
  (SURVEY.md section 8(f)-2 lists on-device decode/resample as a later row).  The reference decodes
  through ``librosa.load`` -> soundfile; here a small RIFF reader does the same conversions
  (int16 / 32768, int24 / 2**23, int32 / 2**31, uint8 (v - 128) / 128, float32 as is, channels
  averaged) because neither librosa nor soundfile is installable in this image.
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

import numpy as np

from ... import engine as _engine

REFERENCE_RATE = 88200  # load_audio.py:8-10: file-path mode always ends at 88.2 kHz


def decode_wav(data):
    """RIFF/WAVE bytes -> (pcm, native_sr).  pcm is int16 (mono PCM16 files, kept as is so it can
    be uploaded at 2 bytes/sample) or float32 in [-1, 1) (everything else, soundfile scaling)."""
    if len(data) < 12 or data[:4] != b"RIFF" or data[8:12] != b"WAVE":
        raise ValueError("not a RIFF/WAVE stream (only WAV decoding is built in)")
    pos, fmt, payload = 12, None, None
    while pos + 8 <= len(data):
        tag, size = data[pos:pos + 4], struct.unpack_from("<I", data, pos + 4)[0]
        body = data[pos + 8: pos + 8 + size]
        if tag == b"fmt ":
            fmt = struct.unpack_from("<HHIIHH", body, 0)
            if fmt[0] == 0xFFFE and len(body) >= 26:       # WAVE_FORMAT_EXTENSIBLE: real tag in GUID
                fmt = (struct.unpack_from("<H", body, 24)[0],) + fmt[1:]
        elif tag == b"data":
            payload = body
            break
        pos += 8 + size + (size & 1)
    if fmt is None or payload is None:
        raise ValueError("WAV stream lacks a fmt or data chunk")
    code, channels, sr, _, _, bits = fmt
    if code == 1 and bits == 16:
        pcm = np.frombuffer(payload, dtype="<i2", count=len(payload) // 2)
        if channels == 1:
            return pcm.copy(), sr
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
    elif code == 3 and bits == 64:
        x = np.frombuffer(payload, dtype="<f8", count=len(payload) // 8).astype(np.float32)
    else:
        raise ValueError(f"unsupported WAV encoding (format {code}, {bits} bit)")
    if channels > 1:
        x = x[: len(x) // channels * channels].reshape(-1, channels).mean(axis=1, dtype=np.float32)
    return np.ascontiguousarray(x, dtype=np.float32), sr


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
    pcm, native = decode_wav(_read(source))
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

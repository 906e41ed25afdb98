"""GPU-backed mirror of the reference's ``dataset/data_processing.py`` (dataset builders).

Host side (unchanged semantics): folder scan, CSV cache of ``audio_features.csv``, the facial CSV
minus ``Timecode`` / ``BlendshapeCount``, ``facial[:, :61] *= 100``.
Device side: feature extraction (``extract_audio_features``) and the whole ``collect_features``
augmentation - centre-trim, fast ``[::2]``, slow ``interpolate_slower`` (+ ``smooth_facial_data``),
``stack_with_blend`` - as one ``nsf_collect_host`` call in float64, bit-identical to the NumPy
arithmetic of the reference (same operation order, IEEE add/mul, no FMA contraction).

``load_data`` keeps the reference signature but builds the whole dataset in ONE pipelined device pass
(``load_data_batched``): the folders are scanned first, every take without a feature cache is read straight
into a page-locked arena (int16 samples when every take is mono PCM16 at 88.2 kHz, else the raw WAV bytes, which
``nsf_convert_host`` decodes, downmixes and resamples on the device), ``nsf_extract_collect_host`` turns PCM + facial rows into augmented rows
without the feature rows ever leaving the GPU, and the examples are float32 (``dataset/dataset.py:75`` casts to
float32 anyway).  ``process_folder`` / ``collect_features`` remain the
per-take float64 route, bit-identical to the reference's NumPy arithmetic.
"""
import os

import numpy as np
import pandas as pd

from .. import _native as nv
from .. import engine as _engine
from ..utils.audio.extraction.extract_features import extract_audio_features
from ..utils.video.mov_extraction import find_files, get_audio

COLUMNS_TO_DROP = ['Timecode', 'BlendshapeCount']


def _engine_any():
    f, h = _engine.frame_params(88200)
    return _engine.get_engine(88200, f, h)


def _rows64(a):
    a = np.asarray(a)
    if a.dtype not in (np.float32, np.float64):
        a = a.astype(np.float64)
    return np.ascontiguousarray(a)


def load_data(root_dir, sr, processed_folders):
    """reference :10-26 -- examples in ``os.listdir`` order, skips (and records) processed folders.

    Same folder scan, cache files, ``collect_features`` defaults and ``facial[:, :61] *= 100`` as the
    reference's loop over ``process_folder``, executed as one batched pass (see ``load_data_batched``);
    examples are float32.  ``load_data_per_folder`` is the literal folder-by-folder loop (float64)."""
    return load_data_batched(root_dir, sr, processed_folders)[0]


def load_data_per_folder(root_dir, sr, processed_folders):
    """The reference's loop verbatim: one ``process_folder`` (float64, bit-exact arithmetic) per folder."""
    examples = []
    for folder in os.listdir(root_dir):
        folder_path = os.path.join(root_dir, folder)
        if os.path.isdir(folder_path) and folder not in processed_folders:
            audio_features, facial_data = process_folder(folder_path, sr)
            if audio_features is not None and facial_data is not None:
                examples.append((audio_features, facial_data))
                processed_folders.add(folder)
    return examples


def scale_facial_data(facial_data, scale_factor=1.1):
    """reference :28-41 (unused helper; host NumPy): scale then clip to [-1, 1]."""
    return np.clip(np.asarray(facial_data) * scale_factor, -1, 1)


def process_folder(folder_path, sr, apply_smoothing=False, apply_over_scale=False):
    """reference :44-78."""
    mov_path, mp4_path, wav_path, facial_csv_path, audio_features_csv_path, _ = find_files(folder_path)
    video_path = mov_path or mp4_path
    have_cache = os.path.exists(audio_features_csv_path)
    if not (facial_csv_path and (video_path or wav_path or have_cache)):
        return None, None
    audio_path = get_audio(video_path, wav_path, folder_path) if (video_path or wav_path) else None
    if not (audio_path or have_cache):
        return None, None
    audio_features, facial_data = collect_features(audio_path if audio_path else _, audio_features_csv_path,
                                                   facial_csv_path, sr)
    if apply_over_scale:
        facial_data = scale_facial_data(facial_data)
    facial_data[:, :61] *= 100                                            # :68
    if apply_smoothing:
        facial_data = smooth_facial_data(facial_data)
    return audio_features, facial_data


def interpolate_slower(data):
    """reference :84-106 -- ``(N, F) -> (2N-1, F)``: originals on even rows, midpoints on odd rows."""
    data = _rows64(data)
    if data.shape[0] == 0:
        raise ValueError("interpolate_slower needs at least one row")
    out = _engine_any().rows_op(nv.ROWS_INTERP_SLOWER, data)
    return out.astype(np.float64, copy=False)  # the reference allocates np.zeros (float64)


def collect_arrays(audio_features, facial_data, include_fast=True, include_slow=False,
                   blend_boundaries=True, blend_frames=30):
    """The arithmetic of collect_features (reference :126-177) for one clip, on the device."""
    a = _rows64(audio_features)
    f = np.ascontiguousarray(facial_data, dtype=a.dtype)
    if not (include_fast or include_slow) or min(len(a), len(f)) == 0:
        # no augmentation: only the (host) length matching remains
        n = min(len(a), len(f))
        la = (len(a) - n) // 2 if len(a) > len(f) else 0
        lf = (len(f) - n) // 2 if len(f) > len(a) else 0
        return a[la:la + n], f[lf:lf + n]
    out_a, out_f, _ = _engine_any().collect_host(a, [0, len(a)], f, [0, len(f)], include_fast,
                                                 include_slow, blend_boundaries, blend_frames)
    return out_a, out_f


def _binary_cache_path(audio_features_csv_path):
    return os.path.splitext(audio_features_csv_path)[0] + ".npy"


def collect_features(audio_path, audio_features_csv_path, facial_csv_path, sr,
                     include_fast=True, include_slow=False, blend_boundaries=True, blend_frames=30,
                     cache_format=None):
    """reference :108-177 -- same CSV cache side effects, same return shapes and dtypes.

    ``cache_format`` (extension, SURVEY section 8(f)-3; default from ``NSF_FEATURE_CACHE`` or "csv"):
    "csv" = the reference's ``audio_features.csv`` (1.3 s and 9 MB per 30 s clip to write);
    "npy" = a float32 ``audio_features.npy`` beside it (milliseconds, 1.8 MB); "both" writes both.
    An existing CSV cache is always honoured first, exactly like the reference."""
    cache_format = cache_format or os.environ.get("NSF_FEATURE_CACHE", "csv")
    if cache_format not in ("csv", "npy", "both"):
        raise ValueError("cache_format must be 'csv', 'npy' or 'both'")
    npy_path = _binary_cache_path(audio_features_csv_path)
    if os.path.exists(audio_features_csv_path):                           # :112-114
        print(f"Loading audio features from {audio_features_csv_path}")
        audio_features = pd.read_csv(audio_features_csv_path).values
    elif cache_format != "csv" and os.path.exists(npy_path):
        print(f"Loading audio features from {npy_path}")
        audio_features = np.load(npy_path).astype(np.float64)
    else:                                                                 # :115-120
        print(f"Extracting audio features from {audio_path}")
        audio_features, _ = extract_audio_features(audio_path, sr)
        if audio_features is not None:
            if cache_format in ("csv", "both"):
                pd.DataFrame(audio_features).to_csv(audio_features_csv_path, index=False)
                print(f"Audio features saved to {audio_features_csv_path}")
            if cache_format in ("npy", "both"):
                np.save(npy_path, audio_features.astype(np.float32))
                print(f"Audio features saved to {npy_path}")
    facial_data = pd.read_csv(facial_csv_path).drop(columns=COLUMNS_TO_DROP).values   # :123
    if audio_features is None:
        # the reference fails here with TypeError: object of type 'NoneType' has no len() (:143)
        raise TypeError("object of type 'NoneType' has no len()")
    return collect_arrays(audio_features, facial_data, include_fast, include_slow, blend_boundaries,
                          blend_frames)


def stack_with_blend(sequences, blend_frames):
    """reference :179-197 -- inclusive-linspace cross-fade over ``min(blend, len, len)`` rows."""
    if not sequences:
        return None
    result = _rows64(sequences[0])
    eng = _engine_any()
    for seq in sequences[1:]:
        seq = np.ascontiguousarray(seq, dtype=result.dtype)
        if len(seq) == 0:
            continue
        if len(result) == 0:
            result = seq
            continue
        result = eng.rows_op(nv.ROWS_BLEND_STACK, result, seq, blend_frames)
    return result


def smooth_facial_data(facial_data):
    """reference :201-204 -- rows 1.. <- mean of (row i-1, row i), from the original rows."""
    x = _rows64(facial_data)
    if len(x) == 0:
        return x.copy()
    return _engine_any().rows_op(nv.ROWS_SMOOTH, x)


def remove_specified_dimensions(facial_data):
    """reference :208-212 (unused helper; host NumPy)."""
    cols = list(range(14)) + list(range(51, 61))
    return np.delete(facial_data, cols, axis=1)


def zero_specified_columns(facial_data):
    """reference :214-220 (unused helper; host NumPy, in place)."""
    cols = list(range(14)) + list(range(51, 61))
    facial_data[:, cols] = 0
    return facial_data


# ------------------------------------------------------------------------------------------------
# B200-first batched builder
# ------------------------------------------------------------------------------------------------
def collect_batch(audio_rows, facial_rows, include_fast=True, include_slow=False,
                  blend_boundaries=True, blend_frames=30, device=None, dtype=np.float32):
    """collect_features arithmetic for MANY clips in one device call.

    ``audio_rows`` / ``facial_rows``: lists of ``[N_i, 256]`` / ``[M_i, 61]`` arrays.  Returns
    ``(audio [sum, 256], facial [sum, 61], offsets)`` in ``dtype`` (float32 = training format,
    float64 = the reference's arithmetic bit for bit)."""
    f0, h0 = _engine.frame_params(88200)
    eng = _engine.get_engine(88200, f0, h0, device=device)
    a_off = np.zeros(len(audio_rows) + 1, dtype=np.int64)
    f_off = np.zeros(len(facial_rows) + 1, dtype=np.int64)
    np.cumsum([len(a) for a in audio_rows], out=a_off[1:])
    np.cumsum([len(f) for f in facial_rows], out=f_off[1:])
    a = np.concatenate([np.asarray(x, dtype=dtype) for x in audio_rows], axis=0)
    f = np.concatenate([np.asarray(x, dtype=dtype) for x in facial_rows], axis=0)
    return eng.collect_host(a, a_off, f, f_off, include_fast, include_slow, blend_boundaries,
                            blend_frames)


def _pcm16_payload(path, sr):
    """(byte offset, sample count) of the data chunk when ``path`` is a mono PCM16 RIFF/WAVE file at ``sr`` -
    the format ffmpeg writes for the takes (utils/video/mov_extraction.py:50-57) - else None."""
    import struct
    try:
        with open(path, "rb") as fh:
            head = fh.read(12)
            if len(head) < 12 or head[:4] != b"RIFF" or head[8:12] != b"WAVE":
                return None
            fmt, pos = None, 12
            while True:
                hdr = fh.read(8)
                if len(hdr) < 8:
                    return None
                tag, size = hdr[:4], struct.unpack("<I", hdr[4:])[0]
                if tag == b"fmt ":
                    fmt = struct.unpack("<HHIIHH", fh.read(16))
                    fh.seek(pos + 8 + size + (size & 1))
                elif tag == b"data":
                    if fmt is None or fmt[0] != 1 or fmt[1] != 1 or fmt[5] != 16 or fmt[2] != sr:
                        return None
                    avail = os.path.getsize(path) - (pos + 8)
                    return pos + 8, min(size, max(avail, 0)) // 2
                else:
                    fh.seek(pos + 8 + size + (size & 1))
                pos += 8 + size + (size & 1)
    except OSError:
        return None


_WAV_ENCODINGS = {(1, 8): nv.ENC_U8, (1, 16): nv.ENC_I16, (1, 24): nv.ENC_I24, (1, 32): nv.ENC_I32,
                  (3, 32): nv.ENC_F32, (3, 64): nv.ENC_F64}
_ENC_BYTES = {nv.ENC_U8: 1, nv.ENC_I16: 2, nv.ENC_I24: 3, nv.ENC_I32: 4, nv.ENC_F32: 4, nv.ENC_F64: 8}


def _wav_source(path):
    """(data offset, data bytes, encoding, channels, rate) of a RIFF/WAVE file, read from its headers only.

    The chunk walk of ``decode_wav`` (utils/audio/load_audio.py), step for step: WAVE_FORMAT_EXTENSIBLE takes its
    format tag from the sub-format GUID, odd-sized chunks are padded, the first ``data`` chunk ends the walk and is
    truncated at the end of the file.  Raises ``decode_wav``'s ``ValueError`` for what ``decode_wav`` rejects.  A
    header declaring 0 channels (which ``decode_wav`` reads as mono) reports 1."""
    import struct
    size_all = os.path.getsize(path)
    with open(path, "rb") as fh:
        head = fh.read(12)
        if len(head) < 12 or head[:4] != b"RIFF" or head[8:12] != b"WAVE":
            raise ValueError("not a RIFF/WAVE stream (only WAV decoding is built in)")
        pos, fmt, data = 12, None, None
        while pos + 8 <= size_all:
            fh.seek(pos)
            hdr = fh.read(8)
            tag, size = hdr[:4], struct.unpack_from("<I", hdr, 4)[0]
            if tag == b"fmt ":
                body = fh.read(size)
                fmt = struct.unpack_from("<HHIIHH", body, 0)
                if fmt[0] == 0xFFFE and len(body) >= 26:
                    fmt = (struct.unpack_from("<H", body, 24)[0],) + fmt[1:]
            elif tag == b"data":
                data = (pos + 8, min(size, size_all - (pos + 8)))
                break
            pos += 8 + size + (size & 1)
    if fmt is None or data is None:
        raise ValueError("WAV stream lacks a fmt or data chunk")
    code, channels, rate, _, _, bits = fmt
    enc = _WAV_ENCODINGS.get((code, bits))
    if enc is None:
        raise ValueError(f"unsupported WAV encoding (format {code}, {bits} bit)")
    return data[0], data[1], enc, max(int(channels), 1), int(rate)


def _read_into(path, offset, dst):
    with open(path, "rb", buffering=0) as fh:
        fh.seek(offset)
        view = memoryview(dst).cast("B")
        got = 0
        while got < len(view):
            n = fh.readinto(view[got:])
            if not n:
                raise OSError(f"short read from {path}")
            got += n


def _facial_rows(path, dtype):
    """The facial CSV minus Timecode / BlendshapeCount (:123).  float64: pandas' default parser, value for value
    what the reference reads.  float32 (training format): Arrow's multi-threaded reader, 4x faster per file and
    free of the GIL - its correctly rounded float64 values differ from pandas' fast parser by at most one ulp,
    which the cast to float32 absorbs."""
    if dtype == np.float32:
        try:
            import pyarrow.csv as pacsv
            # single-threaded parse: the caller's thread pool already runs one file per core, and Arrow drops the GIL
            table = pacsv.read_csv(path, read_options=pacsv.ReadOptions(use_threads=False)).drop_columns(COLUMNS_TO_DROP)
            out = np.empty((table.num_rows, table.num_columns), dtype=np.float32)
            for j, col in enumerate(table.columns):
                out[:, j] = col.to_numpy()
            return out
        except Exception:      # noqa: BLE001 - anything Arrow cannot type as numbers goes the reference's way
            pass
    return np.ascontiguousarray(pd.read_csv(path).drop(columns=COLUMNS_TO_DROP).values, dtype=dtype)


last_timing = {}     # phase -> seconds of the most recent load_data_batched call (bench.py reports it)


def load_data_batched(root_dir, sr, processed_folders, include_fast=True, include_slow=False,
                      blend_boundaries=True, blend_frames=30, rank=0, world=1, cache_format=None,
                      device=None, dtype=np.float32, io_threads=None):
    """``load_data`` (reference :10-26) for a whole dataset in one pipelined device pass.

    Returns ``(examples, indices)``: ``(audio_features, facial_data)`` pairs in ``os.listdir`` order (what
    ``load_data`` + ``process_folder`` + ``collect_features`` produce, including the cache files, the
    ``processed_folders`` updates and ``facial[:, :61] *= 100``) and the position of each example in the
    full take list.  With ``world > 1`` the takes are split by clip over ranks (``shard.lpt_partition``
    on the size of each take's SOURCE file, which exists identically for every rank before anything is
    extracted); a rank only touches - and only runs ffmpeg for - its own takes.

    ``dtype=np.float32`` (default, the training format): takes without a feature cache are read straight
    into page-locked memory by a thread pool (int16 samples, or raw WAV bytes converted to float32 at 88.2 kHz by
    ``nsf_convert_host`` exactly as ``decode_for_path`` would when any take is in another format or rate), go through ``nsf_extract_collect_host`` (features and
    augmentation fused, rows never leave the device in between) and come back as float32 arrays; cached takes are augmented by one float32 ``nsf_collect_host`` call.
    ``dtype=np.float64``: extraction batched, augmentation through the float64 kernel - bit-identical to
    the per-folder builder.  A take shorter than 9 frames raises ``TypeError`` exactly where the
    reference does (``len(None)``, :143)."""
    import time
    from concurrent.futures import ThreadPoolExecutor

    from .. import shard
    from ..utils.audio.extraction.extract_features import MIN_FRAMES
    from ..utils.audio.load_audio import REFERENCE_RATE

    t_start = time.perf_counter()
    timing = {}
    cache_format = cache_format or os.environ.get("NSF_FEATURE_CACHE", "csv")
    if cache_format not in ("csv", "npy", "both"):
        raise ValueError("cache_format must be 'csv', 'npy' or 'both'")
    if dtype not in (np.float32, np.float64):
        raise ValueError("dtype must be numpy.float32 or numpy.float64")
    takes = []                      # (folder, source audio/video, wav, cache_csv, facial_csv, folder_path)
    for folder in os.listdir(root_dir):
        folder_path = os.path.join(root_dir, folder)
        if not os.path.isdir(folder_path) or folder in processed_folders:
            continue
        mov, mp4, wav, facial_csv, cache_csv, _ = find_files(folder_path)
        video = mov or mp4
        have_cache = os.path.exists(cache_csv) or (cache_format != "csv" and
                                                   os.path.exists(_binary_cache_path(cache_csv)))
        if not (facial_csv and (video or wav or have_cache)):
            continue
        takes.append((folder, video, wav, cache_csv, facial_csv, folder_path))
    # partition on files every rank sees identically BEFORE any rank extracts audio (never on audio.wav, which
    # another rank may be writing): the take's video, else its wav, else its cache
    def weight(t):
        for cand in (t[1], t[2], t[3]):
            if cand and os.path.exists(cand):
                return max(1, os.path.getsize(cand))
        return 1
    mine = shard.lpt_partition([weight(t) for t in takes], world)[rank] if world > 1 else list(range(len(takes)))
    timing["scan"] = time.perf_counter() - t_start

    f_len, h_len = _engine.frame_params(REFERENCE_RATE)     # file-path mode always lands at 88.2 kHz
    eng = _engine.get_engine(REFERENCE_RATE, f_len, h_len, device=device)
    threads = io_threads or min(32, len(os.sched_getaffinity(0)) or 1)
    pool = ThreadPoolExecutor(max_workers=threads)
    try:
        # ---- which takes need extraction; where their audio is -------------------------------------------
        t0 = time.perf_counter()
        cached, todo = {}, []            # take -> rows | (take, audio_path)
        for i in mine:
            folder, video, wav, cache_csv, facial_csv, folder_path = takes[i]
            if os.path.exists(cache_csv):                                      # :112-114
                print(f"Loading audio features from {cache_csv}")
                cached[i] = pool.submit(lambda p=cache_csv: pd.read_csv(p).values)
            elif cache_format != "csv" and os.path.exists(_binary_cache_path(cache_csv)):
                print(f"Loading audio features from {_binary_cache_path(cache_csv)}")
                cached[i] = pool.submit(np.load, _binary_cache_path(cache_csv))
            else:
                audio_path = get_audio(video, wav, folder_path) if (video or wav) else None
                if not audio_path:
                    continue                                                   # process_folder returns (None, None)
                print(f"Extracting audio features from {audio_path}")
                todo.append((i, audio_path))
        todo_set = {j for j, _ in todo}
        keep = [i for i in mine if i in cached or i in todo_set]
        facial_jobs = {}

        # ---- PCM of the takes to extract: mono PCM16 files at 88.2 kHz are read straight into page-locked
        # int16 memory (2 bytes per sample over PCIe); every other take's raw bytes are decoded, downmixed and
        # resampled to float32 on the device by nsf_convert_host ------------------------------------------------
        n_rows = {}
        pcm_arena = pcm = off = None
        if todo:
            info = [_pcm16_payload(p, REFERENCE_RATE) if sr == REFERENCE_RATE else None for _, p in todo]
            fast = all(x is not None for x in info)
            if fast:
                lens = [n for _, n in info]
            else:
                # every other take: raw data-chunk bytes, converted on the device (decode_for_path's arithmetic)
                heads = list(pool.map(lambda tp: _wav_source(tp[1]), todo))
                for (_, p), h in zip(todo, heads):
                    print(f"Loaded audio file '{p}' with sample rate {sr if sr is not None else h[4]}")
                # sr=None keeps the native rate in decode(): one conversion, native -> 88.2 kHz
                sr1 = sr if sr is not None else REFERENCE_RATE
                src = np.zeros(len(todo), dtype=nv.PCM_SOURCE)
                pos = 0
                for k, (_, nbytes, enc, ch, rate) in enumerate(heads):
                    frames = nbytes // (_ENC_BYTES[enc] * ch)
                    src[k] = (pos, frames, enc, ch, rate, 0)
                    pos += (frames * _ENC_BYTES[enc] * ch + 7) // 8 * 8          # every take 8-byte aligned
                mid_off = nv.convert_offsets(src, sr1, pos)                       # native rate -> sr
                if sr1 != REFERENCE_RATE:                                          # then sr -> 88.2 kHz (load_audio.py:8-10)
                    mid = np.zeros(len(todo), dtype=nv.PCM_SOURCE)
                    for k in range(len(todo)):
                        mid[k] = (int(mid_off[k]) * 4, int(mid_off[k + 1] - mid_off[k]), nv.ENC_F32, 1, sr1, 0)
                    lens = np.diff(nv.convert_offsets(mid, REFERENCE_RATE, int(mid_off[-1]) * 4))
                else:
                    lens = np.diff(mid_off)
            for (i, _), n in zip(todo, lens):
                g = eng.plan.guard_frames(n)
                if g < MIN_FRAMES:                                             # extract_features.py:16-20 -> :143
                    print(f"Audio file is too short: {g} frames, required: {MIN_FRAMES} frames")
                    raise TypeError("object of type 'NoneType' has no len()")
            off = np.zeros(len(todo) + 1, dtype=np.int64)
            np.cumsum(lens, out=off[1:])
            item = 2 if fast else 4
            pcm_arena = _engine.scratch_pinned("dataset_pcm", int(off[-1]) * item)   # library-owned, reused
            pcm = pcm_arena.view(np.int16 if fast else np.float32, (int(off[-1]),))
            if fast:
                for (_, p) in todo:
                    print(f"Loaded audio file '{p}' with sample rate {REFERENCE_RATE}")
                reads = [pool.submit(_read_into, todo[k][1], info[k][0], pcm[off[k]:off[k + 1]]) for k in range(len(todo))]
                facial_jobs = {i: pool.submit(_facial_rows, takes[i][4], dtype) for i in keep}   # queued behind the reads
                for r in reads:
                    r.result()
            else:
                wav_arena = _engine.scratch_pinned("dataset_wav", max(pos, 1))
                raw = wav_arena.view(np.uint8, (pos,))
                reads = [pool.submit(_read_into, todo[k][1], heads[k][0], raw[int(src[k]["byte_offset"]):
                                     int(src[k]["byte_offset"]) + int(src[k]["frames"]) * _ENC_BYTES[heads[k][2]] *
                                     heads[k][3]]) for k in range(len(todo)) if src[k]["frames"] > 0]
                facial_jobs = {i: pool.submit(_facial_rows, takes[i][4], dtype) for i in keep}
                for r in reads:
                    r.result()
                if sr1 != REFERENCE_RATE:
                    y_sr = _engine.scratch_pinned("dataset_wav_mid", max(int(mid_off[-1]) * 4, 1)).view(
                        np.float32, (int(mid_off[-1]),))
                    eng.convert_host(raw, src, sr1, out=y_sr)
                    eng.convert_host(y_sr.view(np.uint8), mid, REFERENCE_RATE, out=pcm)
                else:
                    eng.convert_host(raw, src, sr1, out=pcm)
            roff = eng.row_offsets(off)
            for k, (i, _) in enumerate(todo):
                n_rows[i] = int(roff[k + 1] - roff[k])
        timing["read_audio"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        for i in keep:
            if i not in facial_jobs:
                facial_jobs[i] = pool.submit(_facial_rows, takes[i][4], dtype)
        facial = {i: j.result() for i, j in facial_jobs.items()}
        cached = {i: j.result() for i, j in cached.items()}
        timing["facial_csv_wait"] = time.perf_counter() - t0

        # ---- device pass ------------------------------------------------------------------------------------
        t0 = time.perf_counter()
        results = {}                    # take -> (audio rows, facial rows)
        feats_by_take = {}
        kw = dict(include_fast=include_fast, include_slow=include_slow, blend_boundaries=blend_boundaries,
                  blend_frames=blend_frames)
        augment = include_fast or include_slow
        if todo:
            order = [i for i, _ in todo]
            f_off = np.zeros(len(order) + 1, dtype=np.int64)
            np.cumsum([len(facial[i]) for i in order], out=f_off[1:])
            if dtype == np.float32 and augment and all(n_rows[i] and len(facial[i]) for i in order):
                f_cols = facial[order[0]].shape[1]
                fac_arena = _engine.scratch_pinned("dataset_facial", int(f_off[-1]) * f_cols * 4)
                fac = fac_arena.view(np.float32, (int(f_off[-1]), f_cols))
                for k, i in enumerate(order):
                    fac[f_off[k]:f_off[k + 1]] = facial[i]
                o_off = eng.collect_rows(roff, f_off, **kw)
                # results go to ordinary (pageable) arrays the caller owns: the library stages the downloads through
                # its own page-locked arenas, which costs a host copy but not a cudaHostAlloc of ~300 MB per call
                out_a = np.empty((int(o_off[-1]), 256), dtype=np.float32)
                out_f = np.empty((int(o_off[-1]), f_cols), dtype=np.float32)
                feats = np.empty((int(roff[-1]), 256), dtype=np.float32)
                eng.extract_collect_host(pcm, off, fac, f_off, nv.PEAK_NORMALIZE, out_audio=out_a, out_facial=out_f,
                                         features_out=feats, **kw)
                for k, i in enumerate(order):
                    results[i] = (out_a[o_off[k]:o_off[k + 1]], out_f[o_off[k]:o_off[k + 1]])
                    feats_by_take[i] = feats[roff[k]:roff[k + 1]]
            else:
                rows = eng.extract_host(pcm, off, nv.PEAK_NORMALIZE)
                for k, i in enumerate(order):
                    feats_by_take[i] = rows[roff[k]:roff[k + 1]]
                    cached[i] = feats_by_take[i]
        if cached:
            order = sorted(cached)
            rows_in = [np.ascontiguousarray(cached[i], dtype=dtype) for i in order]
            if augment and all(len(r) for r in rows_in) and all(len(facial[i]) for i in order):
                a_off = np.zeros(len(order) + 1, dtype=np.int64)
                np.cumsum([len(r) for r in rows_in], out=a_off[1:])
                f_off = np.zeros(len(order) + 1, dtype=np.int64)
                np.cumsum([len(facial[i]) for i in order], out=f_off[1:])
                out_a, out_f, o_off = eng.collect_host(np.concatenate(rows_in, axis=0), a_off,
                                                       np.concatenate([facial[i] for i in order], axis=0), f_off, **kw)
                for k, i in enumerate(order):
                    results[i] = (out_a[o_off[k]:o_off[k + 1]], out_f[o_off[k]:o_off[k + 1]])
            else:
                for r, i in zip(rows_in, order):
                    results[i] = tuple(np.array(x) for x in collect_arrays(r, facial[i], **kw))
        timing["device"] = time.perf_counter() - t0

        # ---- side effects: feature caches (:115-120), facial scaling (:68), processed_folders (:24) ---------
        t0 = time.perf_counter()
        def write_cache(i):
            cache_csv, f = takes[i][3], feats_by_take[i]
            if cache_format in ("csv", "both"):
                pd.DataFrame(np.asarray(f, dtype=np.float64)).to_csv(cache_csv, index=False)
                print(f"Audio features saved to {cache_csv}")
            if cache_format in ("npy", "both"):
                np.save(_binary_cache_path(cache_csv), np.asarray(f, dtype=np.float32))
                print(f"Audio features saved to {_binary_cache_path(cache_csv)}")
        list(pool.map(write_cache, list(feats_by_take)))
        timing["write_cache"] = time.perf_counter() - t0
    finally:
        pool.shutdown(wait=True)
    examples, indices = [], []
    for i in mine:
        if i not in results:
            continue
        a, f = results[i]
        f[:, :61] *= 100                                                   # process_folder :68
        examples.append((a, f))
        indices.append(i)
        processed_folders.add(takes[i][0])
    timing["total"] = time.perf_counter() - t_start
    last_timing.clear()
    last_timing.update(timing)
    return examples, indices


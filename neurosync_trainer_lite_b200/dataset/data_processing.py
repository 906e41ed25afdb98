"""GPU-backed mirror of the reference's ``dataset/data_processing.py`` (dataset builders).

Host side (unchanged semantics): folder scan, reading the ``audio_features.csv`` cache, the facial CSV
minus ``Timecode`` / ``BlendshapeCount``, ``facial[:, :61] *= 100``.  The cache's text is formatted on the device
(``Engine.format_csv``), byte for byte what the reference's pandas writer produces, and the batched builder parses
both kinds of CSV on the device (``Engine.parse_csv``), value for value what pandas reads.
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
from collections import namedtuple

import numpy as np
import pandas as pd

from .. import _native as nv
from .. import engine as _engine
from ..utils.audio.extraction.extract_features import MIN_FRAMES, extract_audio_features
from ..utils.audio.load_audio import REFERENCE_RATE, WAV_ENCODINGS, wav_layout
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


def _cache_format(cache_format):
    """``cache_format``, else ``NSF_FEATURE_CACHE``, else "csv"; validated."""
    cache_format = cache_format or os.environ.get("NSF_FEATURE_CACHE", "csv")
    if cache_format not in ("csv", "npy", "both"):
        raise ValueError("cache_format must be 'csv', 'npy' or 'both'")
    return cache_format


def _binary_cache_path(audio_features_csv_path):
    return os.path.splitext(audio_features_csv_path)[0] + ".npy"


def _cached_features_path(cache_csv, cache_format):
    """The feature cache to read (:112-114): the CSV if it exists, else the ``.npy`` unless the format is "csv"."""
    if os.path.exists(cache_csv):
        return cache_csv
    npy_path = _binary_cache_path(cache_csv)
    return npy_path if cache_format != "csv" and os.path.exists(npy_path) else None


def _read_feature_cache(path):
    return np.load(path) if path.endswith(".npy") else pd.read_csv(path).values


def _write_feature_cache(cache_csv, rows, cache_format, text=None):
    """The cache files of one take's feature rows (:115-120): the CSV from float64, the ``.npy`` from float32.
    The CSV is ``text``, the take's device-formatted bytes of ``Engine.format_csv`` (formatted here when None):
    byte for byte what the reference's ``pd.DataFrame(rows).to_csv(path, index=False)`` writes."""
    if cache_format in ("csv", "both"):
        if text is None:
            text = _engine_any().format_csv(rows)[0]
        with open(cache_csv, "wb") as fh:
            fh.write(text)
        print(f"Audio features saved to {cache_csv}")
    if cache_format in ("npy", "both"):
        npy_path = _binary_cache_path(cache_csv)
        np.save(npy_path, np.asarray(rows, dtype=np.float32))
        print(f"Audio features saved to {npy_path}")


def collect_features(audio_path, audio_features_csv_path, facial_csv_path, sr,
                     include_fast=True, include_slow=False, blend_boundaries=True, blend_frames=30,
                     cache_format=None):
    """reference :108-177 -- same CSV cache side effects, same return shapes and dtypes.

    ``cache_format`` (extension, SURVEY section 8(f)-3; default from ``NSF_FEATURE_CACHE`` or "csv"):
    "csv" = the reference's ``audio_features.csv`` (9.5 MB per 30 s clip, formatted on the device);
    "npy" = a float32 ``audio_features.npy`` beside it (milliseconds, 1.8 MB); "both" writes both.
    An existing CSV cache is always honoured first, exactly like the reference."""
    cache_format = _cache_format(cache_format)
    cache_path = _cached_features_path(audio_features_csv_path, cache_format)
    if cache_path:
        print(f"Loading audio features from {cache_path}")
        audio_features = np.asarray(_read_feature_cache(cache_path), dtype=np.float64)
    else:                                                                 # :115-120
        print(f"Extracting audio features from {audio_path}")
        audio_features, _ = extract_audio_features(audio_path, sr)
        if audio_features is not None:
            _write_feature_cache(audio_features_csv_path, audio_features, cache_format)
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


def _prefix(lengths):
    """``[0, l0, l0 + l1, ...]`` as int64 offsets."""
    off = np.zeros(len(lengths) + 1, dtype=np.int64)
    np.cumsum(lengths, out=off[1:])
    return off


_ENC_BYTES = {nv.ENC_U8: 1, nv.ENC_I16: 2, nv.ENC_I24: 3, nv.ENC_I32: 4, nv.ENC_F32: 4, nv.ENC_F64: 8}


def _wav_source(path):
    """(data offset, data bytes, encoding, declared channels, rate) of a WAV file, from its headers only
    (``wav_layout``: ``decode_wav``'s chunk walk and its ``ValueError`` for what it cannot decode)."""
    with open(path, "rb") as fh:
        h = wav_layout(fh)
    return h.data_offset, h.data_bytes, WAV_ENCODINGS[h.tag, h.bits], h.channels, h.rate


# sources: nv.PCM_SOURCE per take, offsets into the read arena of nbytes bytes; lengths: samples at 88.2 kHz;
# rate: the first conversion's target; mid: the second conversion's sources (float32 at rate), None at 88.2 kHz
_AudioPlan = namedtuple("_AudioPlan", "int16 sources lengths nbytes rate mid")


def _plan_audio(heads, sr):
    """How takes with these WAV headers become ``decode_for_path``'s PCM at 88.2 kHz; host only.  The int16 route,
    when ``sr`` and every take are mono PCM16 at 88.2 kHz (what ffmpeg writes, mov_extraction.py:50-57): the data
    chunks are read back to back and are the samples.  Else each is read 8-byte aligned and ``nsf_convert_host``
    converts it to ``sr`` (88.2 kHz if None: decode() keeps the native rate), then to 88.2 kHz (load_audio.py:8-10)."""
    int16 = sr == REFERENCE_RATE and all(h[2:] == (nv.ENC_I16, 1, REFERENCE_RATE) for h in heads)
    sources = np.zeros(len(heads), dtype=nv.PCM_SOURCE)
    pos = 0
    for k, (_, nbytes, enc, channels, native) in enumerate(heads):
        channels = max(channels, 1)                                 # decode_wav reads 0 declared channels as mono
        frames = nbytes // (_ENC_BYTES[enc] * channels)
        sources[k] = (pos, frames, enc, channels, native, 0)
        pos += frames * _ENC_BYTES[enc] * channels
        if not int16:
            pos += -pos % 8                                         # converted takes start 8-byte aligned
    rate = sr if sr is not None else REFERENCE_RATE
    off = nv.convert_offsets(sources, rate, pos)
    mid = None
    if rate != REFERENCE_RATE:
        mid = nv.pcm_sources([(int(a) * 4, int(b - a), nv.ENC_F32, 1, rate) for a, b in zip(off[:-1], off[1:])])
        off = nv.convert_offsets(mid, REFERENCE_RATE, int(off[-1]) * 4)
    return _AudioPlan(int16, sources, np.diff(off), pos, rate, mid)


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


def _pandas_rows(path, drop, dtype):
    """The reference's read of a CSV (:112-114, :123): ``pd.read_csv`` minus the columns ``drop``, cast to dtype."""
    return np.ascontiguousarray(pd.read_csv(path).drop(columns=drop).values, dtype=dtype)


def _facial_rows(path, dtype):
    """The facial CSV minus Timecode / BlendshapeCount (:123), read by pandas."""
    return _pandas_rows(path, COLUMNS_TO_DROP, dtype)


def _read_texts(pool, paths, tag):
    """``(text, offsets, reads)``: the files ``paths`` back to back in the page-locked arena ``tag``, file k at
    ``text[offsets[k]:offsets[k + 1]]``, once the pool jobs ``reads`` are done."""
    off = _prefix([os.path.getsize(p) for p in paths])
    text = _engine.scratch_pinned(tag, max(int(off[-1]), 1)).view(np.uint8, (int(off[-1]),))
    return text, off, [pool.submit(_read_into, p, 0, text[off[k]:off[k + 1]]) for k, p in enumerate(paths)]


_BOM = b"\xef\xbb\xbf"


def _csv_header(head, drop):
    """Column names of a CSV whose first bytes are ``head``, or None when the device route does not take the file:
    the first line must be printable ASCII without quotes (a '\r' only before its '\n'), with unique, non-empty
    names that include every name in ``drop``.  pandas handles the rest (BOMs, quoting, renamed duplicates, the
    KeyError of a missing column)."""
    if not head or head[:1] in (b"\r", b"\n") or head.startswith(_BOM):
        return None
    nl = head.find(b"\n")
    line = head if nl < 0 else head[:nl]
    if line.endswith(b"\r"):
        line = line[:-1]
    if any(c < 0x20 or c >= 0x7f or c == 0x22 for c in line):
        return None
    names = line.decode("ascii").split(",")
    if "" in names or len(set(names)) != len(names) or any(d not in names for d in drop):
        return None
    return names


def _parse_csvs(eng, pool, paths, text, off, drop, dtype):
    """``[rows]`` of the files ``paths`` (read into ``text`` at ``off``), each ``_pandas_rows(path, drop, dtype)``:
    files with the same header share one ``Engine.parse_csv`` call; a file the device does not accept (its header,
    or a status bit) is read by pandas on ``pool``, so its result, or the exception it raises, is the reference's."""
    groups, out = {}, [None] * len(paths)
    for k in range(len(paths)):
        head = bytes(text[off[k]:min(off[k + 1], off[k] + 65536)])      # a longer header line goes to pandas
        names = _csv_header(head, drop) if b"\n" in head or len(head) == off[k + 1] - off[k] else None
        if names is not None:
            groups.setdefault(tuple(names), []).append(k)
    for names, ks in groups.items():
        kept = [n for n in names if n not in drop]
        out_col = [-1 if n in drop else kept.index(n) for n in names]
        if ks == list(range(len(paths))):
            t, t_off = text, off
        else:
            t = np.concatenate([text[off[k]:off[k + 1]] for k in ks])
            t_off = _prefix([off[k + 1] - off[k] for k in ks])
        rows, r_off, status = eng.parse_csv(t, t_off, len(names), out_col, dtype)
        for j, k in enumerate(ks):
            if not status[j]:
                out[k] = rows[r_off[j]:r_off[j + 1]]
    fallback = {k: pool.submit(_pandas_rows, paths[k], drop, dtype) for k in range(len(paths)) if out[k] is None}
    for k, job in fallback.items():
        out[k] = job.result()
    return out


_Take = namedtuple("_Take", "folder video wav cache_csv facial_csv path")


def _scan(root_dir, processed_folders, cache_format):
    """The takes ``process_folder`` would not skip (:72-79), in ``os.listdir`` order, minus ``processed_folders``."""
    takes = []
    for folder in os.listdir(root_dir):
        path = os.path.join(root_dir, folder)
        if not os.path.isdir(path) or folder in processed_folders:
            continue
        mov, mp4, wav, facial_csv, cache_csv, _ = find_files(path)
        video = mov or mp4
        if facial_csv and (video or wav or _cached_features_path(cache_csv, cache_format)):
            takes.append(_Take(folder, video, wav, cache_csv, facial_csv, path))
    return takes


def _partition(takes, rank, world):
    """This rank's take indices.  The partition weighs files every rank sees identically BEFORE any rank extracts
    audio (never on audio.wav, which another rank may be writing): the take's video, else its wav, else its cache."""
    if world <= 1:
        return list(range(len(takes)))
    from .. import shard

    def weight(t):
        for cand in (t.video, t.wav, t.cache_csv):
            if cand and os.path.exists(cand):
                return max(1, os.path.getsize(cand))
        return 1
    return shard.lpt_partition([weight(t) for t in takes], world)[rank]


def _classify(takes, mine, cache_format, pool):
    """``(loaded, cached_csv, extract)``: take -> pool job loading its ``.npy`` feature cache, take -> its CSV cache
    (parsed with the facial CSVs), and take -> the audio file to extract (``get_audio`` may run ffmpeg).  A take with
    none is dropped, as ``process_folder`` returns (None, None)."""
    loaded, cached_csv, extract = {}, {}, {}
    for i in mine:
        t = takes[i]
        cache_path = _cached_features_path(t.cache_csv, cache_format)
        if cache_path:
            print(f"Loading audio features from {cache_path}")
            if cache_path.endswith(".npy"):
                loaded[i] = pool.submit(_read_feature_cache, cache_path)
            else:
                cached_csv[i] = cache_path
            continue
        audio_path = get_audio(t.video, t.wav, t.path) if (t.video or t.wav) else None
        if audio_path:
            print(f"Extracting audio features from {audio_path}")
            extract[i] = audio_path
    return loaded, cached_csv, extract


def _read_audio(eng, pool, paths, sr, then):
    """``(pcm, offsets, then())``: the WAV files ``paths`` as packed PCM at 88.2 kHz (``_plan_audio``), int16 or float32
    in library-owned page-locked memory.  Headers, then data chunks are read on ``pool``; ``then()`` runs once the
    reads are queued, so what it submits runs behind them.  A take under 9 frames raises ``TypeError`` (:143)."""
    if not paths:
        return None, None, then()
    heads = list(pool.map(_wav_source, paths))
    plan = _plan_audio(heads, sr)
    loaded = [f"Loaded audio file '{p}' with sample rate {sr if sr is not None else h[4]}"
              for p, h in zip(paths, heads)]
    if not plan.int16:                          # the int16 route announces its takes after the length check
        print(*loaded, sep="\n")
    for n in plan.lengths:
        frames = eng.plan.guard_frames(n)
        if frames < MIN_FRAMES:                                            # extract_features.py:16-20 -> :143
            print(f"Audio file is too short: {frames} frames, required: {MIN_FRAMES} frames")
            raise TypeError("object of type 'NoneType' has no len()")
    if plan.int16:
        print(*loaded, sep="\n")
    off = _prefix(plan.lengths)
    sample = np.dtype(np.int16 if plan.int16 else np.float32)
    pcm = _engine.scratch_pinned("dataset_pcm", int(off[-1]) * sample.itemsize).view(sample, (int(off[-1]),))
    dst = pcm.view(np.uint8) if plan.int16 else \
        _engine.scratch_pinned("dataset_wav", max(plan.nbytes, 1)).view(np.uint8, (plan.nbytes,))
    reads = [pool.submit(_read_into, p, h[0], dst[s["byte_offset"]:][:s["frames"] * s["channels"] * _ENC_BYTES[h[2]]])
             for p, h, s in zip(paths, heads, plan.sources)]
    queued = then()
    for r in reads:
        r.result()
    if plan.mid is not None:
        n_mid = int(plan.mid["frames"].sum())
        y_mid = _engine.scratch_pinned("dataset_wav_mid", max(n_mid * 4, 1)).view(np.float32, (n_mid,))
        eng.convert_host(dst, plan.sources, plan.rate, out=y_mid)
        eng.convert_host(y_mid.view(np.uint8), plan.mid, REFERENCE_RATE, out=pcm)
    elif not plan.int16:
        eng.convert_host(dst, plan.sources, plan.rate, out=pcm)
    return pcm, off, queued


def _device_pass(eng, pcm, off, extract, loaded, facial, dtype, kw):
    """``(results, feats, roff)``: take -> augmented (audio, facial) rows, for the takes ``extract`` (PCM ``pcm`` at
    ``off``) and those with ``loaded`` rows; the feature rows extracted, packed in ``extract`` order at ``roff`` (None,
    None without takes to extract).  float32 with augmentation fuses extraction and augmentation in one
    ``nsf_extract_collect_host`` call; otherwise the extracted rows join the loaded ones in the collect pass."""
    results, rows, feats, roff = {}, dict(loaded), None, None
    augment = kw["include_fast"] or kw["include_slow"]
    if extract:
        roff = eng.row_offsets(off)
        f_off = _prefix([len(facial[i]) for i in extract])
        if dtype == np.float32 and augment and all(roff[k + 1] > roff[k] and len(facial[i])
                                                   for k, i in enumerate(extract)):
            f_cols = facial[extract[0]].shape[1]
            fac = _engine.scratch_pinned("dataset_facial", int(f_off[-1]) * f_cols * 4).view(
                np.float32, (int(f_off[-1]), f_cols))
            np.concatenate([facial[i] for i in extract], out=fac)
            o_off = eng.collect_rows(roff, f_off, **kw)
            # results go to ordinary (pageable) arrays the caller owns: the library stages the downloads through
            # its own page-locked arenas, which costs a host copy but not a cudaHostAlloc of ~300 MB per call
            out_a = np.empty((int(o_off[-1]), 256), dtype=np.float32)
            out_f = np.empty((int(o_off[-1]), f_cols), dtype=np.float32)
            feats = np.empty((int(roff[-1]), 256), dtype=np.float32)
            eng.extract_collect_host(pcm, off, fac, f_off, nv.PEAK_NORMALIZE, out_audio=out_a, out_facial=out_f,
                                     features_out=feats, **kw)
            for k, i in enumerate(extract):
                results[i] = (out_a[o_off[k]:o_off[k + 1]], out_f[o_off[k]:o_off[k + 1]])
        else:
            feats = eng.extract_host(pcm, off, nv.PEAK_NORMALIZE)
            for k, i in enumerate(extract):
                rows[i] = feats[roff[k]:roff[k + 1]]
    if rows:
        order = sorted(rows)
        rows_in = [np.ascontiguousarray(rows[i], dtype=dtype) for i in order]
        if augment and all(len(r) for r in rows_in) and all(len(facial[i]) for i in order):
            out_a, out_f, o_off = eng.collect_host(np.concatenate(rows_in, axis=0), _prefix([len(r) for r in rows_in]),
                                                   np.concatenate([facial[i] for i in order], axis=0),
                                                   _prefix([len(facial[i]) for i in order]), **kw)
            for k, i in enumerate(order):
                results[i] = (out_a[o_off[k]:o_off[k + 1]], out_f[o_off[k]:o_off[k + 1]])
        else:
            for r, i in zip(rows_in, order):
                results[i] = tuple(np.array(x) for x in collect_arrays(r, facial[i], **kw))
    return results, feats, roff


def _assemble(takes, mine, results, processed_folders):
    """``(examples, indices)`` in take order with ``facial[:, :61] *= 100`` (:68); records the folders (:24)."""
    examples, indices = [], []
    for i in mine:
        if i not in results:
            continue
        a, f = results[i]
        f[:, :61] *= 100
        examples.append((a, f))
        indices.append(i)
        processed_folders.add(takes[i].folder)
    return examples, indices


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

    t_start = time.perf_counter()
    timing = {}
    cache_format = _cache_format(cache_format)
    if dtype not in (np.float32, np.float64):
        raise ValueError("dtype must be numpy.float32 or numpy.float64")
    takes = _scan(root_dir, processed_folders, cache_format)
    mine = _partition(takes, rank, world)
    timing["scan"] = time.perf_counter() - t_start

    f_len, h_len = _engine.frame_params(REFERENCE_RATE)     # file-path mode always lands at 88.2 kHz
    eng = _engine.get_engine(REFERENCE_RATE, f_len, h_len, device=device)
    kw = dict(include_fast=include_fast, include_slow=include_slow, blend_boundaries=blend_boundaries,
              blend_frames=blend_frames)
    threads = io_threads or min(32, len(os.sched_getaffinity(0)) or 1)
    pool = ThreadPoolExecutor(max_workers=threads)
    try:
        t0 = time.perf_counter()
        loaded, cached_csv, extract = _classify(takes, mine, cache_format, pool)
        keep = [i for i in mine if i in loaded or i in cached_csv or i in extract]
        # the CSV texts are read into page-locked arenas behind the WAV payloads, then parsed on the device
        facial_paths, cache_paths = [takes[i].facial_csv for i in keep], list(cached_csv.values())
        pcm, off, (fac_text, cache_text) = _read_audio(eng, pool, list(extract.values()), sr, then=lambda: (
            _read_texts(pool, facial_paths, "dataset_facial_csv"), _read_texts(pool, cache_paths, "dataset_cache_csv")))
        timing["read_audio"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        for j in fac_text[2] + cache_text[2]:
            j.result()
        loaded = {i: j.result() for i, j in loaded.items()}
        timing["facial_csv_wait"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        facial = dict(zip(keep, _parse_csvs(eng, pool, facial_paths, *fac_text[:2], COLUMNS_TO_DROP, dtype)))
        loaded.update(zip(cached_csv, _parse_csvs(eng, pool, cache_paths, *cache_text[:2], [], dtype)))
        timing["parse_csv"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        extract = list(extract)
        results, feats, roff = _device_pass(eng, pcm, off, extract, loaded, facial, dtype, kw)
        timing["device"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        if extract:
            # every take's CSV in one device call; the pool only writes bytes
            text, t_off = eng.format_csv(feats, roff) if cache_format in ("csv", "both") else (None, None)
            list(pool.map(lambda k: _write_feature_cache(
                takes[extract[k]].cache_csv, feats[roff[k]:roff[k + 1]], cache_format,
                None if text is None else text[t_off[k]:t_off[k + 1]]), range(len(extract))))
        timing["write_cache"] = time.perf_counter() - t0
    finally:
        pool.shutdown(wait=True)
    examples, indices = _assemble(takes, mine, results, processed_folders)
    timing["total"] = time.perf_counter() - t_start
    last_timing.clear()
    last_timing.update(timing)
    return examples, indices

"""Generate ``tests/golden/*.npz`` by running the REFERENCE'S OWN .py files, unmodified.

Run in the build container only (``/root/reference`` does not exist on the GPU box):

    python oracle/make_golden.py

What it does
1. puts ``oracle/librosa_standin`` (librosa is un-installable here) and ``/root/reference`` on
   ``sys.path`` and imports ``utils.audio.extraction.extract_features`` and
   ``dataset.data_processing`` exactly as shipped;
2. runs them on the deterministic synthetic inputs of ``neurosync_trainer_lite_b200.synth`` and on
   the first seconds of the reference's own fixture ``dataset/test_set/audio.wav``;
3. asserts that ``oracle/feature_oracle.py`` (the restatement that travels to the GPU box)
   reproduces every output bit-for-bit;
4. writes small fixtures: full outputs for short clips, strided row samples for the 30 s clip.
"""
import contextlib
import io
import os
import sys
import tempfile
import wave

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = "/root/reference"
OUT = os.path.join(ROOT, "tests", "golden")

sys.path.insert(0, os.path.join(HERE, "librosa_standin"))
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)

import pandas as pd  # noqa: E402

from neurosync_trainer_lite_b200 import synth  # noqa: E402
from oracle import feature_oracle as fo  # noqa: E402

# the reference, verbatim
from utils.audio.extraction import extract_features as ref_ef  # noqa: E402
from utils.audio.extraction import extract_features_utils as ref_u  # noqa: E402
from dataset import data_processing as ref_dp  # noqa: E402
from dataset import dataset as ref_ds  # noqa: E402


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def same(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape and a.dtype == b.dtype, (what, a.shape, b.shape, a.dtype, b.dtype)
    assert np.array_equal(a, b, equal_nan=True), f"oracle restatement differs from reference: {what}"


def fingerprint(y):
    y = np.asarray(y)
    return np.array([y.size, float(np.sum(y.astype(np.float64))),
                     float(np.sum(np.abs(y.astype(np.float64))))])


def sample_rows(n):
    idx = np.unique(np.concatenate([np.arange(0, min(n, 24)), np.arange(max(0, n - 24), n),
                                    np.arange(0, n, 13)]))
    return idx.astype(np.int64)


def write_wav(path, pcm16, sr):
    with wave.open(path, "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(sr)
        w.writeframes(pcm16.astype("<i2").tobytes())


def main():
    os.makedirs(OUT, exist_ok=True)
    made = []

    # ---- A. array entry point, short clips: full input + full output --------------------------
    for name, sr, seconds, seed, kind in [
        ("voiced_2s_16k", 16000, 2.0, 3, "voiced"),
        ("gated_1s5_88k", 88200, 1.5, 5, "gated"),
        ("noise_0s7_88k", 88200, 0.7, 7, "noise"),
        ("voiced_1s_44k1_oddF", 44100, 1.0, 9, "voiced"),
        ("voiced_0s6_22k05_oddF", 22050, 0.6, 11, "voiced"),
    ]:
        y = synth.synth_clip(seconds, sr, seed=seed, kind=kind)
        F, H = fo.frame_params(sr)
        ref = ref_ef.extract_and_combine_features(y, sr, F, H)
        same(fo.extract_and_combine_features(y, sr, F, H), ref, name)
        mf, T = ref_u.extract_mfcc_features(y, sr, F, H)
        same(fo.mfcc_rows(y, sr, F, H)[0], mf, name + " mfcc")
        assert T == fo.hop_frames(len(y), F, H) and ref.shape[0] == fo.feature_rows(len(y), F, H)
        np.savez_compressed(os.path.join(OUT, name + ".npz"), y=y, sr=sr, F=F, H=H, T=T,
                            features=ref)
        made.append((name, ref.shape))

    # smoothing / no-autocorr / autocorr-with-deltas switches on one short clip
    y = synth.synth_clip(0.5, 88200, seed=21, kind="voiced")
    F, H = fo.frame_params(88200)
    sm = ref_ef.extract_and_combine_features(y, 88200, F, H, apply_smoothing=True)
    same(fo.extract_and_combine_features(y, 88200, F, H, apply_smoothing=True), sm, "smoothing")
    na = ref_ef.extract_and_combine_features(y, 88200, F, H, include_autocorr=False)
    same(fo.extract_and_combine_features(y, 88200, F, H, include_autocorr=False), na, "no-ac")
    acd = ref_u.extract_autocorrelation_features(y, 88200, F, H, include_deltas=True)
    same(fo.autocorr_rows(y, 88200, F, H, include_deltas=True), acd, "ac deltas")
    raw = ref_u.extract_overlapping_mfcc(y, 88200, 23, F, H, include_deltas=False,
                                         include_cepstral=False)
    same(fo.mfcc_block(y, 88200, F, H, include_deltas=False, include_cepstral=False), raw, "raw")
    np.savez_compressed(os.path.join(OUT, "switches_0s5_88k.npz"), y=y, sr=88200, F=F, H=H,
                        smoothed=sm, no_autocorr=na, autocorr_deltas=acd, raw_mfcc=raw)
    made.append(("switches_0s5_88k", sm.shape))

    # ---- B. C1: 30 s @ 88.2 kHz, seed 0 (BASELINE configs[0]); strided rows only ----------------
    y = synth.synth_clip(30.0, 88200, seed=0, kind="voiced")
    ref = ref_ef.extract_and_combine_features(y, 88200, 1470, 735)
    same(fo.extract_and_combine_features(y, 88200, 1470, 735), ref, "C1")
    assert ref.shape == (1801, 256) and ref.dtype == np.float64
    rows = sample_rows(ref.shape[0])
    np.savez_compressed(os.path.join(OUT, "c1_voiced_30s_88k.npz"), sr=88200, F=1470, H=735,
                        seconds=30.0, seed=0, shape=np.array(ref.shape), rows=rows,
                        features=ref[rows], input_fingerprint=fingerprint(y),
                        col_absmax=np.abs(ref).max(axis=0))
    made.append(("c1_voiced_30s_88k", ref.shape))
    c1_features = ref

    # ---- C. file / bytes entry points (WAV at the target rate -> no resampling) -----------------
    with tempfile.TemporaryDirectory() as td:
        raw16 = synth.to_int16_pcm(0.8 * synth.synth_clip(1.2, 88200, seed=13, kind="voiced"))
        p = os.path.join(td, "a.wav")
        write_wav(p, raw16, 88200)
        feats, yn = quiet(ref_ef.extract_audio_features, p, 88200)
        with open(p, "rb") as fh:
            blob = fh.read()
        feats_b, yn_b = quiet(ref_ef.extract_audio_features, blob, 88200, True)
        same(feats_b, feats, "bytes vs path")
        of, oy = fo.extract_audio_features_from_array(raw16.astype(np.float32) / np.float32(32768),
                                                      88200)
        same(of, feats, "file entry")
        same(oy, yn, "file entry y")
        raw16k = synth.to_int16_pcm(0.6 * synth.synth_clip(2.0, 16000, seed=14, kind="voiced"))
        blob16 = synth.wav_bytes(raw16k, 16000)
        f16, y16 = quiet(ref_ef.extract_audio_features, blob16, 16000, True)
        o16, oy16 = fo.extract_audio_features_from_array(
            raw16k.astype(np.float32) / np.float32(32768), 16000)
        same(o16, f16, "bytes 16k")
        same(oy16, y16, "bytes 16k y")
        # too short: 8 guard frames
        short = np.zeros(8 * 735 + 1469, dtype=np.int16)
        short[100] = 1000
        ps = os.path.join(td, "s.wav")
        write_wav(ps, short, 88200)
        assert quiet(ref_ef.extract_audio_features, ps, 88200) == (None, None)
        assert quiet(fo.extract_audio_features_from_array, short.astype(np.float32), 88200) == (None, None)
        # one file per rate: every golden file stays under 1 MB
        np.savez_compressed(os.path.join(OUT, "entry_points.npz"), pcm88=raw16, feats88=feats, y88=yn)
        np.savez_compressed(os.path.join(OUT, "entry_points_16k.npz"), pcm16=raw16k, feats16=f16, y16=y16)
        made.append(("entry_points", feats.shape))

        # ---- D. the reference's own fixture, first 3 s, native 44.1 kHz via from_bytes -----------
        with wave.open(os.path.join(REF, "dataset/test_set/audio.wav"), "rb") as w:
            assert w.getframerate() == 44100 and w.getnchannels() == 1 and w.getsampwidth() == 2
            w.setpos(44100 * 2)
            speech = np.frombuffer(w.readframes(44100 * 3), dtype="<i2").copy()
        fsp, ysp = quiet(ref_ef.extract_audio_features, synth.wav_bytes(speech, 44100), 44100, True)
        osp, _ = fo.extract_audio_features_from_array(speech.astype(np.float32) / np.float32(32768),
                                                      44100)
        same(osp, fsp, "speech")
        np.savez_compressed(os.path.join(OUT, "speech_3s_44k1.npz"), pcm=speech, sr=44100,
                            features=fsp)
        made.append(("speech_3s_44k1", fsp.shape))

        # ---- E. collect_features through the real CSV plumbing ----------------------------------
        facial = synth.synth_facial(1800, seed=0)
        cols = ["Timecode", "BlendshapeCount"] + [f"bs{i}" for i in range(61)]
        df = pd.DataFrame(np.hstack([np.zeros((1800, 2)), facial]), columns=cols)
        fcsv = os.path.join(td, "x_iPhone_cal.csv")
        df.to_csv(fcsv, index=False)
        facial_rt = pd.read_csv(fcsv).drop(columns=["Timecode", "BlendshapeCount"]).values
        acsv = os.path.join(td, "audio_features.csv")
        pd.DataFrame(c1_features).to_csv(acsv, index=False)
        cached = pd.read_csv(acsv).values
        shapes = {}
        for tag, kw in [("fast", dict()), ("fast_slow", dict(include_slow=True)),
                        ("noblend", dict(blend_boundaries=False)),
                        ("slow_only_b7", dict(include_fast=False, include_slow=True, blend_frames=7))]:
            a, f = quiet(ref_dp.collect_features, None, acsv, fcsv, 88200, **kw)
            oa, of_ = fo.collect_from_arrays(cached, facial_rt, **kw)
            same(oa, a, "collect audio " + tag)
            same(of_, f, "collect facial " + tag)
            assert a.shape[0] == fo.collected_rows(1800, **kw), (tag, a.shape)
            # rows around every version boundary / blend zone, plus a sparse stride
            extra = [k for b in (0, 1800, 1800 + 900, 2670, a.shape[0]) for k in range(b - 36, b + 6)
                     if 0 <= k < a.shape[0]]
            r = np.unique(np.concatenate([np.arange(0, a.shape[0], 97),
                                          np.array(extra, dtype=np.int64)]))
            # one file per setting: every golden file stays under 1 MB
            np.savez_compressed(os.path.join(OUT, f"collect_c3_{tag}.npz"), **{
                tag + "_rows": r, tag + "_shape": np.array(a.shape), tag + "_audio": a[r], tag + "_facial": f[r]})
            shapes[tag] = a.shape
        assert shapes["fast"] == (2670, 256) and shapes["fast_slow"] == (6239, 256)
        # facial rows are regenerated by the tests (synth_facial(1800, seed=0)); the CSV round trip
        # moves them by <= 1 ulp, far inside the test tolerance
        assert np.abs(facial_rt - facial).max() < 1e-15
        made.append(("collect_c3", shapes["fast"]))

    # ---- F. small known-answer tests of the augmentation helpers (SURVEY 8(c)) ------------------
    A = np.arange(10, dtype=np.float64).reshape(5, 2)
    B = 100 + np.arange(8, dtype=np.float64).reshape(4, 2)
    kat = dict(A=A, B=B,
               blend3=ref_dp.stack_with_blend([A, B], 3),
               blend30=ref_dp.stack_with_blend([A, B], 30),
               blend0=ref_dp.stack_with_blend([A, B], 0),
               slower=ref_dp.interpolate_slower(A),
               smooth=ref_dp.smooth_facial_data(A),
               smooth_feat=ref_u.smooth_features(A),
               reduce_odd=ref_u.reduce_features(np.arange(14, dtype=np.float64).reshape(2, 7)),
               reduce_even=ref_u.reduce_features(np.arange(12, dtype=np.float64).reshape(2, 6)))
    same(fo.stack_with_blend([A, B], 3), kat["blend3"], "blend3")
    same(fo.stack_with_blend([A, B], 30), kat["blend30"], "blend30")
    same(fo.stack_with_blend([A, B], 0), kat["blend0"], "blend0")
    same(fo.interpolate_slower(A), kat["slower"], "slower")
    same(fo.smooth_facial_data(A), kat["smooth"], "smooth")
    same(fo.smooth_rows(A), kat["smooth_feat"], "smooth_feat")
    same(fo.pair_reduce(np.arange(14, dtype=np.float64).reshape(2, 7)), kat["reduce_odd"], "red")
    same(fo.pair_reduce(np.arange(12, dtype=np.float64).reshape(2, 6)), kat["reduce_even"], "red")
    # row-count KATs (SURVEY 8(c)) straight from the reference
    counts = []
    for L in (14700, 14701, 15435, 16169, 7350, 8084, 8 * 735 + 1470, 8 * 735 + 1469):
        yk = synth.synth_clip(L / 88200.0, 88200, seed=L % 97, kind="noise")[:L]
        assert len(yk) == L
        n_guard = (L - 1470) // 735 + 1
        if n_guard < 9:
            counts.append((L, -1, -1))
            continue
        r = ref_ef.extract_and_combine_features(yk, 88200, 1470, 735)
        _, T = ref_u.extract_mfcc_features(yk, 88200, 1470, 735)
        counts.append((L, T, r.shape[0]))
        assert (T, r.shape[0]) == (fo.hop_frames(L, 1470, 735), fo.feature_rows(L, 1470, 735))
    kat["row_counts"] = np.array(counts, dtype=np.int64)
    # silence and DC (no NaN; autocorr exactly zero)
    z = ref_ef.extract_and_combine_features(np.zeros(88200, np.float32), 88200, 1470, 735)
    assert z.shape == (61, 256) and not np.isnan(z).any() and np.all(z == 0)
    dc = ref_ef.extract_and_combine_features(np.ones(88200, np.float32), 88200, 1470, 735)
    assert np.all(dc[:, 69:] == 0) and np.isfinite(dc).all()
    kat["dc_mfcc"] = dc[:, :69]
    imp = np.zeros(40 * 735, np.float32)
    imp[20 * 735] = 1.0
    ri = ref_u.extract_overlapping_autocorr(imp, 88200, 1470, 735)
    kat["impulse_nonzero_frames"] = np.nonzero(np.abs(ri).sum(axis=0))[0]
    # windowing of dataset.py:58-98 (the "next" consumer)
    cfg = dict(root_dir=".", sr=88200, frame_rate=60, micro_batch_size=128)
    ds = ref_ds.AudioFacialDataset.__new__(ref_ds.AudioFacialDataset)
    ds.micro_batch_size = 128
    ra = np.arange(300 * 4, dtype=np.float64).reshape(300, 4)
    rf = np.arange(300 * 3, dtype=np.float64).reshape(300, 3) * 0.5
    ex = ds.process_example(ra, rf)
    oex = fo.window_examples(ra, rf)
    assert len(ex) == len(oex) == 174
    for (a, f), (oa, of_) in zip(ex, oex):
        same(oa, a.numpy(), "window a")
        same(of_, f.numpy(), "window f")
    kat["window_n300_count"] = np.array(len(ex))
    kat["window_n300_last_a"] = ex[-1][0].numpy()
    kat["window_n256_count"] = np.array(len(ds.process_example(ra[:256], rf[:256])))
    del cfg
    np.savez_compressed(os.path.join(OUT, "kat.npz"), **kat)
    made.append(("kat", ()))

    for name, shape in made:
        p = os.path.join(OUT, name + ".npz")
        print(f"{name:28s} {str(shape):14s} {os.path.getsize(p) / 1024:8.1f} KiB")


if __name__ == "__main__":
    main()

"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle and the reference's golden
vectors.  Tolerances (float32 device arithmetic vs the reference's float64/float32 mix):

* frame / row counts, alignment, zero patterns: bit-exact;
* MFCC columns (0..22, CMVN'd, range about +-5):                       max-abs <= 1e-4
* delta, delta-delta columns (23..68, range about +-0.7):              max-abs <= 2e-5
* autocorrelation columns (69..255, range [-1, 1]):                    max-abs <= 2e-5
* collect_features augmentation in float64: bit-exact (same IEEE operation order as NumPy).

Measured (profiles/parity_r01.md, profiles/parity_r02.md): 2.9e-5 / 3.9e-6 / 3.4e-6, so the bounds sit
3-6x above the measurement - tight enough that a 2-product operand split (2e-4 on the MFCC block, 3e-5 on
the autocorrelation block) fails them.
"""
import io

import numpy as np
import pytest

from neurosync_trainer_lite_b200 import synth

pytestmark = pytest.mark.gpu

TOL_MFCC = 1e-4
TOL_DELTA = 2e-5
TOL_AC = 2e-5
SHORT = ["voiced_2s_16k", "gated_1s5_88k", "noise_0s7_88k", "voiced_1s_44k1_oddF",
         "voiced_0s6_22k05_oddF"]


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


@pytest.fixture(scope="module")
def ef(nv):
    from neurosync_trainer_lite_b200.utils.audio.extraction import extract_features
    return extract_features


@pytest.fixture(scope="module")
def efu(nv):
    from neurosync_trainer_lite_b200.utils.audio.extraction import extract_features_utils
    return extract_features_utils


@pytest.fixture(scope="module")
def dp(nv):
    from neurosync_trainer_lite_b200.dataset import data_processing
    return data_processing


def check_rows(got, want, n_mfcc_cols=69, tol_mfcc=TOL_MFCC, tol_ac=TOL_AC):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, (got.shape, want.shape)
    assert np.isfinite(got).all()
    if n_mfcc_cols:
        err = np.abs(got[:, :n_mfcc_cols] - want[:, :n_mfcc_cols]).max()
        assert err <= tol_mfcc, f"MFCC block max-abs error {err:.3e} > {tol_mfcc}"
    if n_mfcc_cols == 69:     # the default layout: delta / delta-delta columns have their own, tighter bound
        err = np.abs(got[:, 23:69] - want[:, 23:69]).max()
        assert err <= TOL_DELTA, f"delta block max-abs error {err:.3e} > {TOL_DELTA}"
    if got.shape[1] > n_mfcc_cols:
        err = np.abs(got[:, n_mfcc_cols:] - want[:, n_mfcc_cols:]).max()
        assert err <= tol_ac, f"autocorr block max-abs error {err:.3e} > {tol_ac}"


# ---- reference golden vectors through the reference-named API -------------------------------------
@pytest.mark.parametrize("name", SHORT)
def test_extract_and_combine_matches_reference_golden(name, golden, ef):
    g = golden(name)
    out = ef.extract_and_combine_features(g["y"], int(g["sr"]), int(g["F"]), int(g["H"]))
    assert out.dtype == np.float64
    check_rows(out, g["features"])


def test_simt_validation_path_agrees(golden, engine, nv):
    """The fp32 CUDA-core STFT (debug flag) and the tcgen05 STFT agree with each other and the oracle."""
    g = golden("gated_1s5_88k")
    eng = engine.get_engine(88200, 1470, 735)
    y = g["y"]
    a = eng.extract_host(y, [0, len(y)], nv.DEBUG_SIMT_DFT)
    b = eng.extract_host(y, [0, len(y)], 0)
    check_rows(a, g["features"])
    check_rows(b, g["features"])
    assert np.abs(a[:, :69] - b[:, :69]).max() <= TOL_MFCC


def test_fused_mel_epilogue_agrees_with_unfused_path(golden, engine, nv):
    """Persistent fused tcgen05 kernel (STFT -> power -> mel -> dB in the epilogue) vs the separate
    GEMM + mel kernels, on even / odd frame lengths, ragged multi-clip batches and tail tiles."""
    for name in ("gated_1s5_88k", "voiced_2s_16k", "voiced_1s_44k1_oddF", "noise_0s7_88k"):
        g = golden(name)
        eng = engine.get_engine(int(g["sr"]), int(g["F"]), int(g["H"]))
        y = g["y"]
        a = eng.extract_host(y, [0, len(y)], nv.NO_AUTOCORR)
        b = eng.extract_host(y, [0, len(y)], nv.NO_AUTOCORR | nv.DEBUG_UNFUSED_MEL)
        assert np.abs(a - g["features"][:, :69]).max() <= TOL_MFCC
        assert np.abs(b - g["features"][:, :69]).max() <= TOL_MFCC
        assert np.abs(a - b).max() <= 2e-4
    eng = engine.get_engine(88200, 1470, 735)
    clips = [synth.synth_clip(s, 88200, seed=i, kind=k) for i, (s, k) in
             enumerate([(0.9, "voiced"), (2.3, "gated"), (0.31, "noise"), (4.1, "voiced")])]
    packed, off = engine.pack_clips(clips)
    a = eng.extract_host(packed, off, nv.NO_AUTOCORR)
    b = eng.extract_host(packed, off, nv.NO_AUTOCORR | nv.DEBUG_UNFUSED_MEL)
    assert np.isfinite(a).all() and np.abs(a - b).max() <= 2e-4


def test_fma_autocorr_validation_path_agrees(golden, engine, nv):
    """The fp32-FMA autocorrelation (debug flag) and the mma.sync Hankel kernel agree with each other
    and with the reference, including odd frame lengths and the 16 kHz geometry."""
    for name in ("gated_1s5_88k", "voiced_2s_16k", "voiced_1s_44k1_oddF", "voiced_0s6_22k05_oddF"):
        g = golden(name)
        eng = engine.get_engine(int(g["sr"]), int(g["F"]), int(g["H"]))
        y = g["y"]
        a = eng.extract_host(y, [0, len(y)], nv.DEBUG_FMA_AUTOCORR | nv.NO_MFCC)
        b = eng.extract_host(y, [0, len(y)], nv.NO_MFCC)
        assert np.abs(a - g["features"][:, 69:]).max() <= TOL_AC
        assert np.abs(b - g["features"][:, 69:]).max() <= TOL_AC
        assert np.abs(a - b).max() <= TOL_AC


def test_switches(golden, ef, efu):
    g = golden("switches_0s5_88k")
    y, sr, F, H = g["y"], int(g["sr"]), int(g["F"]), int(g["H"])
    check_rows(ef.extract_and_combine_features(y, sr, F, H, apply_smoothing=True), g["smoothed"])
    na = ef.extract_and_combine_features(y, sr, F, H, include_autocorr=False)
    assert na.dtype == np.float32
    check_rows(na, g["no_autocorr"])
    acd = efu.extract_autocorrelation_features(y, sr, F, H, include_deltas=True)
    check_rows(acd, g["autocorr_deltas"], n_mfcc_cols=0)
    raw = efu.extract_overlapping_mfcc(y, sr, 23, F, H, include_deltas=False, include_cepstral=False)
    assert raw.shape == g["raw_mfcc"].shape
    # un-normalised MFCCs span about +-200: relative tolerance
    assert np.abs(raw - g["raw_mfcc"]).max() <= 2e-2


def test_c1_30s_clip(golden, ef):
    """BASELINE configs[0]: one 30 s clip @ 88.2 kHz; (1801, 256), sampled rows vs the reference."""
    g = golden("c1_voiced_30s_88k")
    y = synth.synth_clip(30.0, 88200, seed=0, kind="voiced")
    out = ef.extract_and_combine_features(y, 88200, 1470, 735)
    assert out.shape == (1801, 256)
    check_rows(out[g["rows"]], g["features"])


def test_entry_points_file_bytes_and_too_short(golden, ef, tmp_path, capsys):
    g = golden("entry_points")
    p = tmp_path / "a.wav"
    p.write_bytes(synth.wav_bytes(g["pcm88"], 88200))
    feats, y = ef.extract_audio_features(str(p), 88200)
    check_rows(feats, g["feats88"])
    np.testing.assert_array_equal(y, g["y88"])           # y / max|y| in float32: bit-exact
    assert y.dtype == np.float32
    fb, yb = ef.extract_audio_features(synth.wav_bytes(g["pcm88"], 88200), 88200, True)
    np.testing.assert_array_equal(fb, feats)
    g16 = golden("entry_points_16k")
    f16, y16 = ef.extract_audio_features(synth.wav_bytes(g16["pcm16"], 16000), 16000, True)
    check_rows(f16, g16["feats16"])
    np.testing.assert_array_equal(y16, g16["y16"])
    short = np.zeros(8 * 735 + 1469, dtype=np.int16)
    short[100] = 1000
    capsys.readouterr()
    assert ef.extract_audio_features(synth.wav_bytes(short, 88200), 88200, True) == (None, None)
    assert "Audio file is too short: 8 frames, required: 9 frames" in capsys.readouterr().out


def test_reference_speech_fixture(golden, ef):
    g = golden("speech_3s_44k1")
    feats, _ = ef.extract_audio_features(synth.wav_bytes(g["pcm"], 44100), 44100, True)
    check_rows(feats, g["features"])


# ---- known answers / edge cases ---------------------------------------------------------------------
def test_row_counts_bit_exact(golden, ef):
    for n, t, r in golden("kat")["row_counts"]:
        if t < 0:
            continue
        y = synth.synth_clip(int(n) / 88200.0, 88200, seed=int(n) % 97, kind="noise")[:int(n)]
        out = ef.extract_and_combine_features(y, 88200, 1470, 735)
        assert out.shape == (int(r), 256)


def test_silence_dc_impulse(golden, ef, efu):
    z = ef.extract_and_combine_features(np.zeros(88200, np.float32), 88200, 1470, 735)
    assert z.shape == (61, 256) and np.all(z == 0)
    dc = ef.extract_and_combine_features(np.ones(88200, np.float32), 88200, 1470, 735)
    assert np.all(dc[:, 69:] == 0) and np.isfinite(dc).all()
    assert np.abs(dc[:, :69] - golden("kat")["dc_mfcc"]).max() <= TOL_MFCC
    imp = np.zeros(40 * 735, np.float32)
    imp[20 * 735] = 1.0
    ac = efu.extract_overlapping_autocorr(imp, 88200, 1470, 735)
    assert ac.shape == (187, 41)
    np.testing.assert_array_equal(np.nonzero(np.abs(ac).sum(axis=0))[0],
                                  golden("kat")["impulse_nonzero_frames"])


@pytest.mark.parametrize("kind,sr,seconds", [("voiced", 88200, 0.31), ("noise", 16000, 0.4),
                                             ("gated", 88200, 2.2), ("voiced", 48000, 0.5),
                                             # long frames: F = 1600 (three autocorrelation pairs per block) and
                                             # F = 3200 (two pairs, two-pass fold kernel)
                                             ("voiced", 96000, 0.4), ("noise", 192000, 0.25)])
def test_against_oracle_seeded(kind, sr, seconds, oracle, ef):
    y = synth.synth_clip(seconds, sr, seed=77, kind=kind)
    F, H = oracle.frame_params(sr)
    check_rows(ef.extract_and_combine_features(y, sr, F, H),
               oracle.extract_and_combine_features(y, sr, F, H))


def test_batched_ragged_clips_equal_single_calls(engine, oracle, nv):
    """Ragged batch (odd/even T, different kinds) in ONE call == per-clip oracle; rows are packed."""
    lens = [14700, 14701, 15435, 16169, 7350 + 735 * 9, 44100, 30001]
    kinds = ["voiced", "noise", "gated", "voiced", "noise", "gated", "voiced"]
    clips = [synth.synth_clip(n / 88200.0 + 1e-4, 88200, seed=i, kind=k)[:n]
             for i, (n, k) in enumerate(zip(lens, kinds))]
    eng = engine.get_engine(88200, 1470, 735)
    packed, off = engine.pack_clips(clips)
    rows = eng.extract_host(packed, off)
    roff = eng.row_offsets(off)
    assert roff[-1] == sum(oracle.feature_rows(n, 1470, 735) for n in lens)
    for i, y in enumerate(clips):
        check_rows(rows[roff[i]:roff[i + 1]], oracle.extract_and_combine_features(y, 88200, 1470, 735))
    # int16 upload + on-device peak normalisation == host float path
    pcm16 = [synth.to_int16_pcm(0.7 * c) for c in clips]
    p16, off16 = engine.pack_clips(pcm16)
    rows16, y16 = eng.extract_host(p16, off16, nv.PEAK_NORMALIZE, want_y=True)
    for i, c in enumerate(pcm16):
        yn = oracle.peak_normalize(c.astype(np.float32) / np.float32(32768))
        np.testing.assert_array_equal(y16[off16[i]:off16[i + 1]], yn)
        check_rows(rows16[roff[i]:roff[i + 1]], oracle.extract_and_combine_features(yn, 88200, 1470, 735))


def test_device_resident_entry_point(engine, oracle):
    torch = pytest.importorskip("torch")
    clips = [synth.synth_clip(0.5, 88200, seed=i, kind="voiced") for i in range(3)]
    eng = engine.get_engine(88200, 1470, 735)
    packed, off = engine.pack_clips(clips)
    dev = torch.device("cuda", eng.device)
    out, _ = eng.extract_device(torch.from_numpy(packed).to(dev), off)
    torch.cuda.synchronize(dev)
    got = out.cpu().numpy()
    roff = eng.row_offsets(off)
    for i, y in enumerate(clips):
        check_rows(got[roff[i]:roff[i + 1]], oracle.extract_and_combine_features(y, 88200, 1470, 735))


def test_too_short_for_delta_is_an_error_not_garbage(engine, nv):
    eng = engine.get_engine(88200, 1470, 735)
    y = np.zeros(735 * 5, np.float32)
    with pytest.raises(nv.TooShortError):
        eng.extract_host(y, [0, len(y)])


# ---- utils API (channel-major helpers) ----------------------------------------------------------------
def test_utils_helpers_match_oracle(efu, oracle, golden):
    import sys, os
    rng = np.random.default_rng(5)
    x = rng.standard_normal((23, 41)).astype(np.float32)
    np.testing.assert_allclose(efu.cepstral_mean_variance_normalization(x), oracle.cmvn(x), atol=2e-6)
    np.testing.assert_allclose(efu.reduce_features(x), oracle.pair_reduce(x), atol=1e-7)
    np.testing.assert_allclose(efu.reduce_features(x[:, :40]), oracle.pair_reduce(x[:, :40]), atol=1e-7)
    k = golden("kat")
    np.testing.assert_array_equal(efu.smooth_features(k["A"]), k["smooth_feat"])
    lr = oracle._librosa()
    want = np.vstack([x, lr.feature.delta(x), lr.feature.delta(x, order=2)])
    np.testing.assert_allclose(efu.compute_autocorr_with_deltas(x), want, atol=2e-6)
    ac = rng.standard_normal((187, 12))
    ac[:, 0] = 1e-9
    ac[:, -1] = -1e-8
    fixed = efu.fix_edge_frames_autocorr(ac.copy())
    np.testing.assert_allclose(fixed, oracle.fix_edge_frames(ac.copy()), atol=1e-7)
    y = synth.synth_clip(0.4, 88200, seed=4, kind="voiced")
    rows, T = efu.extract_mfcc_features(y, 88200, 1470, 735)
    wrows, wT = oracle.mfcc_rows(y, 88200, 1470, 735)
    assert T == wT and rows.dtype == np.float32
    check_rows(rows, wrows)
    acb = efu.extract_overlapping_autocorr(y, 88200, 1470, 735)
    assert acb.dtype == np.float64
    assert np.abs(acb - oracle.autocorr_block(y, 88200, 1470, 735)).max() <= TOL_AC


# ---- collect_features family: float64, bit-exact ---------------------------------------------------------
def test_augmentation_kats_bit_exact(golden, dp):
    k = golden("kat")
    A, B = k["A"], k["B"]
    np.testing.assert_array_equal(dp.stack_with_blend([A, B], 3), k["blend3"])
    np.testing.assert_array_equal(dp.stack_with_blend([A, B], 30), k["blend30"])
    np.testing.assert_array_equal(dp.stack_with_blend([A, B], 0), k["blend0"])
    np.testing.assert_array_equal(dp.interpolate_slower(A), k["slower"])
    np.testing.assert_array_equal(dp.smooth_facial_data(A), k["smooth"])


@pytest.mark.parametrize("tag,kw", [("fast", {}), ("fast_slow", dict(include_slow=True)),
                                    ("noblend", dict(blend_boundaries=False)),
                                    ("slow_only_b7", dict(include_fast=False, include_slow=True,
                                                          blend_frames=7))])
def test_collect_matches_reference_golden(tag, kw, golden, dp, oracle):
    """C3 shapes: 1801 audio rows (oracle features of the C1 clip) + 1800 facial rows -> bit-exact."""
    g = golden("collect_c3_" + tag)
    y = synth.synth_clip(30.0, 88200, seed=0, kind="voiced")
    audio = oracle.extract_and_combine_features(y, 88200, 1470, 735)   # the checker makes the input
    facial = synth.synth_facial(1800, seed=0)
    a, f = dp.collect_arrays(audio, facial, **kw)
    assert a.shape == tuple(g[tag + "_shape"]) and a.dtype == np.float64
    r = g[tag + "_rows"]
    wa, wf = oracle.collect_from_arrays(audio, facial, **kw)
    np.testing.assert_array_equal(a, wa)
    np.testing.assert_array_equal(f, wf)
    # the golden rows came through the reference's CSV round trip (<= 1 ulp on the inputs)
    np.testing.assert_allclose(a[r], g[tag + "_audio"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(f[r], g[tag + "_facial"], rtol=0, atol=1e-12)


def test_collect_batch_ragged_float32_and_trim(dp, oracle):
    rng = np.random.default_rng(3)
    audio = [rng.standard_normal((n, 256)).astype(np.float32) for n in (40, 41, 75, 12, 1)]
    facial = [rng.uniform(0, 1, (n, 61)).astype(np.float32) for n in (44, 38, 75, 13, 1)]
    for kw in (dict(), dict(include_slow=True), dict(include_fast=False, include_slow=True,
                                                     blend_boundaries=False)):
        oa, of, off = dp.collect_batch(audio, facial, **kw)
        for i, (a, f) in enumerate(zip(audio, facial)):
            wa, wf = oracle.collect_from_arrays(a.astype(np.float64), f.astype(np.float64), **kw)
            assert off[i + 1] - off[i] == len(wa)
            np.testing.assert_allclose(oa[off[i]:off[i + 1]], wa, rtol=0, atol=1e-6)
            np.testing.assert_allclose(of[off[i]:off[i + 1]], wf, rtol=0, atol=1e-6)


def test_collect_features_with_csv_plumbing(tmp_path, dp, oracle):
    import pandas as pd
    take = tmp_path / "data" / "take_001"
    take.mkdir(parents=True)
    y = synth.synth_clip(3.0, 88200, seed=8, kind="voiced")
    pcm = synth.to_int16_pcm(0.9 * y)
    wav = take / "audio.wav"
    wav.write_bytes(synth.wav_bytes(pcm, 88200))
    facial = synth.synth_facial(178, seed=2)
    cols = ["Timecode", "BlendshapeCount"] + [f"bs{i}" for i in range(61)]
    fcsv = take / "take_iPhone_cal.csv"
    pd.DataFrame(np.hstack([np.zeros((178, 2)), facial]), columns=cols).to_csv(fcsv, index=False)
    cache = take / "audio_features.csv"
    a, f = dp.collect_features(str(wav), str(cache), str(fcsv), 88200)
    assert cache.exists() and a.shape[1] == 256 and f.shape[1] == 61 and len(a) == len(f)
    a2, f2 = dp.collect_features(None, str(cache), str(fcsv), 88200)        # cache hit
    np.testing.assert_allclose(a2, a, rtol=0, atol=1e-12)
    yn = oracle.peak_normalize(pcm.astype(np.float32) / np.float32(32768))
    feats = oracle.extract_and_combine_features(yn, 88200, 1470, 735)
    facial_rt = pd.read_csv(fcsv).drop(columns=cols[:2]).values
    wa, wf = oracle.collect_from_arrays(feats, facial_rt)
    assert a.shape == wa.shape
    assert np.abs(a[:, :69] - wa[:, :69]).max() <= TOL_MFCC
    assert np.abs(a[:, 69:] - wa[:, 69:]).max() <= TOL_AC
    np.testing.assert_array_equal(f, wf)
    # binary cache extension (SURVEY 8(f)-3): float32 .npy beside the CSV path, CSV still wins if present
    take2 = tmp_path / "data2" / "take_002"
    take2.mkdir(parents=True)
    (take2 / "audio.wav").write_bytes(synth.wav_bytes(pcm, 88200))
    a3, _ = dp.collect_features(str(take2 / "audio.wav"), str(take2 / "audio_features.csv"), str(fcsv), 88200,
                                cache_format="npy")
    assert (take2 / "audio_features.npy").exists() and not (take2 / "audio_features.csv").exists()
    a4, _ = dp.collect_features(None, str(take2 / "audio_features.csv"), str(fcsv), 88200, cache_format="npy")
    np.testing.assert_allclose(a4, a3, rtol=0, atol=1e-6)                   # float32 cache
    np.testing.assert_allclose(a3, a, rtol=0, atol=1e-12)
    done = set()
    ex = dp.load_data_per_folder(str(tmp_path / "data"), 88200, done)       # the reference's loop, float64
    assert len(ex) == 1 and done == {"take_001"}
    np.testing.assert_allclose(ex[0][0], a, rtol=0, atol=1e-12)
    np.testing.assert_allclose(ex[0][1], wf * 100, rtol=1e-15, atol=0)      # facial[:, :61] *= 100
    ex32 = dp.load_data(str(tmp_path / "data"), 88200, set())               # batched float32 builder, CSV cache hit
    assert len(ex32) == 1 and ex32[0][0].dtype == np.float32
    np.testing.assert_allclose(ex32[0][0], a, rtol=0, atol=2e-6)
    np.testing.assert_allclose(ex32[0][1], wf * 100, rtol=3e-7, atol=0)


def test_batched_dataset_builder_equals_per_folder_builder(tmp_path, dp):
    """load_data_batched (one extraction batch + one augmentation batch, optional clip sharding) gives
    the same examples, in os.listdir order, as the reference-shaped load_data."""
    import pandas as pd
    cols = ["Timecode", "BlendshapeCount"] + [f"bs{i}" for i in range(61)]
    for root in ("a", "b"):
        for k, (secs, rows) in enumerate([(2.0, 118), (3.1, 190), (1.4, 80)]):
            take = tmp_path / root / f"take_{k:03d}"
            take.mkdir(parents=True)
            y = synth.synth_clip(secs, 88200, seed=40 + k, kind=("voiced", "gated", "noise")[k])
            (take / "audio.wav").write_bytes(synth.wav_bytes(synth.to_int16_pcm(0.8 * y), 88200))
            pd.DataFrame(np.hstack([np.zeros((rows, 2)), synth.synth_facial(rows, seed=k)]),
                         columns=cols).to_csv(take / f"t{k}_iPhone_cal.csv", index=False)
    ref = dp.load_data_per_folder(str(tmp_path / "a"), 88200, set())       # process_folder per take, float64
    done = set()
    got, order = dp.load_data_batched(str(tmp_path / "b"), 88200, done, dtype=np.float64)
    assert len(ref) == len(got) == 3 and len(done) == 3 and order == [0, 1, 2]
    # os.listdir order is the same for both roots (same names), so examples pair up; the float64 mode runs the
    # same float64 augmentation kernel on the same float32 features: bit-identical
    for (ra, rf), (ga, gf) in zip(ref, got):
        assert ra.shape == ga.shape and rf.shape == gf.shape and ga.dtype == np.float64
        np.testing.assert_array_equal(ga, ra)
        np.testing.assert_array_equal(gf, rf)
    # default float32 mode = what load_data() returns: fused extract + collect from page-locked int16 PCM
    for p in (tmp_path / "b").glob("*/audio_features.csv"):
        p.unlink()
    done32 = set()
    got32 = dp.load_data(str(tmp_path / "b"), 88200, done32)
    assert len(got32) == 3 and len(done32) == 3
    assert all((tmp_path / "b" / f"take_{k:03d}" / "audio_features.csv").exists() for k in range(3))   # cache side effect
    for (ra, rf), (ga, gf) in zip(ref, got32):
        assert ga.dtype == np.float32 and gf.dtype == np.float32 and ra.shape == ga.shape and rf.shape == gf.shape
        np.testing.assert_allclose(ga, ra, rtol=0, atol=2e-6)     # float32 cross-fades of values in about +-5
        np.testing.assert_allclose(gf, rf, rtol=3e-7, atol=1e-5)
    # the cache written by the float32 builder holds the un-augmented rows the per-folder builder cached
    import pandas as pd2
    ca = pd2.read_csv(tmp_path / "a" / "take_001" / "audio_features.csv").values
    cb = pd2.read_csv(tmp_path / "b" / "take_001" / "audio_features.csv").values
    np.testing.assert_array_equal(ca, cb)
    # sharded over two "ranks": union of the shards == the full list, positions returned; a rank touches only
    # its own takes
    for p in (tmp_path / "b").glob("*/audio_features.csv"):
        p.unlink()
    parts = [dp.load_data_batched(str(tmp_path / "b"), 88200, set(), rank=r, world=2, dtype=np.float64)
             for r in range(2)]
    seen = sorted(i for _, idx in parts for i in idx)
    assert seen == [0, 1, 2]
    for ex, idx in parts:
        for (ga, gf), i in zip(ex, idx):
            np.testing.assert_array_equal(ga, ref[i][0])
    # a take under 9 frames fails where the reference fails (TypeError from len(None))
    short = tmp_path / "c" / "take_000"
    short.mkdir(parents=True)
    (short / "audio.wav").write_bytes(synth.wav_bytes(np.zeros(5000, np.int16), 88200))
    pd.DataFrame(np.zeros((10, 63)), columns=cols).to_csv(short / "s_iPhone_cal.csv", index=False)
    with pytest.raises(TypeError):
        dp.load_data(str(tmp_path / "c"), 88200, set())
    with pytest.raises(TypeError):
        dp.load_data_per_folder(str(tmp_path / "c"), 88200, set())


def test_dataset_windows_match_reference_semantics(golden, nv):
    from neurosync_trainer_lite_b200.dataset.dataset import AudioFacialDataset
    k = golden("kat")
    ds = AudioFacialDataset.__new__(AudioFacialDataset)
    ds.micro_batch_size = 128
    ra = np.arange(300 * 4, dtype=np.float64).reshape(300, 4)
    rf = np.arange(300 * 3, dtype=np.float64).reshape(300, 3) * 0.5
    ex = ds.process_example(ra, rf)
    assert len(ex) == int(k["window_n300_count"]) == 174
    np.testing.assert_array_equal(ex[-1][0].numpy(), k["window_n300_last_a"])
    assert len(ds.process_example(ra[:256], rf[:256])) == int(k["window_n256_count"])
    with pytest.raises(ValueError):
        ds.process_example(ra[:121], rf[:121])


# ---- size-independent properties at full size ---------------------------------------------------------------
def test_properties_at_c2_scale(engine, nv):
    """60 x 30 s @ 88.2 kHz in one batch: row counts, lag-0 normalisation bound, per-clip CMVN
    statistics, batch == single-clip determinism, amplitude invariance of the peak-normalised path."""
    eng = engine.get_engine(88200, 1470, 735)
    base = [synth.synth_clip(30.0, 88200, seed=s, kind=("voiced", "noise", "gated")[s % 3]) for s in range(6)]
    clips = [base[i % 6] for i in range(60)]
    packed, off = engine.pack_clips(clips)
    rows = eng.extract_host(packed, off)
    roff = eng.row_offsets(off)
    assert rows.shape == (60 * 1801, 256) and np.isfinite(rows).all()
    assert np.abs(rows[:, 69:]).max() <= 1.0 + 1e-5            # |r[l] / r[0]| <= 1 (Cauchy-Schwarz)
    for i in range(6, 60):                                       # identical clips -> identical rows
        np.testing.assert_array_equal(rows[roff[i]:roff[i + 1]], rows[roff[i % 6]:roff[i % 6 + 1]])
    single = eng.extract_host(base[1], [0, len(base[1])])
    np.testing.assert_array_equal(single, rows[roff[1]:roff[2]])
    # scaling the PCM does not change peak-normalised features
    a = eng.extract_host(base[0] * np.float32(0.25), [0, len(base[0])], nv.PEAK_NORMALIZE)
    b = eng.extract_host(base[0], [0, len(base[0])], nv.PEAK_NORMALIZE)
    np.testing.assert_array_equal(a, b)
    # CMVN: un-reduced MFCC columns have zero mean / unit variance per clip
    t = eng.extract_host(base[2], [0, len(base[2])], nv.NO_AUTOCORR | nv.NO_REDUCE | nv.NO_DELTAS)
    assert np.abs(t.mean(axis=0, dtype=np.float64)).max() < 1e-4
    assert np.abs(t.std(axis=0, dtype=np.float64) - 1).max() < 1e-4


def test_collect_properties_at_c4_rank_scale(engine, oracle):
    """One rank's share of C4 (60 clips x 1801 feature rows + 1800 facial rows, fast + slow + blend(30)):
    row counts of SURVEY section 8 (6239 per clip), float64 bit-exactness against the oracle on sampled clips,
    cross-fade end points, and that identical inputs give identical outputs wherever they sit in the batch."""
    eng = engine.get_engine(88200, 1470, 735)
    rng = np.random.default_rng(5)
    base_a = [rng.standard_normal((1801, 256)) for _ in range(3)]
    base_f = [rng.uniform(0, 1, (1800, 61)) for _ in range(3)]
    n = 60
    audio = np.concatenate([base_a[i % 3] for i in range(n)])
    facial = np.concatenate([base_f[i % 3] for i in range(n)])
    a_off = np.arange(n + 1, dtype=np.int64) * 1801
    f_off = np.arange(n + 1, dtype=np.int64) * 1800
    oa, of, o_off = eng.collect_host(audio, a_off, facial, f_off, True, True, True, 30)
    assert np.array_equal(np.diff(o_off), np.full(n, 6239))                 # 2670 + 3599 - 30
    assert oa.shape == (n * 6239, 256) and of.shape == (n * 6239, 61)
    for i in (0, 1, 2):
        wa, wf = oracle.collect_from_arrays(base_a[i], base_f[i], True, True, True, 30)
        np.testing.assert_array_equal(oa[o_off[i]:o_off[i + 1]], wa)
        np.testing.assert_array_equal(of[o_off[i]:o_off[i + 1]], wf)
    for i in range(3, n):                                                     # position independence
        np.testing.assert_array_equal(oa[o_off[i]:o_off[i + 1]], oa[o_off[i % 3]:o_off[i % 3 + 1]])
    # first blended row is purely the original stream, last blended row purely the next one (linspace ends)
    trimmed = base_a[0][:1800]                                                # centre trim of 1801 vs 1800: diff 1 -> left 0
    np.testing.assert_array_equal(oa[:1770], trimmed[:1770])
    np.testing.assert_array_equal(oa[1770], trimmed[1770])


def test_properties_at_c5_scale(engine, oracle):
    """C5: 10 000 clips x 2 s @ 16 kHz in ONE batched call: 121 rows per clip, finite, bounded
    autocorrelation, identical clips -> identical rows, sampled clips against the oracle."""
    eng = engine.get_engine(16000, 266, 133)
    base = [synth.synth_clip(2.0, 16000, seed=40 + s, kind=("voiced", "noise", "gated", "voiced")[s % 4]) for s in range(8)]
    n = 10000
    packed, off = engine.pack_clips([base[i % 8] for i in range(n)])
    rows = eng.extract_host(packed, off)
    assert rows.shape == (n * 121, 256) and np.isfinite(rows).all()
    assert np.abs(rows[:, 69:]).max() <= 1.0 + 1e-5
    r = rows.reshape(n, 121, 256)
    for s in range(8):
        assert np.array_equal(r[s::8], np.broadcast_to(r[s], r[s::8].shape))
    for s in (0, 2, 5):
        want = oracle.extract_and_combine_features(base[s], 16000, 266, 133)
        d = np.abs(r[s] - want)
        assert d[:, :69].max() < 1e-3 and d[:, 69:].max() < 2e-5


def test_fused_extract_collect_equals_two_calls(engine, nv):
    """nsf_extract_collect_host (features stay on the device) == nsf_extract_host followed by nsf_collect_host,
    bit for bit in float32, on a ragged batch that spans several pipeline groups."""
    eng = engine.get_engine(88200, 1470, 735)
    secs = [0.9, 2.3, 0.4, 31.0, 1.7, 30.0, 12.0, 30.5, 29.0, 3.1]          # > 24 Mi samples in total: 2+ groups
    clips = [synth.synth_clip(s, 88200, seed=60 + i, kind=("voiced", "gated", "noise")[i % 3]) for i, s in enumerate(secs)]
    packed, off = engine.pack_clips(clips)
    roff = eng.row_offsets(off)
    n_f = [int(roff[i + 1] - roff[i]) + (i % 3) - 1 for i in range(len(clips))]   # facial rows: R-1, R, R+1
    facial = np.concatenate([synth.synth_facial(n, seed=i) for i, n in enumerate(n_f)]).astype(np.float32)
    f_off = np.concatenate([[0], np.cumsum(n_f)]).astype(np.int64)
    for kw in (dict(include_fast=True, include_slow=False), dict(include_fast=True, include_slow=True),
               dict(include_fast=False, include_slow=False, blend_boundaries=False)):
        rows = eng.extract_host(packed, off)
        wa, wf, wo = eng.collect_host(rows, roff, facial, f_off, blend_frames=30, **kw)
        ga, gf, go = eng.extract_collect_host(packed, off, facial, f_off, blend_frames=30, **kw)
        assert np.array_equal(go, wo)
        np.testing.assert_array_equal(ga, wa)
        np.testing.assert_array_equal(gf, wf)


def test_dct_kernels_agree(engine, tmp_path):
    """Three DCT kernels: k_dct_mma (default: tensor-pipe, split fp16), k_dct_const (NSF_DCT_CONST: coefficients as a
    kernel parameter, uniform-register FFMA operands) and k_dct_rows (NSF_DCT_SMEM: shared-memory coefficients).  The
    two FFMA kernels keep one accumulation order: bit-identical feature matrices.  The MMA kernel sums in another order
    and from split operands: MFCC / delta columns within 2e-5 / 5e-6 of them, autocorrelation columns identical.  The
    environment switches are read once per process, so the FFMA kernels run in child processes."""
    import os
    import subprocess
    import sys
    rng = np.random.default_rng(77)
    lens = [88200 * 2 + 311, 9 * 735 + 5, 88200 + 1, 40000, 735 * 33, 735 * 64 + 1470]   # tiles straddle clips
    clips = [synth.synth_clip(n / 88200.0 + 0.01, 88200, seed=int(rng.integers(1 << 30)),
                              kind=("voiced", "gated", "noise")[i % 3])[:n] for i, n in enumerate(lens)]
    y = np.concatenate(clips).astype(np.float32)
    off = np.concatenate([[0], np.cumsum([len(c) for c in clips])]).astype(np.int64)
    np.save(tmp_path / "y.npy", y)
    np.save(tmp_path / "off.npy", off)
    got = engine.get_engine(88200, 1470, 735).extract_host(y, off, 0)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    refs = {}
    for tag in ("NSF_DCT_CONST", "NSF_DCT_SMEM"):
        out = tmp_path / (tag + ".npy")
        code = ("import sys, numpy as np; sys.path.insert(0, %r)\n"
                "from neurosync_trainer_lite_b200 import engine\n"
                "y, off = np.load(%r), np.load(%r)\n"
                "np.save(%r, engine.get_engine(88200, 1470, 735).extract_host(y, off, 0))\n"
                % (root, str(tmp_path / "y.npy"), str(tmp_path / "off.npy"), str(out)))
        subprocess.run([sys.executable, "-c", code], check=True, env=dict(os.environ, **{tag: "1"}), timeout=600)
        refs[tag] = np.load(out)
    want = refs["NSF_DCT_CONST"]
    assert got.shape == want.shape and got.shape[0] > 0
    assert np.array_equal(want, refs["NSF_DCT_SMEM"])
    assert np.array_equal(got[:, 69:], want[:, 69:])
    d = np.abs(got - want)
    assert d[:, :23].max() <= 2e-5 and d[:, 23:69].max() <= 5e-6, (d[:, :23].max(), d[:, 23:69].max())

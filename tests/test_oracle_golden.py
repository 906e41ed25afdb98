"""The travelling oracle (oracle/feature_oracle.py) against the vectors the REFERENCE produced.

tests/golden/*.npz were written by oracle/make_golden.py, which ran the reference's own files from
/root/reference and asserted bit-equality with the oracle at generation time.  Replaying them here
(and on the GPU box, where /root/reference does not exist) guards against drift of the oracle, of
numpy/scipy, or of the synthetic generators.
"""
import numpy as np
import pytest

from neurosync_trainer_lite_b200 import synth

SHORT = ["voiced_2s_16k", "gated_1s5_88k", "noise_0s7_88k", "voiced_1s_44k1_oddF",
         "voiced_0s6_22k05_oddF"]


@pytest.mark.parametrize("name", SHORT)
def test_short_clips_bit_exact(name, golden, oracle):
    g = golden(name)
    out = oracle.extract_and_combine_features(g["y"], int(g["sr"]), int(g["F"]), int(g["H"]))
    assert out.dtype == np.float64 and out.shape == g["features"].shape
    np.testing.assert_array_equal(out, g["features"])
    assert oracle.hop_frames(len(g["y"]), int(g["F"]), int(g["H"])) == int(g["T"])


def test_switches(golden, oracle):
    g = golden("switches_0s5_88k")
    y, sr, F, H = g["y"], int(g["sr"]), int(g["F"]), int(g["H"])
    np.testing.assert_array_equal(
        oracle.extract_and_combine_features(y, sr, F, H, apply_smoothing=True), g["smoothed"])
    np.testing.assert_array_equal(
        oracle.extract_and_combine_features(y, sr, F, H, include_autocorr=False), g["no_autocorr"])
    np.testing.assert_array_equal(oracle.autocorr_rows(y, sr, F, H, include_deltas=True),
                                  g["autocorr_deltas"])
    np.testing.assert_array_equal(
        oracle.mfcc_block(y, sr, F, H, include_deltas=False, include_cepstral=False), g["raw_mfcc"])


def test_c1_30s(golden, oracle):
    """BASELINE configs[0]: one 30 s clip @ 88.2 kHz through the CPU path."""
    g = golden("c1_voiced_30s_88k")
    y = synth.synth_clip(30.0, 88200, seed=0, kind="voiced")
    fp = g["input_fingerprint"]
    assert y.size == int(fp[0])
    # libm differences between hosts may move single samples by an ulp; the fingerprint is loose
    assert abs(float(np.sum(y.astype(np.float64))) - fp[1]) < 1e-2
    out = oracle.extract_and_combine_features(y, 88200, 1470, 735)
    assert out.shape == tuple(g["shape"]) == (1801, 256)
    np.testing.assert_allclose(out[g["rows"]], g["features"], rtol=0, atol=5e-5)


def test_entry_points(golden, oracle):
    g = golden("entry_points")
    f, y = oracle.extract_audio_features_from_array(
        g["pcm88"].astype(np.float32) / np.float32(32768), 88200)
    np.testing.assert_array_equal(f, g["feats88"])
    np.testing.assert_array_equal(y, g["y88"])
    g = golden("entry_points_16k")
    f, y = oracle.extract_audio_features_from_array(
        g["pcm16"].astype(np.float32) / np.float32(32768), 16000)
    np.testing.assert_array_equal(f, g["feats16"])
    np.testing.assert_array_equal(y, g["y16"])


def test_reference_speech_fixture(golden, oracle):
    """3 s of the reference's own dataset/test_set/audio.wav at its native 44.1 kHz (odd F)."""
    g = golden("speech_3s_44k1")
    f, _ = oracle.extract_audio_features_from_array(
        g["pcm"].astype(np.float32) / np.float32(32768), 44100)
    np.testing.assert_array_equal(f, g["features"])


def test_too_short_returns_none(oracle, capsys):
    y = np.zeros(8 * 735 + 1469, np.float32)
    y[5] = 1
    assert oracle.extract_audio_features_from_array(y, 88200) == (None, None)
    assert "Audio file is too short: 8 frames, required: 9 frames" in capsys.readouterr().out


def test_row_count_kats(golden, oracle):
    for L, T, R in golden("kat")["row_counts"]:
        if T < 0:
            assert oracle.guard_frames(int(L), 1470, 735) < 9
        else:
            assert oracle.hop_frames(int(L), 1470, 735) == T
            assert oracle.feature_rows(int(L), 1470, 735) == R
    assert oracle.frame_params(88200) == (1470, 735)
    assert oracle.frame_params(16000) == (266, 133)
    assert oracle.frame_params(44100) == (735, 367)
    assert oracle.frame_params(22050) == (367, 183)


def test_silence_dc_impulse(golden, oracle):
    z = oracle.extract_and_combine_features(np.zeros(88200, np.float32), 88200, 1470, 735)
    assert z.shape == (61, 256) and np.all(z == 0)
    dc = oracle.extract_and_combine_features(np.ones(88200, np.float32), 88200, 1470, 735)
    assert np.all(dc[:, 69:] == 0)
    np.testing.assert_array_equal(dc[:, :69], golden("kat")["dc_mfcc"])
    imp = np.zeros(40 * 735, np.float32)
    imp[20 * 735] = 1.0
    ac = oracle.autocorr_block(imp, 88200, 1470, 735)
    np.testing.assert_array_equal(np.nonzero(np.abs(ac).sum(axis=0))[0],
                                  golden("kat")["impulse_nonzero_frames"])


def test_augmentation_kats(golden, oracle):
    k = golden("kat")
    A, B = k["A"], k["B"]
    np.testing.assert_array_equal(oracle.stack_with_blend([A, B], 3), k["blend3"])
    np.testing.assert_array_equal(k["blend3"][:, 0], [0, 2, 4, 54, 104, 106])
    np.testing.assert_array_equal(oracle.stack_with_blend([A, B], 30), k["blend30"])
    assert k["blend30"].shape == (5, 2)
    np.testing.assert_array_equal(oracle.stack_with_blend([A, B], 0), k["blend0"])
    np.testing.assert_array_equal(oracle.interpolate_slower(A), k["slower"])
    np.testing.assert_array_equal(k["slower"][:, 0], np.arange(9))
    np.testing.assert_array_equal(oracle.smooth_facial_data(A), k["smooth"])
    np.testing.assert_array_equal(oracle.smooth_rows(A), k["smooth_feat"])
    np.testing.assert_array_equal(oracle.pair_reduce(np.arange(14.).reshape(2, 7)), k["reduce_odd"])
    np.testing.assert_array_equal(oracle.pair_reduce(np.arange(12.).reshape(2, 6)), k["reduce_even"])


def test_collect_c3(golden, oracle):
    """configs[2]/[3] shapes: 30 s + 1800 facial rows -> 2670 (fast) / 6239 (fast+slow) rows."""
    y = synth.synth_clip(30.0, 88200, seed=0, kind="voiced")
    feats = oracle.extract_and_combine_features(y, 88200, 1470, 735)
    facial = synth.synth_facial(1800, seed=0)
    for tag, kw in [("fast", {}), ("fast_slow", dict(include_slow=True)),
                    ("noblend", dict(blend_boundaries=False)),
                    ("slow_only_b7", dict(include_fast=False, include_slow=True, blend_frames=7))]:
        g = golden("collect_c3_" + tag)
        a, f = oracle.collect_from_arrays(feats, facial, **kw)
        assert a.shape == tuple(g[tag + "_shape"]) and f.shape == (a.shape[0], 61)
        assert a.shape[0] == oracle.collected_rows(1800, **kw)
        r = g[tag + "_rows"]
        np.testing.assert_allclose(a[r], g[tag + "_audio"], rtol=0, atol=5e-5)
        np.testing.assert_allclose(f[r], g[tag + "_facial"], rtol=0, atol=1e-12)
    assert tuple(golden("collect_c3_fast")["fast_shape"]) == (2670, 256)
    assert tuple(golden("collect_c3_fast_slow")["fast_slow_shape"]) == (6239, 256)


def test_windowing_kats(golden, oracle):
    k = golden("kat")
    ra = np.arange(300 * 4, dtype=np.float64).reshape(300, 4)
    rf = np.arange(300 * 3, dtype=np.float64).reshape(300, 3) * 0.5
    ex = oracle.window_examples(ra, rf)
    assert len(ex) == int(k["window_n300_count"]) == 174
    np.testing.assert_array_equal(ex[-1][0], k["window_n300_last_a"])
    np.testing.assert_array_equal(ex[-1][0], ex[-2][0])  # the duplicated last window
    assert len(oracle.window_examples(ra[:256], rf[:256])) == int(k["window_n256_count"]) == 129


# the reference returned identical arrays for these knobs on both clips: autocorr_knobs.npz stores them once
KNOB_STORED_AS = {"trim": "nopad", "edge_trim": "nopad"}


@pytest.mark.parametrize("knob,kw", [("nopad", dict(pad_signal=False)), ("constant", dict(padding_mode="constant")),
                                     ("edge", dict(padding_mode="edge")), ("symmetric", dict(padding_mode="symmetric")),
                                     ("trim", dict(trim_padded=True)),
                                     ("edge_trim", dict(padding_mode="edge", trim_padded=True))])
def test_autocorr_knobs_restatement_is_bit_identical_to_the_reference_vectors(knob, kw, golden, oracle):
    """tests/golden/autocorr_knobs.npz comes from the reference's own extract_overlapping_autocorr
    (oracle/make_golden_knobs.py); the restatement must reproduce every knob setting bit for bit."""
    g = golden("autocorr_knobs")
    for clip in ("a", "b"):
        y, sr = g[f"{clip}_y"], int(g[f"{clip}_sr"])
        F, H = oracle.frame_params(sr)
        got = oracle.autocorr_block(y, sr, F, H, **kw)
        assert got.dtype == np.float64 and np.array_equal(got, g[f"{clip}_{KNOB_STORED_AS.get(knob, knob)}"])
    assert np.array_equal(oracle.fix_edge_frames(g["thr_in"].copy(), zero_threshold=0.5), g["thr_out"])

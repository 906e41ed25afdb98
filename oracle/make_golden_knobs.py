"""Golden vectors for the non-default knobs of the autocorrelation branch
(``extract_overlapping_autocorr(pad_signal, padding_mode, trim_padded)`` and
``fix_edge_frames_autocorr(zero_threshold)``, reference utils/audio/extraction/extract_features_utils.py:54-113).

TEST INFRASTRUCTURE.  Runs HERE (needs /root/reference, which does not travel to the GPU box): imports the
reference's own file on top of the librosa stand-in, asserts that ``oracle/feature_oracle.py`` reproduces it
bit for bit for every knob setting, and writes ``tests/golden/autocorr_knobs.npz``.

    python oracle/make_golden_knobs.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = "/root/reference"
sys.path.insert(0, os.path.join(HERE, "librosa_standin"))
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)

from utils.audio.extraction import extract_features_utils as ref_u   # noqa: E402  (the reference file)
from neurosync_trainer_lite_b200 import synth                        # noqa: E402
from oracle import feature_oracle as fo                              # noqa: E402

SETTINGS = {
    "nopad": dict(pad_signal=False),
    "constant": dict(padding_mode="constant"),
    "edge": dict(padding_mode="edge"),
    "symmetric": dict(padding_mode="symmetric"),
    "trim": dict(trim_padded=True),
    "edge_trim": dict(padding_mode="edge", trim_padded=True),
}


def main():
    out = {}
    for tag, sr, seconds, seed, kind in (("a", 88200, 0.4, 31, "voiced"), ("b", 16000, 0.5, 32, "gated")):
        y = synth.synth_clip(seconds, sr, seed=seed, kind=kind)
        F, H = fo.frame_params(sr)
        out[f"{tag}_y"], out[f"{tag}_sr"] = y, sr
        for name, kw in SETTINGS.items():
            ref = ref_u.extract_overlapping_autocorr(y, sr, F, H, **kw)
            mine = fo.autocorr_block(y, sr, F, H, **kw)
            assert ref.dtype == mine.dtype and np.array_equal(ref, mine), (tag, name)
            if name.endswith("trim"):
                # identical to the unpadded result on these clips: stored once, which keeps the file under 1 MB
                assert np.array_equal(ref, out[f"{tag}_nopad"]), (tag, name)
                continue
            out[f"{tag}_{name}"] = ref
    # a clip whose leading frames are silent: constant padding makes frame 0 all-zero, the edge fix copies frame 1
    y = synth.synth_clip(0.3, 88200, seed=33, kind="voiced")
    y[:740] = 0.0
    F, H = fo.frame_params(88200)
    ref = ref_u.extract_overlapping_autocorr(y, 88200, F, H, padding_mode="constant")
    assert np.array_equal(ref, fo.autocorr_block(y, 88200, F, H, padding_mode="constant"))
    assert np.array_equal(ref[:, 0], ref[:, 1]) and np.abs(ref[:, 1]).max() > 0.1
    out["c_y"], out["c_constant"] = y, ref
    # zero_threshold: a matrix whose first column is below 0.5 everywhere and whose last column is not
    rng = np.random.default_rng(34)
    m = rng.uniform(-1, 1, size=(187, 12))
    m[:, 0] *= 0.4
    fixed = ref_u.fix_edge_frames_autocorr(m.copy(), zero_threshold=0.5)
    assert np.array_equal(fixed, fo.fix_edge_frames(m.copy(), zero_threshold=0.5))
    assert np.array_equal(fixed[:, 0], m[:, 1]) and np.array_equal(fixed[:, -1], m[:, -1])
    out["thr_in"], out["thr_out"] = m, fixed
    path = os.path.join(ROOT, "tests", "golden", "autocorr_knobs.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()

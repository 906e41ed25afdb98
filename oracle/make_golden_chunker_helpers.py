"""Digests of the reference chunker's ``blend_chunks`` / ``pad_audio_chunk`` results on the inputs of
tests/test_audio_processing.py::test_matches_reference_module, written to tests/golden/audio_processing_helpers.json.

The reference module is not part of this repository.  The package's host chunker was compared with it bit for bit on
exactly these calls when the chunker was added (commit edd8eed), and its host route has not changed since, so its
results stand for the reference's.  SHA-256 digests of the result bytes instead of the arrays: the arrays would take
1.3 MB.  Run from the repo root:  python oracle/make_golden_chunker_helpers.py"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from test_audio_processing import CASES, _features  # noqa: E402

from neurosync_trainer_lite_b200.utils.audio.processing import audio_processing as ap  # noqa: E402


def describe(array):
    """dtype, shape and SHA-256 of the C-ordered bytes: equal descriptions mean bit-identical arrays."""
    array = np.ascontiguousarray(array)
    return {"dtype": array.dtype.str, "shape": list(array.shape), "sha256": hashlib.sha256(array.tobytes()).hexdigest()}


def helper_calls(n):
    """The two helper calls of test_matches_reference_module for the input of case n."""
    feats = _features(n, seed=n)
    a, b = feats[:40].astype(np.float32), feats[40:70].astype(np.float32)
    return {"blend_chunks": ap.blend_chunks(a, b, 16), "pad_audio_chunk": ap.pad_audio_chunk(a, 128, 256)}


if __name__ == "__main__":
    out = {str(n): {name: describe(v) for name, v in helper_calls(n).items()} for n in sorted({c[0] for c in CASES})}
    path = os.path.join(ROOT, "tests", "golden", "audio_processing_helpers.json")
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1, sort_keys=True)
        fh.write("\n")
    print(path)

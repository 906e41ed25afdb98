"""Inference-side chunker (SURVEY.md section 8(f)-4): the package's mirror of the reference's
``utils/audio/processing/audio_processing.py`` against what the reference module returned on a small
deterministic model: its ``process_audio_features`` results (tests/golden/audio_processing.npz, made by
oracle/make_golden_chunker.py) and digests of its helper results (tests/golden/audio_processing_helpers.json,
oracle/make_golden_chunker_helpers.py)."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

from neurosync_trainer_lite_b200.utils.audio.processing import audio_processing as ap

HERE = os.path.dirname(os.path.abspath(__file__))


class ToyModel(torch.nn.Module):
    """encoder/decoder pair with the reference's interface; mixes rows so chunk position matters."""

    def __init__(self, features=256, out=68):
        super().__init__()
        g = torch.Generator().manual_seed(7)
        self.w1 = torch.nn.Parameter(torch.randn(features, 32, generator=g) * 0.05)
        self.w2 = torch.nn.Parameter(torch.randn(32, out, generator=g) * 0.3)

    def encoder(self, x):
        h = torch.tanh(x @ self.w1)
        return h + 0.25 * torch.roll(h, 1, dims=1)      # depends on neighbouring rows of the chunk

    def decoder(self, h):
        return h @ self.w2


def _features(n, seed):
    return np.random.default_rng(seed).standard_normal((n, 256)).astype(np.float64)


CASES = [(300, 128, 16), (128, 128, 16), (129, 128, 16), (50, 128, 16), (257, 64, 8), (1000, 128, 32), (7, 64, 16)]


def test_helpers_match_known_answers():
    a = np.arange(10, dtype=np.float32).reshape(5, 2)
    b = 100 + np.arange(8, dtype=np.float32).reshape(4, 2)
    got = ap.blend_chunks(a, b, 3)
    assert got.shape == (6, 2)
    np.testing.assert_array_equal(got[:2], a[:2])
    np.testing.assert_array_equal(got[2], a[2])                            # alpha = 0: pure chunk1
    np.testing.assert_allclose(got[3], (1 - 1 / 3) * a[3] + (1 / 3) * b[1], rtol=1e-6)
    np.testing.assert_array_equal(got[5], b[3])
    assert ap.blend_chunks(a, b, 0).shape == (9, 2)
    padded = ap.pad_audio_chunk(a, 8, 2)
    np.testing.assert_array_equal(padded[5:], a[[3, 2, 1]])                # reflect, edge not repeated
    assert ap.ensure_2d(np.zeros((2, 3, 4))).shape == (6, 4)
    assert ap.add_specified_dimensions_back(np.ones((3, 48))).shape == (3, 68)
    z = ap.zero_columns(np.ones((2, 68)))
    assert z[:, :14].sum() == 0 and z[:, 51:61].sum() == 0 and z[:, 14:51].all()


@pytest.mark.parametrize("n,frame,overlap", CASES)
def test_matches_golden(n, frame, overlap):
    gold = np.load(os.path.join(HERE, "golden", "audio_processing.npz"))
    model = ToyModel()
    feats = _features(n, seed=n)
    want = gold[f"out_{n}_{frame}_{overlap}"]
    for batched in (False, True):
        got = ap.process_audio_features(feats, model, "cpu", {"frame_size": frame, "overlap": overlap}, batched=batched)
        assert got.shape == want.shape == (n, 68)
        # chunk-by-chunk decoding is the reference's own arithmetic; the batched forward pass may differ
        # by the matmul blocking of the batch (float32 round-off)
        np.testing.assert_allclose(got, want, rtol=0, atol=0 if not batched else 2e-6)


@pytest.mark.parametrize("n,frame,overlap", CASES)
def test_matches_reference_module(n, frame, overlap):
    """Chunk-by-chunk decoding reproduces the reference module's result, and the cross-fade / reflect-padding
    helpers its results (dtype, shape and SHA-256 of the bytes: bit for bit)."""
    gold = np.load(os.path.join(HERE, "golden", "audio_processing.npz"))
    with open(os.path.join(HERE, "golden", "audio_processing_helpers.json")) as fh:
        ref = json.load(fh)[str(n)]
    model = ToyModel()
    feats = _features(n, seed=n)
    cfg = {"frame_size": frame, "overlap": overlap}
    want = gold[f"out_{n}_{frame}_{overlap}"]
    got = ap.process_audio_features(feats, model, "cpu", cfg, batched=False)
    np.testing.assert_array_equal(got, want)
    a, b = feats[:40].astype(np.float32), feats[40:70].astype(np.float32)
    for name, out in (("blend_chunks", ap.blend_chunks(a, b, 16)), ("pad_audio_chunk", ap.pad_audio_chunk(a, 128, 256))):
        out = np.ascontiguousarray(out)
        assert (out.dtype.str, list(out.shape)) == (ref[name]["dtype"], ref[name]["shape"]), name
        assert hashlib.sha256(out.tobytes()).hexdigest() == ref[name]["sha256"], name


@pytest.mark.gpu
def test_chunker_on_device_features():
    """Feature rows straight from the CUDA path through the batched chunker on cuda:0."""
    from neurosync_trainer_lite_b200 import synth
    from neurosync_trainer_lite_b200.utils.audio.extraction.extract_features import extract_and_combine_features
    y = synth.synth_clip(3.0, 88200, seed=11, kind="voiced")
    feats = extract_and_combine_features(y, 88200, 1470, 735)
    model = ToyModel().to("cuda:0")
    cfg = {"frame_size": 128, "overlap": 16}
    got = ap.process_audio_features(feats, model, "cuda:0", cfg)
    want = ap.process_audio_features(feats, ToyModel(), "cpu", cfg, batched=False)
    assert got.shape == (len(feats), 68)
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("n,frame,overlap", CASES + [(230, 128, 16), (240, 128, 16), (1801, 128, 16), (1, 128, 16)])
def test_device_resident_chunker_equals_host_chunker(n, frame, overlap):
    """nsf_chunk_gather / nsf_chunk_blend against the host route: the gathered chunks are bit-identical to the
    NumPy chunks (reflect-completed tails included), and given the SAME decoded chunks the cross-faded result is
    bit-identical too (the reference's float32 arithmetic, separate multiply and add)."""
    import ctypes as C

    from neurosync_trainer_lite_b200 import _native as nv
    from neurosync_trainer_lite_b200 import engine
    feats = _features(n, seed=n).astype(np.float32)
    cfg = {"frame_size": frame, "overlap": overlap}
    dev = torch.device("cuda", 0)
    eng = engine.get_engine(88200, 1470, 735, device=0)
    n_chunks = int(nv.lib.nsf_chunk_count(n, frame, overlap))
    starts = list(range(0, n, frame - overlap))
    assert n_chunks == len(starts)
    want_chunks = np.stack([ap.pad_audio_chunk(feats[s0:min(s0 + frame, n)], frame, 256) for s0 in starts])
    rows = torch.from_numpy(feats).to(dev)
    chunks = torch.empty((n_chunks, frame, 256), dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream(dev)
    nv.check(nv.lib.nsf_chunk_gather(eng.handle, C.c_void_p(stream.cuda_stream), C.c_void_p(rows.data_ptr()), n, 256, 256,
                                     frame, overlap, C.c_void_p(chunks.data_ptr())))
    np.testing.assert_array_equal(chunks.cpu().numpy(), want_chunks)
    # one set of decoded chunks for both blenders
    model = ToyModel().to(dev)
    with torch.no_grad():
        decoded = model.decoder(model.encoder(chunks)).contiguous()
    dec_h = decoded.cpu().numpy()
    acc = []
    for k, s0 in enumerate(starts):
        part = dec_h[k][:min(s0 + frame, n) - s0]
        acc = [ap.blend_chunks(acc.pop(), part, overlap)] if acc else [part]
    want = np.concatenate(acc, axis=0)[:n].copy()
    want[:, :61] /= 100
    out = torch.empty((n, 68), dtype=torch.float32, device=dev)
    nv.check(nv.lib.nsf_chunk_blend(eng.handle, C.c_void_p(stream.cuda_stream), C.c_void_p(decoded.data_ptr()), n, 68, frame,
                                    overlap, 61, C.c_float(100.0), C.c_void_p(out.data_ptr())))
    np.testing.assert_array_equal(out.cpu().numpy(), want)
    # and the public entry point end to end (same model, same batch -> same numbers)
    got = ap.process_audio_features(feats, model, "cuda:0", cfg)
    np.testing.assert_array_equal(got, want)
    got_t = ap.process_audio_features_device(rows, model, dev, cfg, return_tensor=True)
    assert got_t.is_cuda and torch.equal(got_t.cpu(), torch.from_numpy(want))


@pytest.mark.gpu
def test_chunker_rejects_overlap_beyond_half_a_chunk():
    from neurosync_trainer_lite_b200 import _native as nv
    feats = _features(300, seed=1).astype(np.float32)
    with pytest.raises(nv.NsfError) as e:
        ap.process_audio_features(feats, ToyModel().to("cuda:0"), "cuda:0", {"frame_size": 64, "overlap": 40})
    assert e.value.status == nv.ERR_UNSUPPORTED

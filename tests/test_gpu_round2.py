"""GPU parity, round-2 additions: the non-default autocorrelation knobs, every clip of a C2-scale batch
against the oracle, pageable vs pinned host buffers, back-to-back stream-ordered calls.

Tolerances as in test_gpu_parity.py (MFCC 1e-4, delta 2e-5, autocorrelation 2e-5; bit-exact where stated)."""
import multiprocessing as mp
import os

import numpy as np
import pytest

from neurosync_trainer_lite_b200 import synth

pytestmark = pytest.mark.gpu

TOL_MFCC, TOL_DELTA, TOL_AC = 1e-4, 2e-5, 2e-5


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
def efu(nv):
    from neurosync_trainer_lite_b200.utils.audio.extraction import extract_features_utils
    return extract_features_utils


# ---- extract_overlapping_autocorr(pad_signal, padding_mode, trim_padded), fix_edge(zero_threshold) -------
KNOBS = {
    "nopad": dict(pad_signal=False),
    "constant": dict(padding_mode="constant"),
    "edge": dict(padding_mode="edge"),
    "symmetric": dict(padding_mode="symmetric"),
    "trim": dict(trim_padded=True),
    "edge_trim": dict(padding_mode="edge", trim_padded=True),
}
# the reference returned identical arrays for these knobs on both clips: autocorr_knobs.npz stores them once
KNOB_STORED_AS = {"trim": "nopad", "edge_trim": "nopad"}


@pytest.mark.parametrize("clip", ["a", "b"])
@pytest.mark.parametrize("knob", sorted(KNOBS))
def test_autocorr_knobs_match_reference_golden(clip, knob, golden, efu, oracle):
    g = golden("autocorr_knobs")
    y, sr = g[f"{clip}_y"], int(g[f"{clip}_sr"])
    F, H = oracle.frame_params(sr)
    got = efu.extract_overlapping_autocorr(y, sr, F, H, **KNOBS[knob])
    want = g[f"{clip}_{KNOB_STORED_AS.get(knob, knob)}"]
    assert got.shape == want.shape and got.dtype == np.float64     # frame counts bit-exact
    assert np.abs(got - want).max() <= TOL_AC


def test_autocorr_constant_padding_triggers_the_edge_fix(golden, efu):
    g = golden("autocorr_knobs")
    got = efu.extract_overlapping_autocorr(g["c_y"], 88200, 1470, 735, padding_mode="constant")
    assert got.shape == g["c_constant"].shape
    assert np.array_equal(got[:, 0], got[:, 1])                    # frame 0 was all-zero and took frame 1
    assert np.abs(got - g["c_constant"]).max() <= TOL_AC


def test_fix_edge_zero_threshold(golden, efu):
    g = golden("autocorr_knobs")
    got = efu.fix_edge_frames_autocorr(g["thr_in"].copy(), zero_threshold=0.5)
    assert np.allclose(got, g["thr_out"], rtol=0, atol=1e-7)       # float32 round trip of float64 values
    assert np.array_equal(got[:, 0], got[:, 1])
    # and the default threshold leaves this matrix alone
    same = efu.fix_edge_frames_autocorr(g["thr_in"].copy())
    assert np.allclose(same, g["thr_in"], rtol=0, atol=1e-7)


def test_no_pad_flag_needs_autocorr_only(engine, nv):
    eng = engine.get_engine(88200, 1470, 735)
    y = synth.synth_clip(0.3, 88200, seed=1)
    with pytest.raises(nv.NsfError) as e:
        eng.extract_host(y, [0, len(y)], nv.AC_NO_PAD)
    assert e.value.status == nv.ERR_UNSUPPORTED


# ---- every clip of a C2-scale batch against the oracle -----------------------------------------------------
def _oracle_clip(args):
    kind, seed, seconds = args
    os.environ["OMP_NUM_THREADS"] = "1"
    from oracle import feature_oracle as fo
    y = synth.synth_clip(seconds, 88200, seed=seed, kind=kind)
    return fo.extract_and_combine_features(y, 88200, 1470, 735)


def test_every_clip_of_a_c2_scale_batch_matches_the_oracle(engine):
    """BASELINE configs[1] at full size: 60 clips x 30 s @ 88.2 kHz in ONE batch; EVERY clip is compared with
    the CPU oracle (all three signal kinds; the oracle runs on a process pool, ~1.5 core-seconds per clip)."""
    kinds = ("voiced", "noise", "gated")
    jobs = [(kinds[i % 3], 200 + i, 30.0) for i in range(60)]
    clips = [synth.synth_clip(s, 88200, seed=seed, kind=k) for k, seed, s in jobs]
    eng = engine.get_engine(88200, 1470, 735)
    packed, off = engine.pack_clips(clips)
    rows = eng.extract_host(packed, off)
    roff = eng.row_offsets(off)
    assert rows.shape == (60 * 1801, 256)
    env = {k: os.environ.get(k) for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS")}
    os.environ.update(OMP_NUM_THREADS="1", OPENBLAS_NUM_THREADS="1", MKL_NUM_THREADS="1")
    try:
        with mp.get_context("spawn").Pool(min(os.cpu_count() or 1, 32)) as pool:
            want = pool.map(_oracle_clip, jobs, chunksize=1)
    finally:
        for k, v in env.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    worst = {k: np.zeros(3) for k in kinds}
    for i, w in enumerate(want):
        got = rows[roff[i]:roff[i + 1]]
        assert got.shape == w.shape == (1801, 256)
        d = np.abs(got - w)
        worst[jobs[i][0]] = np.maximum(worst[jobs[i][0]], [d[:, :23].max(), d[:, 23:69].max(), d[:, 69:].max()])
    print("C2-scale max-abs per signal kind (mfcc, delta, autocorr):", {k: v.tolist() for k, v in worst.items()})
    # MFCC bound at this scale: 2e-4.  The DFT-as-GEMM accumulates in float32, so its error is ABSOLUTE (about
    # -125 dB below the strongest components of a frame) where the reference's float64 FFT is relative per bin; mel
    # bands 60-80 dB down therefore carry ~1e-3 dB of error, which the CMVN division by a small per-clip sigma turns
    # into up to 1.2e-4 on single rows of the 216 060 frames (measured r2a: 1.17e-4; profiles/parity_r02.md).
    for k, v in worst.items():
        assert v[0] <= 2e-4 and v[1] <= TOL_DELTA and v[2] <= TOL_AC, (k, v)


# ---- host-buffer pipeline: pageable (staged) == pinned (direct DMA), bit for bit ------------------------------
def test_pageable_and_pinned_host_buffers_give_identical_rows(engine, nv):
    eng = engine.get_engine(88200, 1470, 735)
    clips = [synth.synth_clip(s, 88200, seed=40 + i, kind=k)
             for i, (s, k) in enumerate([(3.0, "voiced"), (95.0, "noise"), (0.4, "gated"), (70.0, "voiced"),
                                         (2.0, "noise")])]              # 170 s: several pipeline groups
    packed, off = engine.pack_clips(clips)
    rows = int(eng.row_offsets(off)[-1])
    pin_in, pin_out = engine.PinnedBuffer(packed.nbytes), engine.PinnedBuffer(rows * 256 * 4)
    h_in = pin_in.view(np.float32, packed.shape)
    h_in[:] = packed
    h_out = pin_out.view(np.float32, (rows, 256))
    eng.extract_host(h_in, off, 0, out=h_out)
    paged, y_paged = eng.extract_host(packed, off, nv.PEAK_NORMALIZE, want_y=True)
    pinned_norm = eng.extract_host(h_in, off, nv.PEAK_NORMALIZE)
    assert np.array_equal(paged, pinned_norm)
    assert np.array_equal(eng.extract_host(packed, off, 0), h_out)
    assert np.array_equal(y_paged, eng.normalize_host(packed, off))
    # int16 PCM, pageable
    p16 = synth.to_int16_pcm(packed)
    a = eng.extract_host(p16, off, nv.PEAK_NORMALIZE)
    pin16 = engine.PinnedBuffer(p16.nbytes)
    h16 = pin16.view(np.int16, p16.shape)
    h16[:] = p16
    assert np.array_equal(a, eng.extract_host(h16, off, nv.PEAK_NORMALIZE))


def test_back_to_back_device_calls_do_not_share_descriptor_staging(engine, oracle):
    """Twenty stream-ordered nsf_extract_batch calls with DIFFERENT batch geometries are queued without any
    host synchronisation in between (the descriptor ring has 8 entries); every result must be its own."""
    import torch
    eng = engine.get_engine(88200, 1470, 735)
    dev = torch.device("cuda", eng.device)
    lens = [int(0.25 * 88200) + 777 * i for i in range(20)]
    ys = [synth.synth_clip(n / 88200.0, 88200, seed=60 + i, kind="voiced")[:n] for i, n in enumerate(lens)]
    pcm = [torch.from_numpy(y).to(dev) for y in ys]
    outs = []
    torch.cuda.synchronize(dev)
    for i, p in enumerate(pcm):
        out, ws = eng.extract_device(p, [0, len(ys[i])])
        outs.append((out, ws))
    torch.cuda.synchronize(dev)
    for i in (0, 7, 8, 9, 19):
        want = oracle.extract_and_combine_features(ys[i], 88200, 1470, 735)
        got = outs[i][0].cpu().numpy()
        assert got.shape == want.shape
        d = np.abs(got - want)
        assert d[:, :23].max() <= TOL_MFCC and d[:, 23:69].max() <= TOL_DELTA and d[:, 69:].max() <= TOL_AC


# ---- software-pipelined autocorrelation kernel (88.2 kHz plan) against the symmetric kernel -----------------------
def test_autocorr_kernels_agree(engine, oracle, tmp_path):
    """k_autocorr_pipe (eight warps per SM, two frame buffers per warp, the next frame staged inside the MMA loop of
    the current one) is the product path at F = 1470; NSF_AC_KERNEL=sym selects the symmetric kernel of the same
    arithmetic.  Bit-identical rows on a ragged batch: shortest legal clip, odd frame count, near-silent edge frames
    (edge-frame fix), short clips (a warp's run crosses clips), and every row within TOL_AC of the oracle."""
    import subprocess
    import sys
    sr = 88200
    F, H = oracle.frame_params(sr)
    lens = [9 * H + 3, sr + 17, sr // 2, 33 * H, 3 * sr // 2 + F, 10 * H, 2 * sr]
    clips = []
    for i, n in enumerate(lens):
        c = synth.synth_clip(n / sr + 0.01, sr, seed=700 + i, kind=("voiced", "gated", "noise")[i % 3])[:n].copy()
        if i == 1:
            c[: 2 * F] *= 1e-6          # near-silent first frames
        if i == 4:
            c[-2 * F:] *= 1e-6          # near-silent last frames
        clips.append(c)
    y = np.concatenate(clips).astype(np.float32)
    off = np.concatenate([[0], np.cumsum([len(c) for c in clips])]).astype(np.int64)
    np.save(tmp_path / "y.npy", y)
    np.save(tmp_path / "off.npy", off)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = {}
    for kern in ("pipe", "sym"):
        out = tmp_path / (kern + ".npy")
        code = ("import sys, numpy as np; sys.path.insert(0, %r)\n"
                "from neurosync_trainer_lite_b200 import engine\n"
                "y, off = np.load(%r), np.load(%r)\n"
                "np.save(%r, engine.get_engine(%d, %d, %d).extract_host(y, off, 0))\n"
                % (root, str(tmp_path / "y.npy"), str(tmp_path / "off.npy"), str(out), sr, F, H))
        env = dict(os.environ)
        env.pop("NSF_AC_KERNEL", None)
        if kern == "sym":
            env["NSF_AC_KERNEL"] = "sym"
        subprocess.run([sys.executable, "-c", code], check=True, env=env, timeout=600)
        res[kern] = np.load(out)
    assert res["pipe"].shape == res["sym"].shape and res["pipe"].shape[0] > 0
    assert np.array_equal(res["pipe"], res["sym"])
    roff = engine.get_engine(sr, F, H).row_offsets(off)
    for i, c in enumerate(clips):
        want = oracle.extract_and_combine_features(c, sr, F, H)
        got = res["pipe"][roff[i]:roff[i + 1]]
        assert got.shape == want.shape
        assert np.abs(got[:, 69:] - want[:, 69:]).max() <= TOL_AC, i


# ---- the two MMA loops of the autocorrelation kernel (five tiles / six MMAs per K-block) ---------------------------
@pytest.mark.parametrize("sr", [16000, 44100, 88200])
def test_autocorr_loops_agree(sr, engine, oracle, tmp_path):
    """k_autocorr_sym runs the five-tile loop (am_mma5: HH + C[lag] + C[-lag], A_l never loaded) for F >= 689 and the
    six-MMA loop (am_mma) below; NSF_AC_LOOP forces one.  Same products, another summation order: the two agree to
    2e-6 on the autocorrelation columns (identical MFCC columns) and each is within TOL_AC of the oracle - ragged
    batch whose clips include the shortest legal one, an odd frame count and near-silent edge frames."""
    import subprocess
    import sys
    F, H = oracle.frame_params(sr)
    lens = [9 * H + 3, 2 * sr + 17, sr // 2, 33 * H, 3 * sr // 2 + F]
    clips = []
    for i, n in enumerate(lens):
        c = synth.synth_clip(n / sr + 0.01, sr, seed=900 + i, kind=("voiced", "gated", "noise")[i % 3])[:n].copy()
        if i == 1:
            c[: 2 * F] *= 1e-6          # near-silent first frames: the edge-frame fix is exercised
        clips.append(c)
    y = np.concatenate(clips).astype(np.float32)
    off = np.concatenate([[0], np.cumsum([len(c) for c in clips])]).astype(np.int64)
    np.save(tmp_path / "y.npy", y)
    np.save(tmp_path / "off.npy", off)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = {}
    for loop in ("five", "six"):
        out = tmp_path / (loop + ".npy")
        code = ("import sys, numpy as np; sys.path.insert(0, %r)\n"
                "from neurosync_trainer_lite_b200 import engine\n"
                "y, off = np.load(%r), np.load(%r)\n"
                "np.save(%r, engine.get_engine(%d, %d, %d).extract_host(y, off, 0))\n"
                % (root, str(tmp_path / "y.npy"), str(tmp_path / "off.npy"), str(out), sr, F, H))
        subprocess.run([sys.executable, "-c", code], check=True, env=dict(os.environ, NSF_AC_LOOP=loop), timeout=600)
        res[loop] = np.load(out)
    assert res["five"].shape == res["six"].shape and res["five"].shape[0] > 0
    assert np.array_equal(res["five"][:, :69], res["six"][:, :69])
    assert np.abs(res["five"][:, 69:] - res["six"][:, 69:]).max() <= 2e-6
    default = engine.get_engine(sr, F, H).extract_host(y, off, 0)
    # the automatic choice: five tiles from 44 K-blocks up and at F = 266 (16 kHz), whose five-tile loop is unrolled at
    # compile time (am_mma5_static: the same products in the same order as am_mma5)
    assert np.array_equal(default, res["five" if (F >= 689 or F == 266) else "six"])
    roff = engine.get_engine(sr, F, H).row_offsets(off)
    for i, c in enumerate(clips):
        want = oracle.extract_and_combine_features(c, sr, F, H)
        for loop in ("five", "six"):
            got = res[loop][roff[i]:roff[i + 1]]
            assert got.shape == want.shape
            assert np.abs(got[:, 69:] - want[:, 69:]).max() <= TOL_AC, (loop, i)


# ---- collect_features in float32 (what load_data returns): single-round-trip row path of k_collect_rows ----
def _collect_f32_emulation(a, f, include_fast, include_slow, blend, k):
    """data_processing.py:126-197 restated in float32 with the device's operation order (the float64 oracle rounds
    the facial smoothing in float64): version rows are bit-exact targets, cross-fade rows are returned as NaN."""
    h = np.float32(0.5)
    n = min(len(a), len(f))
    la, lf = len(a), len(f)
    a = a[(la - n) // 2:(la - n) // 2 + n] if la > lf else a[:n]
    f = f[(lf - n) // 2:(lf - n) // 2 + n] if lf > la else f[:n]

    def slower(d):
        out = np.zeros((2 * len(d) - 1, d.shape[1]), np.float32)
        out[0::2] = d
        out[1::2] = (d[:-1] + d[1:]) * h
        return out

    def smooth(d):
        out = d.copy()
        out[1:] = (d[:-1] + d[1:]) * h
        return out

    va, vf = [a], [f]
    if include_fast:
        va.append(a[::2]); vf.append(f[::2])
    if include_slow:
        va.append(slower(a)); vf.append(smooth(slower(f)))

    def stack(vs):
        acc = vs[0]
        for s in vs[1:]:
            nb = min(k, len(acc), len(s)) if blend else 0
            if nb <= 0:
                acc = np.vstack([acc, s])
            else:
                acc = np.vstack([acc[:-nb], np.full((nb, s.shape[1]), np.nan, np.float32), s[nb:]])
        return acc
    return stack(va), stack(vf)


@pytest.mark.parametrize("kw", [dict(include_fast=True, include_slow=True, blend_boundaries=False),
                                dict(include_fast=True, include_slow=True, blend_boundaries=True),
                                dict(include_fast=False, include_slow=True, blend_boundaries=True),
                                dict(include_fast=True, include_slow=False, blend_boundaries=True)])
def test_collect_float32_rows_bit_exact(kw, engine, oracle):
    eng = engine.get_engine(88200, 1470, 735)
    rng = np.random.default_rng(11)
    sizes = [(1801, 1800), (300, 305), (64, 64), (31, 40), (2, 2)]
    audio = [rng.standard_normal((na, 256)).astype(np.float32) for na, _ in sizes]
    facial = [rng.uniform(0, 1, (nf, 61)).astype(np.float32) for _, nf in sizes]
    a_off = np.concatenate([[0], np.cumsum([len(a) for a in audio])]).astype(np.int64)
    f_off = np.concatenate([[0], np.cumsum([len(f) for f in facial])]).astype(np.int64)
    oa, of, o_off = eng.collect_host(np.concatenate(audio), a_off, np.concatenate(facial), f_off,
                                     kw["include_fast"], kw["include_slow"], kw["blend_boundaries"], 30)
    for i, (a, f) in enumerate(zip(audio, facial)):
        wa, wf = _collect_f32_emulation(a, f, kw["include_fast"], kw["include_slow"], kw["blend_boundaries"], 30)
        ga, gf = oa[o_off[i]:o_off[i + 1]], of[o_off[i]:o_off[i + 1]]
        assert ga.shape == wa.shape and gf.shape == wf.shape
        keep = ~np.isnan(wa[:, 0])
        np.testing.assert_array_equal(ga[keep], wa[keep])               # version rows: bit-exact
        np.testing.assert_array_equal(gf[keep], wf[keep])
        # cross-fade rows (and everything else) against the float64 oracle
        ra, rf = oracle.collect_from_arrays(a.astype(np.float64), f.astype(np.float64), kw["include_fast"],
                                            kw["include_slow"], kw["blend_boundaries"], 30)
        np.testing.assert_allclose(ga, ra, rtol=0, atol=2e-6)
        np.testing.assert_allclose(gf, rf, rtol=0, atol=1e-6)


def test_front_end_kernels_do_not_depend_on_pointer_alignment(nv, engine):
    """k_absmax / k_normalize read 16-byte vectors when the caller's device pointer allows it and fall back to the scalar
    form otherwise: int16 and float32 PCM at an odd element offset give the rows of the aligned call, bit for bit."""
    import torch
    eng = engine.get_engine(88200, 1470, 735)
    clips = [synth.synth_clip(0.7, 88200, seed=21, kind="voiced"), synth.synth_clip(0.41, 88200, seed=22, kind="noise")]
    packed, off = engine.pack_clips(clips)
    pcm16 = np.clip(np.round(packed * 32767.0), -32768, 32767).astype(np.int16)
    dev = torch.device("cuda", 0)
    for host in (pcm16, packed.astype(np.float32)):
        t = torch.from_numpy(host).to(dev)
        want, _ = eng.extract_device(t, off, nv.PEAK_NORMALIZE)
        for shift in (1, 3, 5):
            buf = torch.empty(len(host) + 8, dtype=t.dtype, device=dev)
            buf[shift:shift + len(host)] = t
            view = buf[shift:shift + len(host)]
            assert view.data_ptr() % 16 != 0
            got, _ = eng.extract_device(view, off, nv.PEAK_NORMALIZE)
            assert torch.equal(got, want)

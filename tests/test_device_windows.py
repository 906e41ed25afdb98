"""Training windows served from GPU memory (include/nsf.h nsf_window_offsets / nsf_window_gather, dataset/dataset.py
DeviceWindows / DeviceWindowLoader).

The host statement is AudioFacialDataset: ``collate_fn([ds[i] for i in batch])`` over ``_WindowedClip``'s windows.
The device route is a pure copy, so every comparison is bit for bit, and the device loaders must draw from the global
generator exactly as ``DataLoader`` does, so one seed gives the same batches in the same order."""
import numpy as np
import pytest
import torch

WINDOWS = (1, 2, 64, 100, 127, 128)


@pytest.fixture(scope="module")
def nv():
    from neurosync_trainer_lite_b200 import _native
    return _native


def host_count(na, nf, window):
    """len(_WindowedClip) when the host route can serve every window of the clip, else None."""
    from neurosync_trainer_lite_b200.dataset.dataset import _WindowedClip
    try:
        clip = _WindowedClip(np.zeros((na, 2)), np.zeros((nf, 3)), window)
        clip.get(len(clip) - 1)          # the reflected tail window is where short streams fail
    except (ValueError, RuntimeError):
        return None
    return len(clip)


def sizes(window):
    return sorted({window, window + 1, 2 * window - 1, 2 * window, 256, 300})


# ---- CPU ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("window", WINDOWS)
def test_window_offsets_are_the_prefix_sum_of_the_host_counts(window, nv):
    pairs = [(na, nf) for na in sizes(window) for nf in sizes(window)]
    counts = [host_count(na, nf, window) for na, nf in pairs]
    good = [(p, c) for p, c in zip(pairs, counts) if c is not None]
    assert any(na == nf for (na, nf), _ in good) and any(na != nf for (na, nf), _ in good)
    a_off = np.concatenate([[0], np.cumsum([na for (na, _), _ in good])])
    f_off = np.concatenate([[0], np.cumsum([nf for (_, nf), _ in good])])
    got = nv.window_offsets(a_off, f_off, window)
    want = np.concatenate([[0], np.cumsum([c for _, c in good])])
    np.testing.assert_array_equal(got, want)
    if window == 128:                    # the reference's counts
        assert nv.window_offsets([0, 300], [0, 300], 128)[-1] == 174
        assert nv.window_offsets([0, 256], [0, 256], 128)[-1] == 129


@pytest.mark.parametrize("window", WINDOWS)
def test_window_offsets_reject_exactly_what_the_host_route_rejects(window, nv):
    grid = sorted(set(sizes(window)) | {0, 1, max(window - 1, 0), window // 2, window // 2 + 1, window + 2})
    rejected = 0
    for na in grid:
        for nf in grid:
            want = host_count(na, nf, window)
            if want is None:
                rejected += 1
                with pytest.raises(nv.NsfError) as e:
                    nv.window_offsets([0, na], [0, nf], window)
                assert e.value.status == nv.ERR_BAD_ARG
            else:
                assert nv.window_offsets([0, na], [0, nf], window)[-1] == want, (na, nf)
    assert rejected > 0


def test_window_offsets_reject_bad_offsets_and_windows(nv):
    for a_off, f_off, window in [([0, 300, 200], [0, 300, 600], 128),     # decreasing audio offsets
                                 ([0, 300, 600], [0, 400, 300], 128),     # decreasing facial offsets
                                 ([-1, 300], [0, 301], 128),              # negative offset
                                 ([0, 300], [-5, 295], 128),
                                 ([0, 300], [0, 300], 0),                 # window < 1
                                 ([0, 300], [0, 300], -128)]:
        with pytest.raises(nv.NsfError) as e:
            nv.window_offsets(a_off, f_off, window)
        assert e.value.status == nv.ERR_BAD_ARG
    with pytest.raises(ValueError):
        nv.window_offsets([0, 300], [0, 300, 600], 128)                   # one facial clip too many
    # offsets need not start at 0: a clip's rows are wherever its offsets say
    np.testing.assert_array_equal(nv.window_offsets([10, 310, 566], [7, 307, 563], 128), [0, 174, 303])


# ---- GPU ---------------------------------------------------------------------------------------------
def ragged_dataset(window, audio_cols, seed=0):
    """An AudioFacialDataset (rows given directly, no files) whose clips cover every window shape: audio longer than
    facial and the reverse (tails that mirror the shorter stream, a one-row tail segment), equal lengths with and
    without a tail, exact multiples of the window, regular windows that run past a shorter stream (zero rows)."""
    from neurosync_trainer_lite_b200.dataset.dataset import AudioFacialDataset
    w = window
    pairs = [(2 * w + w // 3 + 5, 2 * w + w // 3 + 5 - w // 4),     # audio longer, tail
             (2 * w + w // 2 + 3 - w // 3, 2 * w + w // 2 + 3),     # facial longer, tail
             (3 * w + 7, 3 * w + 7),                                # equal, tail
             (2 * w, 2 * w),                                        # equal, exact multiple: no tail
             (3 * w, 2 * w + 1),                                    # unequal, no tail: facial zero-padded
             (w, 2 * w),                                            # audio a window long: later windows all zero
             (2 * w + 1, w + 2),                                    # tail segment of one facial row (repeated)
             (w, w)]                                                # a single window
    ds = AudioFacialDataset.__new__(AudioFacialDataset)
    ds.micro_batch_size = w
    ds.zero_copy_windows = False
    ds.clips, ds._starts = [], [0]
    rng = np.random.default_rng(seed)
    for na, nf in pairs:
        ds.add_clip(rng.standard_normal((na, audio_cols)).astype(np.float32),
                    rng.standard_normal((nf, 61)).astype(np.float32))
    return ds


def host_batch(ds, idx):
    from neurosync_trainer_lite_b200.dataset.dataset import AudioFacialDataset
    return AudioFacialDataset.collate_fn([ds[int(i)] for i in idx])


def assert_same_batches(got, want, chunk=512):
    """got: device (src, trg); want: callable(lo, hi) -> host (src, trg) of rows [lo, hi)."""
    n = got[0].shape[0]
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        wa, wf = want(lo, hi)
        assert torch.equal(got[0][lo:hi].cpu(), wa)
        assert torch.equal(got[1][lo:hi].cpu(), wf)


@pytest.fixture(scope="module")
def windows_factory():
    from neurosync_trainer_lite_b200.dataset.dataset import DeviceWindows
    cache = {}

    def make(window, audio_cols):
        key = (window, audio_cols)
        if key not in cache:
            ds = ragged_dataset(window, audio_cols)
            cache[key] = (ds, DeviceWindows(ds, device=0))
        return cache[key]
    return make


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [1, 7, 4096])
@pytest.mark.parametrize("audio_cols", [256, 69])
@pytest.mark.parametrize("window", [128, 64, 100])
def test_window_gather_equals_collate_of_getitem(window, audio_cols, batch, windows_factory):
    ds, dw = windows_factory(window, audio_cols)
    rng = np.random.default_rng(window * 1000 + audio_cols + batch)
    idx = rng.integers(0, len(ds), size=batch)
    if batch >= 7:                          # duplicates, the first window and the last (a tail)
        idx[3], idx[5], idx[6] = idx[1], 0, len(ds) - 1
    rng.shuffle(idx)
    before = dw.engine.launch_count()
    got = dw.gather(idx)
    assert dw.engine.launch_count() == before + 1
    assert got[0].shape == (batch, window, audio_cols) and got[1].shape == (batch, window, 61)
    assert got[0].is_cuda and got[0].dtype == torch.float32 and got[0].is_contiguous()
    torch.cuda.synchronize()
    assert_same_batches(got, lambda lo, hi: host_batch(ds, idx[lo:hi]))


@pytest.mark.gpu
def test_every_window_of_the_dataset(windows_factory):
    ds, dw = windows_factory(128, 256)
    idx = np.arange(len(ds))
    got = dw.gather(torch.from_numpy(idx))        # a CPU tensor of indices is a host sequence too
    assert_same_batches(got, lambda lo, hi: host_batch(ds, idx[lo:hi]))


@pytest.mark.gpu
def test_bad_index_raises_and_leaves_outputs_untouched(windows_factory, nv):
    ds, dw = windows_factory(128, 256)
    for bad in ([0, 5, len(ds)], [-1, 3], [2, len(ds) + 1000]):
        oa = torch.full((len(bad), 128, 256), 7.0, device="cuda:0")
        of = torch.full((len(bad), 128, 61), 7.0, device="cuda:0")
        before = dw.engine.launch_count()
        with pytest.raises(nv.NsfError) as e:
            dw.gather(bad, out_audio=oa, out_facial=of)
        assert e.value.status == nv.ERR_BAD_ARG
        assert dw.engine.launch_count() == before
        torch.cuda.synchronize()
        assert bool((oa == 7.0).all()) and bool((of == 7.0).all())
    with pytest.raises(ValueError):
        dw.gather(torch.tensor([0, 1], device="cuda:0"))     # indices are validated on the host
    before = dw.engine.launch_count()
    ea, ef = dw.gather([])                                   # empty batch: no launch
    assert ea.shape == (0, 128, 256) and ef.shape == (0, 128, 61) and dw.engine.launch_count() == before


@pytest.mark.gpu
def test_gather_on_a_side_stream_and_into_given_outputs(windows_factory):
    ds, dw = windows_factory(100, 256)
    idx = np.random.default_rng(5).integers(0, len(ds), size=300)
    ref = dw.gather(idx)
    torch.cuda.synchronize()
    side = torch.cuda.Stream(device=0)
    with torch.cuda.stream(side):
        oa = torch.empty((300, 100, 256), device="cuda:0")
        of = torch.empty((300, 100, 61), device="cuda:0")
    got = dw.gather(idx, out_audio=oa, out_facial=of, stream=side)
    assert got[0] is oa and got[1] is of
    side.synchronize()
    assert torch.equal(oa, ref[0]) and torch.equal(of, ref[1])


def _loaders(data, batch, shuffle, drop_last, windows):
    from torch.utils.data import DataLoader

    from neurosync_trainer_lite_b200.dataset.dataset import AudioFacialDataset, DeviceWindowLoader
    host = DataLoader(data, batch_size=batch, shuffle=shuffle, drop_last=drop_last,
                      collate_fn=AudioFacialDataset.collate_fn)
    dev = DeviceWindowLoader(data, batch, shuffle, drop_last=drop_last, windows=windows)
    return host, dev


def _epoch(loader, seed):
    torch.manual_seed(seed)
    batches = list(loader)
    return batches, torch.rand(4)          # the global generator after the epoch


@pytest.mark.gpu
@pytest.mark.parametrize("drop_last", [False, True])
@pytest.mark.parametrize("shuffle", [True, False])
@pytest.mark.parametrize("subset", [False, True])
def test_device_loader_matches_dataloader(subset, shuffle, drop_last, windows_factory):
    from torch.utils.data import Subset, random_split
    ds, dw = windows_factory(128, 256)
    data = ds
    if subset:
        data, _ = random_split(ds, [len(ds) - 200, 200], generator=torch.Generator().manual_seed(3))
        data = Subset(data, list(range(0, len(data), 2)))       # a subset of a subset
        assert isinstance(data, Subset)
    host, dev = _loaders(data, 37, shuffle, drop_last, dw)
    assert len(dev) == len(host)
    hb, h_rng = _epoch(host, 11)
    db, d_rng = _epoch(dev, 11)
    assert len(db) == len(hb) == len(host)
    assert torch.equal(h_rng, d_rng)
    for (ha, hf), (da, df) in zip(hb, db):
        assert da.is_cuda and df.is_cuda
        assert torch.equal(da.cpu(), ha) and torch.equal(df.cpu(), hf)
    if shuffle:                              # a second epoch reshuffles the same way
        hb2, _ = _epoch(host, 12)
        db2, _ = _epoch(dev, 12)
        assert not torch.equal(hb2[0][0], hb[0][0])
        assert all(torch.equal(d[0].cpu(), h[0]) for h, d in zip(hb2, db2))


def write_take_tree(root, takes=((3.2, 190), (4.0, 240), (2.7, 161), (3.6, 215))):
    import pandas as pd

    from neurosync_trainer_lite_b200 import synth
    cols = ["Timecode", "BlendshapeCount"] + [f"bs{i}" for i in range(61)]
    for k, (secs, rows) in enumerate(takes):
        take = root / f"take_{k:03d}"
        take.mkdir(parents=True)
        y = synth.synth_clip(secs, 88200, seed=70 + k, kind=("voiced", "gated", "noise")[k % 3])
        (take / "audio.wav").write_bytes(synth.wav_bytes(synth.to_int16_pcm(0.8 * y), 88200))
        pd.DataFrame(np.hstack([np.zeros((rows, 2)), synth.synth_facial(rows, seed=k)]),
                     columns=cols).to_csv(take / f"t{k}_iPhone_cal.csv", index=False)


@pytest.mark.gpu
def test_prepare_dataloader_with_split_serves_the_host_batches(tmp_path):
    from neurosync_trainer_lite_b200.dataset import dataset as dmod
    write_take_tree(tmp_path / "data")
    config = {"root_dir": str(tmp_path / "data"), "sr": 88200, "frame_rate": 60, "micro_batch_size": 128,
              "batch_size": 16}
    dmod.prepare_dataloader(config)          # writes the feature caches: both runs below read the same rows
    torch.manual_seed(0)
    h_train, h_val, h_tl, h_vl = dmod.prepare_dataloader_with_split(config)
    hb = [list(h_tl), list(h_vl)]
    torch.manual_seed(0)
    d_train, d_val, d_tl, d_vl = dmod.prepare_dataloader_with_split(dict(config, device_windows=True))
    assert isinstance(d_tl, dmod.DeviceWindowLoader) and isinstance(d_vl, dmod.DeviceWindowLoader)
    assert d_tl.windows is d_vl.windows                       # one upload for both loaders
    assert list(d_train.indices) == list(h_train.indices) and list(d_val.indices) == list(h_val.indices)
    assert len(d_val) > 0 and len(d_tl) == len(h_tl) and len(d_vl) == len(h_vl)
    seen = []
    gather = d_tl.windows.gather
    d_tl.windows.gather = lambda idx, *a, **k: (seen.append(np.array(idx)), gather(idx, *a, **k))[1]
    db = [list(d_tl), None]
    train_seen = np.concatenate(seen)
    seen.clear()
    db[1] = list(d_vl)
    val_seen = np.concatenate(seen)
    # every window of each subset exactly once per epoch
    np.testing.assert_array_equal(np.sort(train_seen), np.sort(np.asarray(d_train.indices)))
    np.testing.assert_array_equal(np.sort(val_seen), np.sort(np.asarray(d_val.indices)))
    for h_batches, d_batches in zip(hb, db):
        assert len(h_batches) == len(d_batches)
        for (ha, hf), (da, df) in zip(h_batches, d_batches):
            assert torch.equal(da.cpu(), ha) and torch.equal(df.cpu(), hf)
    # prepare_dataloader: same batches under the same seed, and dataset[i] still serves the host copy
    torch.manual_seed(1)
    h_ds, h_loader = dmod.prepare_dataloader(config)
    hb = list(h_loader)
    torch.manual_seed(1)
    d_ds, d_loader = dmod.prepare_dataloader(dict(config, device_windows="cuda:0"))
    assert d_loader.windows.device == 0 and not d_ds[0][0].is_cuda
    db = list(d_loader)
    assert len(hb) == len(db) == len(d_loader)
    assert all(torch.equal(d[0].cpu(), h[0]) and torch.equal(d[1].cpu(), h[1]) for h, d in zip(hb, db))

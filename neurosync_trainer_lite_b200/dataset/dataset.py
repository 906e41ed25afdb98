"""Mirror of the reference's ``dataset/dataset.py`` - the consumer of the feature rows.

``AudioFacialDataset`` keeps the reference's constructor, ``__len__``, ``__getitem__`` and
``collate_fn`` contracts: item ``i`` is ``(float32[128, 256], float32[128, 61])``.  The difference
is memory: the reference materialises every stride-1 window (``process_example`` :58-98, the source
of its 128-256 GB host-RAM advice); here each clip's rows are stored once as float32 and a window is
produced at ``__getitem__`` time: an independent tensor by default (what the reference hands out, safe
for in-place augmentation), or - ``config['zero_copy_windows'] = True`` - a read-only-by-contract
``narrow`` view that shares the clip's storage with the 127 windows overlapping it.  The duplicated, reflected last window
the reference appends when ``N % 128 != 0`` (:77-96) and its failure for ``N < 128`` are preserved.
Pure host-side indexing - no arithmetic - so it needs no kernel.

``config['device_windows']`` moves the batches to the GPU instead: ``DeviceWindows`` uploads the dataset's rows to
one device once, and ``DeviceWindowLoader`` serves each batch with one ``nsf_window_gather`` launch - the same
windows in the same order as the ``DataLoader`` it replaces, already on the device.
"""
import numpy as np
import torch
from torch.nn.utils.rnn import pad_sequence
from torch.utils.data import (BatchSampler, DataLoader, Dataset, RandomSampler, SequentialSampler, Subset,
                              random_split)

from .. import engine as _engine
from .data_processing import load_data


def prepare_dataloader_with_split(config, val_split=0.1):
    """reference :12-21.  With ``config['device_windows']`` set (``True``: ``engine.default_device()``, or a device
    such as ``'cuda:1'``; ``0`` is falsy and keeps the host loaders), the two loaders are ``DeviceWindowLoader``s over
    the same split, sharing one upload of the rows; the batches and their order are those of the host loaders."""
    dataset = AudioFacialDataset(config)
    val_size = int(len(dataset) * val_split)
    train_dataset, val_dataset = random_split(dataset, [len(dataset) - val_size, val_size])
    device = config.get('device_windows')
    if device:
        windows = DeviceWindows(dataset, device)
        return (train_dataset, val_dataset,
                DeviceWindowLoader(train_dataset, config['batch_size'], shuffle=True, windows=windows),
                DeviceWindowLoader(val_dataset, config['batch_size'], shuffle=False, windows=windows))
    train_dataloader = DataLoader(train_dataset, batch_size=config['batch_size'], shuffle=True,
                                  collate_fn=AudioFacialDataset.collate_fn)
    val_dataloader = DataLoader(val_dataset, batch_size=config['batch_size'], shuffle=False,
                                collate_fn=AudioFacialDataset.collate_fn)
    return train_dataset, val_dataset, train_dataloader, val_dataloader


def prepare_dataloader(config):
    """reference :23-26.  ``config['device_windows']``: see ``prepare_dataloader_with_split``."""
    dataset = AudioFacialDataset(config)
    device = config.get('device_windows')
    if device:
        return dataset, DeviceWindowLoader(dataset, config['batch_size'], shuffle=True, device=device)
    return dataset, DataLoader(dataset, batch_size=config['batch_size'], shuffle=True,
                               collate_fn=AudioFacialDataset.collate_fn)


class _WindowedClip:
    """Rows of one clip + the window list ``process_example`` would have materialised."""

    def __init__(self, audio_features, facial_data, window):
        na, nf = len(audio_features), len(facial_data)
        top = max(na, nf)
        if top < window:
            # the reference crashes here too (broadcast error in the tail branch, dataset.py:77-91)
            raise ValueError(f"clip has {top} rows, fewer than micro_batch_size={window}")
        self.window = window
        self.n_audio, self.n_facial = na, nf
        # float32 once per clip (the reference casts every window separately, :75)
        self.audio = torch.from_numpy(np.ascontiguousarray(audio_features, dtype=np.float32))
        self.facial = torch.from_numpy(np.ascontiguousarray(facial_data, dtype=np.float32))
        self.n_regular = top - window + 1
        self.has_tail = top % window != 0
        self.top = top

    def __len__(self):
        return self.n_regular + (1 if self.has_tail else 0)

    def _window(self, rows, n_rows, start):
        avail = min(self.window, n_rows - start)
        if avail == self.window:
            return rows.narrow(0, start, self.window)            # zero-copy view
        out = torch.zeros((self.window, rows.shape[1]), dtype=torch.float32)
        if avail > 0:
            out[:avail] = rows[start:start + avail]
        return out

    def get(self, i):
        # the tail window (:77-96) starts at top - window: a full window whenever both streams have
        # `top` rows (always true after collect_features), i.e. a duplicate of the last regular one
        if i < self.n_regular:
            return (self._window(self.audio, self.n_audio, i),
                    self._window(self.facial, self.n_facial, i))
        start = self.top - self.window
        return (self._tail(self.audio, self.n_audio, start),
                self._tail(self.facial, self.n_facial, start))

    def _tail(self, rows, n_rows, start):
        seg = rows[start:min(self.top, n_rows)]
        if len(seg) == self.window:
            return rows.narrow(0, start, self.window)
        out = torch.zeros((self.window, rows.shape[1]), dtype=torch.float32)
        out[:len(seg)] = seg
        fill = torch.flip(seg, dims=(0,))[:self.window - len(seg)]   # reflection fill (:87-94)
        out[len(seg):] = fill                                        # raises like the reference if short
        return out


class AudioFacialDataset(Dataset):
    def __init__(self, config):
        self.root_dir = config['root_dir']
        self.sr = config['sr']
        self.frame_rate = config['frame_rate']
        self.micro_batch_size = config['micro_batch_size']
        # False (default): items are independent copies, as in the reference.  True: items are views into the
        # clip's rows - no copy, but modifying one in place corrupts every overlapping window
        self.zero_copy_windows = bool(config.get('zero_copy_windows', False))
        self.processed_folders = set()
        self.clips = []
        self._starts = [0]
        for audio_features, facial_data in load_data(self.root_dir, self.sr, self.processed_folders):
            self.add_clip(audio_features, facial_data)

    def add_clip(self, audio_features, facial_data):
        clip = _WindowedClip(audio_features, facial_data, self.micro_batch_size)
        self.clips.append(clip)
        self._starts.append(self._starts[-1] + len(clip))

    @property
    def examples(self):
        """The reference's materialised list, produced lazily (for code that iterates it)."""
        return [self[i] for i in range(len(self))]

    def __len__(self):
        return self._starts[-1]

    def __getitem__(self, idx):
        if idx < 0:
            idx += len(self)
        if not 0 <= idx < len(self):
            raise IndexError(idx)
        c = int(np.searchsorted(self._starts, idx, side="right")) - 1
        a, f = self.clips[c].get(idx - self._starts[c])
        if getattr(self, "zero_copy_windows", False):
            return a, f
        return a.clone(), f.clone()

    @staticmethod
    def collate_fn(batch):
        """reference :52-56."""
        src_batch, trg_batch = zip(*batch)
        return (pad_sequence(src_batch, batch_first=True, padding_value=0),
                pad_sequence(trg_batch, batch_first=True, padding_value=0))

    def process_example(self, audio_features, facial_data):
        """reference :58-98 -- kept for API parity: the explicit list of windows of ONE clip."""
        clip = _WindowedClip(audio_features, facial_data, self.micro_batch_size)
        return [tuple(t.clone() for t in clip.get(i)) for i in range(len(clip))]


def _device_index(device):
    """CUDA device index of ``True`` / ``None`` (``engine.default_device()``), an int, ``'cuda:N'`` or a
    ``torch.device``."""
    if device is None or device is True:
        return _engine.default_device()
    if isinstance(device, (str, torch.device)):
        d = torch.device(device)
        if d.type != "cuda":
            raise ValueError(f"device windows live on a CUDA device, not {device!r}")
        return _engine.default_device() if d.index is None else d.index
    return int(device)


class DeviceWindows:
    """The rows of an ``AudioFacialDataset`` on one GPU: ``audio [sum N, cols]`` and ``facial [sum N, 61]`` float32,
    clip i owning rows ``[audio_offsets[i], audio_offsets[i + 1])`` / ``[facial_offsets[i], facial_offsets[i + 1])``,
    uploaded once (one async copy per clip and stream).  ``window_offsets`` numbers the windows exactly as the
    dataset numbers its items; ``gather(indices)`` returns ``collate_fn([dataset[i] for i in indices])`` as CUDA
    tensors, bit for bit."""

    def __init__(self, dataset, device=None):
        clips = dataset.clips
        if not clips:
            raise ValueError("DeviceWindows: the dataset has no clips")
        self.dataset = dataset
        self.device = _device_index(device)
        self.window = int(dataset.micro_batch_size)
        self.audio_offsets = np.zeros(len(clips) + 1, dtype=np.int64)
        self.facial_offsets = np.zeros(len(clips) + 1, dtype=np.int64)
        np.cumsum([c.n_audio for c in clips], out=self.audio_offsets[1:])
        np.cumsum([c.n_facial for c in clips], out=self.facial_offsets[1:])
        self.window_offsets = _engine.Engine.window_offsets(self.audio_offsets, self.facial_offsets, self.window)
        if int(self.window_offsets[-1]) != len(dataset):
            raise RuntimeError(f"window count {int(self.window_offsets[-1])} != dataset length {len(dataset)}")
        a_cols, f_cols = clips[0].audio.shape[1], clips[0].facial.shape[1]
        if any(c.audio.shape[1] != a_cols or c.facial.shape[1] != f_cols for c in clips):
            raise ValueError("DeviceWindows: every clip needs the same audio and facial column counts")
        dev = torch.device("cuda", self.device)
        f, h = _engine.frame_params(88200)
        self.engine = _engine.get_engine(88200, f, h, device=self.device)
        self.audio = torch.empty((int(self.audio_offsets[-1]), a_cols), dtype=torch.float32, device=dev)
        self.facial = torch.empty((int(self.facial_offsets[-1]), f_cols), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            for c, a0, f0 in zip(clips, self.audio_offsets, self.facial_offsets):
                self.audio[a0:a0 + c.n_audio].copy_(c.audio, non_blocking=True)
                self.facial[f0:f0 + c.n_facial].copy_(c.facial, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()

    def __len__(self):
        return int(self.window_offsets[-1])

    def gather(self, indices, out_audio=None, out_facial=None, stream=None):
        """Windows ``indices`` (host sequence of dataset item numbers) -> ``(src [n, window, cols], trg [n, window,
        61])`` CUDA float32, stream-ordered on ``stream`` (default: the current stream)."""
        return self.engine.window_gather(self.audio, self.audio_offsets, self.facial, self.facial_offsets,
                                         self.window, indices, out_audio, out_facial, stream)


class DeviceWindowLoader:
    """``DataLoader(data, batch_size, shuffle, drop_last, collate_fn=AudioFacialDataset.collate_fn)`` served from GPU
    memory: every batch is one ``nsf_window_gather`` launch into fresh ``(src [B, window, 256], trg [B, window, 61])``
    CUDA tensors.  ``data`` is an ``AudioFacialDataset`` or a ``Subset`` of one (``random_split``'s output); a subset's
    positions map to dataset items through ``subset.indices``.  The batches come from the same
    ``BatchSampler(RandomSampler | SequentialSampler)`` with the same draws from the global generator (one int64
    when the iterator is created, as ``DataLoader``'s iterator draws its base seed, then the sampler's own seed at
    the first batch), so one ``torch.manual_seed`` gives the host loader's batches in the host loader's order.
    ``windows``: a ``DeviceWindows`` of the underlying dataset to share (the train and validation loaders of one
    split use one upload); without it the loader uploads the dataset to ``device``."""

    def __init__(self, data, batch_size, shuffle, drop_last=False, device=None, windows=None):
        base, positions = data, None
        while isinstance(base, Subset):
            idx = np.asarray(base.indices, dtype=np.int64)
            positions = idx if positions is None else idx[positions]
            base = base.dataset
        if not isinstance(base, AudioFacialDataset):
            raise TypeError(f"DeviceWindowLoader needs an AudioFacialDataset or a Subset of one, got {type(base)}")
        if windows is None:
            windows = DeviceWindows(base, device)
        elif windows.dataset is not base:
            raise ValueError("DeviceWindowLoader: `windows` holds the rows of another dataset")
        elif device is not None and _device_index(device) != windows.device:
            raise ValueError(f"DeviceWindowLoader: `windows` lives on cuda:{windows.device}, not {device!r}")
        self.dataset = data
        self.windows = windows
        self.batch_size, self.drop_last = batch_size, drop_last
        self._positions = positions
        sampler = RandomSampler(data) if shuffle else SequentialSampler(data)
        self.sampler = sampler
        self.batch_sampler = BatchSampler(sampler, batch_size, drop_last)

    def __len__(self):
        return len(self.batch_sampler)

    def __iter__(self):
        return _DeviceWindowIter(self)


class _DeviceWindowIter:
    def __init__(self, loader):
        self._loader = loader
        self._batches = iter(loader.batch_sampler)
        # DataLoader's iterator draws its base seed here (_BaseDataLoaderIter.__init__); drawing it too keeps the
        # global generator - and so every later shuffle - in step with the host loaders
        torch.empty((), dtype=torch.int64).random_()

    def __iter__(self):
        return self

    def __next__(self):
        idx = np.asarray(next(self._batches), dtype=np.int64)
        if self._loader._positions is not None:
            idx = self._loader._positions[idx]
        return self._loader.windows.gather(idx)

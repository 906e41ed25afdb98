"""Host-side engine: plans, per-device contexts, pinned buffers and the two ways into the C ABI.

* ``extract_host``   - NumPy in / NumPy out through ``nsf_extract_host`` (what the reference-facing
  functions use; H2D, kernels and D2H are pipelined inside the library);
* ``extract_device`` - torch CUDA tensors in / out through ``nsf_extract_batch`` (device-resident,
  stream-ordered; torch is only the allocator and stream provider).

Nothing here computes features on the CPU.
"""
import ctypes as C
import os
import threading

import numpy as np

from . import _native as nv

DEFAULT_N_MFCC, DEFAULT_N_MELS, DEFAULT_N_LAGS = 23, 128, 187  # extract_features_utils.py:11,54


def default_device():
    return int(os.environ.get("NSF_DEVICE", os.environ.get("LOCAL_RANK", "0")))


def frame_params(sr):
    """(frame_length, hop_length) exactly as extract_features.py:12-13 computes them."""
    f = nv.lib.nsf_frame_length(int(sr))
    return f, nv.lib.nsf_hop_length(f)


class _HostBlock:
    """Owner of one cudaHostAlloc allocation: frees it when the last array viewing it is gone."""

    def __init__(self, ptr):
        self.ptr = ptr

    def __del__(self):
        try:
            if self.ptr is not None and self.ptr.value:
                nv.lib.nsf_host_free(self.ptr)
                self.ptr = None
        except Exception:
            pass


class PinnedBuffer:
    """Page-locked host memory (cudaHostAlloc through the C ABI) exposed as NumPy arrays.

    The allocation is owned by the ctypes block every view is built on, so arrays handed to callers
    (e.g. the dataset examples of ``load_data``) stay valid after the ``PinnedBuffer`` object itself
    is dropped; the memory is released when the last view dies."""

    def __init__(self, nbytes):
        p = C.c_void_p()
        nv.check(nv.lib.nsf_host_alloc(C.byref(p), int(max(nbytes, 1))))
        self.nbytes = int(nbytes)
        self.address = p.value
        self._raw = (C.c_char * max(self.nbytes, 1)).from_address(p.value)
        self._raw._block = _HostBlock(p)

    def view(self, dtype, shape, offset=0):
        count = int(np.prod(shape))
        arr = np.frombuffer(self._raw, dtype=dtype, count=count, offset=int(offset))
        return arr.reshape(shape)

    def close(self):
        """Drop this object's reference; the memory goes when no view is left."""
        self._raw = None


_scratch = {}


def scratch_pinned(tag, nbytes):
    """Grow-only page-locked scratch buffer kept for the life of the process (library-owned staging for the
    dataset builders: cudaHostAlloc costs ~1 ms per MB, far more than filling the buffer).  The caller must be
    done with the previous contents of ``tag`` - views handed out earlier alias the same memory."""
    buf = _scratch.get(tag)
    if buf is None or buf.nbytes < nbytes:
        _scratch[tag] = buf = PinnedBuffer(int(nbytes * 1.25) + 4096)
    return buf


class Plan:
    """Constant tables for one (sr, F, H) geometry.  Pure host object: usable without a GPU."""

    def __init__(self, sr, frame_length, hop_length, n_mfcc=DEFAULT_N_MFCC, n_mels=DEFAULT_N_MELS,
                 n_lags=DEFAULT_N_LAGS):
        h = C.c_void_p()
        nv.check(nv.lib.nsf_plan_create(int(sr), int(frame_length), int(hop_length), int(n_mfcc),
                                        int(n_mels), int(n_lags), C.byref(h)))
        self.handle = h
        self.sr, self.F, self.H = int(sr), int(frame_length), int(hop_length)
        self.n_mfcc, self.n_mels, self.n_lags = int(n_mfcc), int(n_mels), int(n_lags)
        b, c, k, kp = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
        nv.lib.nsf_plan_info(h, C.byref(b), C.byref(c), C.byref(k), C.byref(kp))
        self.bins, self.chains, self.fold_k, self.fold_kp = b.value, c.value, k.value, kp.value

    def table(self, which):
        n = nv.lib.nsf_plan_table(self.handle, which, None, 0)
        out = np.empty(n, dtype=np.float32)
        nv.lib.nsf_plan_table(self.handle, which, out.ctypes.data_as(C.POINTER(C.c_float)), n)
        return out

    def mel_basis(self):
        return self.table(nv.TABLE_MEL).reshape(self.n_mels, self.bins)

    def dct_matrix(self):
        return self.table(nv.TABLE_DCT).reshape(self.n_mfcc, self.n_mels)

    def fold_check(self, frame):
        """DFT of one frame through the fold tables, float64 on the host (table verification)."""
        frame = np.ascontiguousarray(frame, dtype=np.float32)
        assert frame.shape == (self.F,)
        re = np.empty(self.bins, dtype=np.float64)
        im = np.empty(self.bins, dtype=np.float64)
        nv.check(nv.lib.nsf_plan_fold_check(self.handle, frame.ctypes.data_as(C.POINTER(C.c_float)),
                                            re.ctypes.data_as(C.POINTER(C.c_double)),
                                            im.ctypes.data_as(C.POINTER(C.c_double))))
        return re + 1j * im

    def feature_cols(self, flags=0):
        return nv.lib.nsf_feature_cols(self.handle, flags)

    def hop_frames(self, n):
        return nv.lib.nsf_hop_frames(int(n), self.F, self.H)

    def feature_rows(self, n):
        return nv.lib.nsf_feature_rows(int(n), self.F, self.H)

    def guard_frames(self, n):
        return nv.lib.nsf_guard_frames(int(n), self.F, self.H)

    def __del__(self):
        try:
            if self.handle:
                nv.lib.nsf_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


def pack_clips(clips, dtype=None):
    """Concatenate 1-D clips into one packed array + int64 offsets."""
    lens = [len(c) for c in clips]
    offsets = np.zeros(len(clips) + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    if dtype is None:
        dtype = np.int16 if all(np.asarray(c).dtype == np.int16 for c in clips) else np.float32
    packed = np.empty(int(offsets[-1]), dtype=dtype)
    for c, o in zip(clips, offsets[:-1]):
        packed[o:o + len(c)] = c
    return packed, offsets


class Engine:
    """One CUDA context of the library on one device for one plan."""

    def __init__(self, plan, device=None):
        self.plan = plan
        self.device = default_device() if device is None else int(device)
        h = C.c_void_p()
        nv.check(nv.lib.nsf_ctx_create(plan.handle, self.device, C.byref(h)))
        self.handle = h
        self._lock = threading.Lock()

    # ---- geometry ------------------------------------------------------------------------
    def row_offsets(self, offsets, flags=0):
        """Prefix sum of the per-clip row counts (``nsf_row_offsets``: one call for the whole batch)."""
        off, off_p = nv.i64_array(offsets)
        out = np.empty(len(off), dtype=np.int64)
        nv.check(nv.lib.nsf_row_offsets(self.plan.F, self.plan.H, off_p, len(off) - 1, int(flags),
                                        out.ctypes.data_as(nv._i64p)))
        return out

    @staticmethod
    def _pcm_format(arr):
        if arr.dtype == np.float32:
            return nv.PCM_F32
        if arr.dtype == np.int16:
            return nv.PCM_I16
        raise TypeError(f"PCM must be float32 or int16, got {arr.dtype}")

    # ---- host buffers ----------------------------------------------------------------------
    def extract_host(self, pcm, offsets, flags=0, out=None, want_y=False):
        """pcm: packed 1-D float32/int16 host array; returns (rows x cols float32[, y float32])."""
        pcm = np.ascontiguousarray(pcm)
        fmt = self._pcm_format(pcm)
        off, off_p = nv.i64_array(offsets)
        n = len(off) - 1
        cols = self.plan.feature_cols(flags)
        rows = int(self.row_offsets(off, flags)[-1])
        if out is None:
            out = np.empty((rows, cols), dtype=np.float32)
        assert out.dtype == np.float32 and out.shape == (rows, cols) and out.flags["C_CONTIGUOUS"]
        y = np.empty(int(off[-1] - off[0]), dtype=np.float32) if want_y else None
        with self._lock:
            nv.check(nv.lib.nsf_extract_host(self.handle, nv.ptr(pcm), fmt, off_p, n, flags, nv.ptr(out),
                                             cols, nv.ptr(y) if want_y else None))
        return (out, y) if want_y else out

    def normalize_host(self, pcm, offsets=None):
        """Peak-normalise packed clips on the device (load_audio.py:12-14) -> float32 host array."""
        pcm = np.ascontiguousarray(pcm)
        fmt = self._pcm_format(pcm)
        if offsets is None:
            offsets = [0, len(pcm)]
        off, off_p = nv.i64_array(offsets)
        y = np.empty(int(off[-1] - off[0]), dtype=np.float32)
        if y.size == 0:
            return y
        with self._lock:
            nv.check(nv.lib.nsf_normalize_host(self.handle, nv.ptr(pcm), fmt, off_p, len(off) - 1,
                                               nv.ptr(y), None))
        return y

    def resample_host(self, pcm, orig_sr, target_sr, quality="hq"):
        """``librosa.resample(y, orig_sr=, target_sr=)`` stand-in on the device (load_audio.py:8-10):
        rational polyphase filter -> float32 host array of ``nsf_resample_len`` samples.  ``quality``:
        "hq" = band-limited windowed sinc (64 zero crossings, Kaiser beta 14.77; torchaudio's
        sinc_interp_kaiser arithmetic, the class of the reference's soxr_hq), "poly" = the
        scipy.signal.resample_poly design (see include/nsf.h)."""
        q = {"hq": nv.RESAMPLE_HQ, "poly": nv.RESAMPLE_POLY}[quality]
        nv.check(nv.lib.nsf_ctx_set_option(self.handle, nv.OPT_RESAMPLE_QUALITY, float(q)))
        pcm = np.ascontiguousarray(pcm)
        fmt = self._pcm_format(pcm)
        n_out = int(nv.lib.nsf_resample_len(len(pcm), int(orig_sr), int(target_sr)))
        out = np.empty(n_out, dtype=np.float32)
        if n_out == 0:
            return out
        with self._lock:
            nv.check(nv.lib.nsf_resample_host(self.handle, nv.ptr(pcm), fmt, len(pcm), int(orig_sr),
                                              int(target_sr), nv.ptr(out), n_out))
        return out

    def _set_quality(self, quality):
        q = {"hq": nv.RESAMPLE_HQ, "poly": nv.RESAMPLE_POLY}[quality]
        nv.check(nv.lib.nsf_ctx_set_option(self.handle, nv.OPT_RESAMPLE_QUALITY, float(q)))

    # ---- WAV conversion: raw data-chunk bytes -> mono float32 at a target rate -----------------------
    @staticmethod
    def convert_offsets(sources, target_sr, payload_bytes):
        """Output packing of a conversion: prefix sum of the per-clip lengths (``nsf_convert_offsets``)."""
        return nv.convert_offsets(sources, target_sr, payload_bytes)

    def convert_host(self, payload, sources, target_sr, quality="hq", out=None):
        """Decode + downmix + resample a ragged batch of WAV clips on the device (``nsf_convert_host``).

        ``payload``: 1-D uint8 host array of raw data-chunk bytes; ``sources``: ``nv.PCM_SOURCE`` array (or
        tuples ``(byte_offset, frames, encoding, channels, sample_rate)``).  Returns ``(float32 samples,
        offsets)``; clip i is ``out[offsets[i]:offsets[i + 1]]``, bit for bit ``decode_wav`` followed by
        ``resample_host(.., quality)``."""
        payload = np.ascontiguousarray(payload).view(np.uint8).reshape(-1)
        src = nv.pcm_sources(sources)
        off = nv.convert_offsets(src, target_sr, payload.nbytes)
        if out is None:
            out = np.empty(int(off[-1]), dtype=np.float32)
        assert out.dtype == np.float32 and out.flags["C_CONTIGUOUS"] and out.size >= int(off[-1])
        with self._lock:
            self._set_quality(quality)
            nv.check(nv.lib.nsf_convert_host(self.handle, nv.ptr(payload), payload.nbytes, nv.ptr(src), len(src),
                                             int(target_sr), nv.ptr(out)))
        return out[:int(off[-1])], off

    def convert_device(self, payload, sources, target_sr, quality="hq", out=None, stream=None):
        """``convert_host`` on device memory (``nsf_convert_batch``, stream-ordered): ``payload`` is a 1-D uint8
        CUDA tensor; returns ``(float32 CUDA tensor, offsets)``, ready for ``extract_device``."""
        import torch
        assert payload.is_cuda and payload.device.index == self.device and payload.is_contiguous()
        assert payload.dtype == torch.uint8
        src = nv.pcm_sources(sources)
        off = nv.convert_offsets(src, target_sr, payload.numel())
        if out is None:
            out = torch.empty(int(off[-1]), dtype=torch.float32, device=payload.device)
        assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() >= int(off[-1])
        s = torch.cuda.current_stream(payload.device) if stream is None else stream
        with self._lock:
            self._set_quality(quality)
            nv.check(nv.lib.nsf_convert_batch(self.handle, C.c_void_p(s.cuda_stream), C.c_void_p(payload.data_ptr()),
                                              payload.numel(), nv.ptr(src), len(src), int(target_sr),
                                              C.c_void_p(out.data_ptr()), off.ctypes.data_as(nv._i64p)))
        return out[:int(off[-1])], off

    # ---- training windows of a packed dataset (dataset/dataset.py:58-98) ------------------------------
    @staticmethod
    def window_offsets(audio_offsets, facial_offsets, window):
        """First window of every clip, plus the total (``nsf_window_offsets``): the numbering of
        ``AudioFacialDataset``'s items.  Raises ``NsfError`` for the clips the host windowing rejects."""
        return nv.window_offsets(audio_offsets, facial_offsets, window)

    def window_gather(self, audio, audio_offsets, facial, facial_offsets, window, indices, out_audio=None,
                      out_facial=None, stream=None):
        """Windows ``indices`` of a packed dataset on the device (``nsf_window_gather``, stream-ordered):
        ``audio [sum N, a_cols]`` / ``facial [sum N, f_cols]`` float32 CUDA tensors, clip i owning rows
        ``[offsets[i], offsets[i + 1])`` of each; ``indices`` a host sequence (list, NumPy array or CPU tensor).
        Returns ``(out_audio [n, window, a_cols], out_facial [n, window, f_cols])``, bit for bit what
        ``collate_fn([dataset[i] for i in indices])`` gives.  Indices and geometry are checked on the host first:
        on error nothing is launched and the outputs are not touched."""
        import torch
        for t in (audio, facial):
            assert t.is_cuda and t.device.index == self.device and t.dtype == torch.float32
            assert t.dim() == 2 and t.is_contiguous()
        if isinstance(indices, torch.Tensor):
            if indices.is_cuda:
                raise ValueError("window_gather: indices are validated on the host; pass a host sequence")
            indices = indices.numpy()
        idx, idx_p = nv.i64_array(np.asarray(indices).reshape(-1))
        a_off, a_p = nv.i64_array(audio_offsets)
        f_off, f_p = nv.i64_array(facial_offsets)
        if len(a_off) != len(f_off) or len(a_off) < 2:
            raise ValueError("audio and facial offsets need the same length, at least 2")
        if a_off[-1] > audio.shape[0] or f_off[-1] > facial.shape[0]:
            raise ValueError("offsets run past the rows of the packed tensors")
        n, window = len(idx), int(window)
        a_cols, f_cols = audio.shape[1], facial.shape[1]
        if out_audio is None:
            out_audio = torch.empty((n, window, a_cols), dtype=torch.float32, device=audio.device)
        if out_facial is None:
            out_facial = torch.empty((n, window, f_cols), dtype=torch.float32, device=audio.device)
        for t, cols in ((out_audio, a_cols), (out_facial, f_cols)):
            assert t.is_cuda and t.device.index == self.device and t.dtype == torch.float32 and t.is_contiguous()
            assert tuple(t.shape) == (n, window, cols), (tuple(t.shape), (n, window, cols))
        s = torch.cuda.current_stream(audio.device) if stream is None else stream
        with self._lock:
            nv.check(nv.lib.nsf_window_gather(
                self.handle, C.c_void_p(s.cuda_stream), C.c_void_p(audio.data_ptr()), a_cols, a_p,
                C.c_void_p(facial.data_ptr()), f_cols, f_p, len(a_off) - 1, window, idx_p, n,
                C.c_void_p(out_audio.data_ptr()), C.c_void_p(out_facial.data_ptr())))
        return out_audio, out_facial

    # ---- device buffers (torch used for memory and streams only) -------------------------------
    def workspace_bytes(self, total_samples, n_clips, flags=0):
        return nv.lib.nsf_workspace_bytes(self.plan.handle, int(total_samples), int(n_clips), flags)

    def extract_device(self, pcm, offsets, flags=0, out=None, workspace=None, y_norm=None, stream=None):
        """pcm: 1-D CUDA tensor (float32 or int16) on this engine's device.  Stream-ordered."""
        import torch
        assert pcm.is_cuda and pcm.device.index == self.device and pcm.is_contiguous()
        fmt = {torch.float32: nv.PCM_F32, torch.int16: nv.PCM_I16}[pcm.dtype]
        off, off_p = nv.i64_array(offsets)
        n = len(off) - 1
        cols = self.plan.feature_cols(flags)
        rows = int(self.row_offsets(off, flags)[-1])
        if out is None:
            out = torch.empty((rows, cols), dtype=torch.float32, device=pcm.device)
        assert out.dtype == torch.float32 and out.shape[0] == rows and out.stride(1) == 1
        need = self.workspace_bytes(int(off[-1] - off[0]), n, flags)
        if workspace is None or workspace.numel() < need:
            workspace = torch.empty(need, dtype=torch.uint8, device=pcm.device)
        s = torch.cuda.current_stream(pcm.device) if stream is None else stream
        base = pcm.data_ptr() + int(off[0]) * pcm.element_size()
        with self._lock:
            nv.check(nv.lib.nsf_extract_batch(
                self.handle, C.c_void_p(s.cuda_stream), C.c_void_p(base), fmt, off_p, n, flags,
                C.c_void_p(out.data_ptr()), out.stride(0), None,
                C.c_void_p(y_norm.data_ptr()) if y_norm is not None else None,
                C.c_void_p(workspace.data_ptr()), workspace.numel()))
        return out, workspace

    # ---- collect_features augmentation -----------------------------------------------------
    @staticmethod
    def collect_flags(include_fast=True, include_slow=False, blend_boundaries=True):
        return ((nv.COLLECT_FAST if include_fast else 0) | (nv.COLLECT_SLOW if include_slow else 0) |
                (nv.COLLECT_BLEND if blend_boundaries else 0))

    def collect_rows(self, audio_offsets, facial_offsets, include_fast=True, include_slow=False,
                     blend_boundaries=True, blend_frames=30):
        """Prefix sum of ``nsf_collect_rows`` per clip (output packing of the collect calls)."""
        a_off = np.asarray(audio_offsets, dtype=np.int64)
        f_off = np.asarray(facial_offsets, dtype=np.int64)
        flags = self.collect_flags(include_fast, include_slow, blend_boundaries)
        rows = [nv.lib.nsf_collect_rows(int(a_off[i + 1] - a_off[i]), int(f_off[i + 1] - f_off[i]), flags,
                                        int(blend_frames)) for i in range(len(a_off) - 1)]
        o_off = np.zeros(len(rows) + 1, dtype=np.int64)
        np.cumsum(rows, out=o_off[1:])
        return o_off

    def collect_device(self, audio, audio_offsets, facial, facial_offsets, include_fast=True,
                       include_slow=False, blend_boundaries=True, blend_frames=30, out_audio=None,
                       out_facial=None, stream=None, out_offsets=None):
        """Device-resident ``collect_features`` arithmetic (``nsf_collect_batch``): CUDA tensors in
        (float32 or float64, packed rows), CUDA tensors out.  Stream-ordered, no host sync."""
        import torch
        assert audio.is_cuda and facial.is_cuda and audio.dtype == facial.dtype
        assert audio.is_contiguous() and facial.is_contiguous()
        dtype = {torch.float32: nv.F32, torch.float64: nv.F64}[audio.dtype]
        a_off, a_p = nv.i64_array(audio_offsets)
        f_off, f_p = nv.i64_array(facial_offsets)
        # out_offsets: the caller's cached result of collect_rows() for these inputs (saves n_clips small calls)
        o_off = (self.collect_rows(a_off, f_off, include_fast, include_slow, blend_boundaries, blend_frames)
                 if out_offsets is None else np.ascontiguousarray(out_offsets, dtype=np.int64))
        _, o_p = nv.i64_array(o_off)
        n_out = int(o_off[-1])
        if out_audio is None:
            out_audio = torch.empty((n_out, audio.shape[1]), dtype=audio.dtype, device=audio.device)
        if out_facial is None:
            out_facial = torch.empty((n_out, facial.shape[1]), dtype=audio.dtype, device=audio.device)
        s = torch.cuda.current_stream(audio.device) if stream is None else stream
        flags = self.collect_flags(include_fast, include_slow, blend_boundaries)
        with self._lock:
            nv.check(nv.lib.nsf_collect_batch(
                self.handle, C.c_void_p(s.cuda_stream), dtype, C.c_void_p(audio.data_ptr()), audio.shape[1], a_p,
                C.c_void_p(facial.data_ptr()), facial.shape[1], f_p, len(a_off) - 1, flags, int(blend_frames),
                C.c_void_p(out_audio.data_ptr()), C.c_void_p(out_facial.data_ptr()), o_p))
        return out_audio, out_facial, o_off

    def extract_collect_host(self, pcm, offsets, facial, facial_offsets, flags=0, include_fast=True,
                             include_slow=False, blend_boundaries=True, blend_frames=30, out_audio=None,
                             out_facial=None, features_out=None):
        """Features of a batch of clips AND their ``collect_features`` augmentation in one pipelined pass
        (``nsf_extract_collect_host``): the feature rows stay on the device between the two steps.
        float32 in (facial) and out; returns (audio rows, facial rows, output row offsets).
        ``features_out`` (optional ``[sum R_i, cols]`` float32) also receives the un-augmented rows."""
        pcm = np.ascontiguousarray(pcm)
        fmt = self._pcm_format(pcm)
        facial = np.ascontiguousarray(facial, dtype=np.float32)
        off, off_p = nv.i64_array(offsets)
        f_off, f_p = nv.i64_array(facial_offsets)
        cols = self.plan.feature_cols(flags)
        o_off = self.collect_rows(self.row_offsets(off, flags), f_off, include_fast, include_slow,
                                  blend_boundaries, blend_frames)
        n_out = int(o_off[-1])
        if out_audio is None:
            out_audio = np.empty((n_out, cols), dtype=np.float32)
        if out_facial is None:
            out_facial = np.empty((n_out, facial.shape[1]), dtype=np.float32)
        assert out_audio.shape == (n_out, cols) and out_facial.shape == (n_out, facial.shape[1])
        cflags = self.collect_flags(include_fast, include_slow, blend_boundaries)
        if features_out is not None:
            n_rows = int(self.row_offsets(off, flags)[-1])
            assert features_out.dtype == np.float32 and features_out.shape == (n_rows, cols)
        with self._lock:
            nv.check(nv.lib.nsf_extract_collect_host(self.handle, nv.ptr(pcm), fmt, off_p, len(off) - 1, flags,
                                                     nv.ptr(facial), facial.shape[1], f_p, cflags,
                                                     int(blend_frames), nv.ptr(out_audio), nv.ptr(out_facial),
                                                     nv.ptr(features_out)))
        return out_audio, out_facial, o_off

    def collect_host(self, audio, audio_offsets, facial, facial_offsets, include_fast=True,
                     include_slow=False, blend_boundaries=True, blend_frames=30):
        """Packed row-major audio / facial rows (same float dtype) -> augmented (audio, facial, offsets)."""
        audio = np.ascontiguousarray(audio)
        facial = np.ascontiguousarray(facial, dtype=audio.dtype)
        dtype = {np.dtype(np.float32): nv.F32, np.dtype(np.float64): nv.F64}[audio.dtype]
        a_off, a_p = nv.i64_array(audio_offsets)
        f_off, f_p = nv.i64_array(facial_offsets)
        n = len(a_off) - 1
        flags = self.collect_flags(include_fast, include_slow, blend_boundaries)
        rows = [nv.lib.nsf_collect_rows(int(a_off[i + 1] - a_off[i]), int(f_off[i + 1] - f_off[i]), flags,
                                        int(blend_frames)) for i in range(n)]
        o_off = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(rows, out=o_off[1:])
        out_a = np.empty((int(o_off[-1]), audio.shape[1]), dtype=audio.dtype)
        out_f = np.empty((int(o_off[-1]), facial.shape[1]), dtype=audio.dtype)
        with self._lock:
            nv.check(nv.lib.nsf_collect_host(self.handle, dtype, nv.ptr(audio), audio.shape[1], a_p,
                                             nv.ptr(facial), facial.shape[1], f_p, n, flags,
                                             int(blend_frames), nv.ptr(out_a), nv.ptr(out_f)))
        return out_a, out_f, o_off

    def rows_op(self, op, a, b=None, blend_frames=0):
        a = np.ascontiguousarray(a)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)
        dtype = nv.F64 if a.dtype == np.float64 else nv.F32
        na, cols = a.shape
        nb = 0
        if b is not None:
            b = np.ascontiguousarray(b, dtype=a.dtype)
            nb = b.shape[0]
            assert b.shape[1] == cols
        if op == nv.ROWS_INTERP_SLOWER:
            rows = 2 * na - 1
        elif op == nv.ROWS_SMOOTH:
            rows = na
        else:
            rows = na + nb - max(0, min(int(blend_frames), na, nb))
        out = np.empty((rows, cols), dtype=a.dtype)
        with self._lock:
            nv.check(nv.lib.nsf_rows_host(self.handle, op, dtype, nv.ptr(a), na, nv.ptr(b) if b is not None
                                          else None, nb, cols, int(blend_frames), nv.ptr(out)))
        return out

    def post(self, frame_major, post_flags):
        x = np.ascontiguousarray(frame_major, dtype=np.float32)
        t, c = x.shape
        rows = (t + 1) // 2 if post_flags & 0x8 else t
        out = np.empty((rows, c * (3 if post_flags & 0x4 else 1)), dtype=np.float32)
        with self._lock:
            nv.check(nv.lib.nsf_post_host(self.handle, x.ctypes.data_as(C.POINTER(C.c_float)), t, c,
                                          post_flags, nv.ptr(out)))
        return out

    # ---- instrumentation ---------------------------------------------------------------------
    def launch_count(self):
        return nv.lib.nsf_launch_count(self.handle)

    def set_edge_zero_threshold(self, value):
        """``zero_threshold`` of ``fix_edge_frames_autocorr`` (extract_features_utils.py:105) for this context."""
        nv.check(nv.lib.nsf_ctx_set_option(self.handle, nv.OPT_EDGE_ZERO_THRESHOLD, float(value)))

    def set_profiling(self, on):
        nv.lib.nsf_set_profiling(self.handle, 1 if on else 0)

    def stage_times_ms(self):
        buf = (C.c_float * 8)()
        n = nv.lib.nsf_stage_times_ms(self.handle, buf, 8)
        return {nv.STAGE_NAMES[i]: float(buf[i]) for i in range(n)}

    def close(self):
        if self.handle:
            nv.lib.nsf_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_plans = {}
_engines = {}
_cache_lock = threading.Lock()


def get_plan(sr, frame_length, hop_length, n_mfcc=DEFAULT_N_MFCC, n_lags=DEFAULT_N_LAGS):
    key = (int(sr), int(frame_length), int(hop_length), int(n_mfcc), DEFAULT_N_MELS, int(n_lags))
    with _cache_lock:
        if key not in _plans:
            _plans[key] = Plan(*key)
        return _plans[key]


def get_engine(sr, frame_length, hop_length, device=None, n_mfcc=DEFAULT_N_MFCC, n_lags=DEFAULT_N_LAGS):
    device = default_device() if device is None else int(device)
    key = (int(sr), int(frame_length), int(hop_length), int(n_mfcc), int(n_lags), device)
    plan = get_plan(sr, frame_length, hop_length, n_mfcc, n_lags)
    with _cache_lock:
        if key not in _engines:
            _engines[key] = Engine(plan, device)
        return _engines[key]

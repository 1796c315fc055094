"""The HotwordDetector.start loop (detector.py:148-209) for S lock-step streams.

``StreamingDetector.step(chunk)`` is one pass of the reference's ``while True`` body
for every stream at once: VAD reset, tail carry, model call, 15-chunk window,
``ctc_decode2`` + ``ctc_predict``, trigger reset -- all on the device, all per-stream
state in HBM (kws_stream_* in include/kws_b200.h).
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib, _tensors
from .rnn_ctc import DeployModel


class StreamingDetector:
    def __init__(self, model: DeployModel, n_streams: int, max_chunk: int = None, window_chunks: int = None,
                 vad_threshold: int = None, decode_thres: float = None, keyword: str = None):
        cfg = model.config
        self.model = model
        self.device = model.device
        self.n_streams = int(n_streams)
        self.max_chunk = int(max_chunk if max_chunk is not None else cfg.chunk_samples)
        self._lib = _lib.load()
        sc = _lib.StreamConfig()
        sc.n_streams = self.n_streams
        sc.max_chunk = self.max_chunk
        sc.window_chunks = int(window_chunks if window_chunks is not None else cfg.window_chunks)
        sc.vad_threshold = int(vad_threshold if vad_threshold is not None else cfg.vad_threshold)
        sc.decode_thres = float(decode_thres if decode_thres is not None else cfg.decode_thres)
        sc.keyword = (keyword if keyword is not None else cfg.label_seqs).encode("ascii")
        handle = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.kws_stream_create(model.handle, ctypes.byref(sc), ctypes.byref(handle)))
        self._handle = handle
        self.max_frames = int(self._lib.kws_stream_max_frames(handle))
        self._trigger = torch.zeros(self.n_streams, dtype=torch.int32, device=self.device)
        self._pinned_trigger = None

    def close(self):
        if getattr(self, "_handle", None):
            self._lib.kws_stream_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        with torch.cuda.device(self.device):
            _lib.check(self._lib.kws_stream_reset(self._handle, _tensors.stream_ptr(self.device)))

    def step(self, chunk, want_probs=False):
        """chunk ``[S, n]`` int16 (numpy -> numpy results, CUDA tensor -> CUDA results).

        Returns ``trigger [S]`` int32, or ``(trigger, probs [S, max_frames, C], nframes [S])``.
        """
        host = _tensors.is_host(chunk)
        x = _tensors.to_device(chunk, torch.int16, self.device)
        if x.dim() != 2 or x.shape[0] != self.n_streams:
            raise _lib.InvalidArgumentError("chunk must be [%d, n] int16" % self.n_streams)
        C = self.model.config.num_classes
        trig = torch.empty(self.n_streams, dtype=torch.int32, device=self.device)
        probs = nfr = None
        if want_probs:
            probs = torch.zeros((self.n_streams, self.max_frames, C), dtype=torch.float32, device=self.device)
            nfr = torch.empty(self.n_streams, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.kws_stream_step(self._handle, _tensors.ptr(x), x.shape[1], x.stride(0), _tensors.ptr(trig),
                                                 _tensors.ptr(probs), _tensors.ptr(nfr), _tensors.stream_ptr(self.device)))
        outs = (trig, probs, nfr) if want_probs else (trig,)
        if host:
            torch.cuda.current_stream(self.device).synchronize()
            outs = tuple(_tensors.to_host(o) for o in outs)
        return outs if want_probs else outs[0]

    def step_host(self, pinned_chunk: torch.Tensor, pinned_trigger: torch.Tensor = None):
        """Enqueue H2D(chunk) -> step -> D2H(trigger) without synchronising.
        ``pinned_chunk`` ``[S, n]`` int16 pinned host tensor; returns the pinned trigger tensor
        (valid after the current stream is synchronised)."""
        if pinned_chunk.dtype != torch.int16 or pinned_chunk.dim() != 2 or pinned_chunk.shape[0] != self.n_streams \
                or not pinned_chunk.is_contiguous() or pinned_chunk.is_cuda:
            raise _lib.InvalidArgumentError("pinned_chunk must be a contiguous host int16 [%d, n] tensor" % self.n_streams)
        if pinned_trigger is None:
            if self._pinned_trigger is None:
                self._pinned_trigger = torch.zeros(self.n_streams, dtype=torch.int32).pin_memory()
            pinned_trigger = self._pinned_trigger
        with torch.cuda.device(self.device):
            _lib.check(self._lib.kws_stream_step_host(self._handle, pinned_chunk.data_ptr(), pinned_chunk.shape[1],
                                                      pinned_trigger.data_ptr(), _tensors.stream_ptr(self.device)))
        return pinned_trigger

    def state(self) -> torch.Tensor:
        """Copy of the carried GRU state ``[layers, S, H]`` (CUDA tensor)."""
        cfg = self.model.config
        out = torch.empty((cfg.num_layers, self.n_streams, cfg.hidden_size), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.kws_stream_copy_state(self._handle, _tensors.ptr(out), _tensors.stream_ptr(self.device)))
        return out

    def window_labels(self, max_labels=None):
        """Window decode of every stream as of the last step -> (labels [S, max_labels], counts [S]) numpy."""
        if max_labels is None:
            max_labels = 2 * self.max_frames * self.model.config.window_chunks + 1
        labels = torch.empty((self.n_streams, max_labels), dtype=torch.int32, device=self.device)
        counts = torch.empty(self.n_streams, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.kws_stream_labels(self._handle, _tensors.ptr(labels), max_labels, _tensors.ptr(counts),
                                                   _tensors.stream_ptr(self.device)))
        torch.cuda.current_stream(self.device).synchronize()
        return _tensors.to_host(labels), _tensors.to_host(counts)

    # -- per-stream records (kws_stream_export / kws_stream_import)
    @property
    def record_bytes(self) -> int:
        """Bytes of one stream's record (layout in include/kws_b200.h)."""
        return int(self._lib.kws_stream_record_bytes(self._handle))

    def export_streams(self, ids) -> torch.Tensor:
        """Records of streams ``ids`` -> ``torch.uint8`` CUDA ``[n, record_bytes]``: everything each stream carries
        into its next chunk, as plain bytes (move them to another GPU with ``.to(device)``, or to disk)."""
        idx = record_ids(ids, self.n_streams, self.device, distinct=False)
        out = torch.empty((idx.numel(), self.record_bytes), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.kws_stream_export(self._handle, _tensors.ptr(idx), idx.numel(), _tensors.ptr(out),
                                                   _tensors.stream_ptr(self.device)))
        return out

    def import_streams(self, ids, records):
        """Make streams ``ids`` continue from ``records`` (from ``export_streams`` of an object of the same layout,
        host or device).  Raises ``InvalidArgumentError`` naming every rejected record; those streams are left as
        they were.  Reads the status back, so it synchronises the current stream."""
        idx = record_ids(ids, self.n_streams, self.device, distinct=True)
        recs = record_input(records, idx.numel(), self.record_bytes, self.device)
        status = torch.empty(idx.numel(), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.kws_stream_import(self._handle, _tensors.ptr(idx), idx.numel(), _tensors.ptr(recs),
                                                   _tensors.ptr(status), _tensors.stream_ptr(self.device)))
        raise_rejected(idx, status)


_REJECTED = {1: "id out of range", 2: "header does not match this object", 3: "malformed field"}


def record_ids(ids, n_streams: int, device, distinct: bool) -> torch.Tensor:
    """ids -> int64 CUDA [n].  Host ids are validated (integers in [0, n_streams), distinct when ``distinct``); CUDA
    ids are left to the kernels (reading them here would synchronise the stream)."""
    if not _tensors.is_host(ids):
        if ids.dim() != 1 or ids.dtype.is_floating_point or ids.dtype.is_complex or ids.dtype == torch.bool:
            raise _lib.InvalidArgumentError("ids must be integers [n], got %s %r" % (ids.dtype, tuple(ids.shape)))
        return _tensors.to_device(ids, torch.int64, device)
    a = np.asarray(ids.numpy() if isinstance(ids, torch.Tensor) else ids)
    if a.ndim == 1 and a.size == 0:
        a = a.astype(np.int64)
    if a.ndim != 1 or a.dtype.kind not in "iu":
        raise _lib.InvalidArgumentError("ids must be integers [n], got %s %r" % (a.dtype, a.shape))
    if a.size and (a.min() < 0 or a.max() >= n_streams):
        raise _lib.InvalidArgumentError("ids must lie in [0, %d), got [%d, %d]" % (n_streams, a.min(), a.max()))
    if distinct and np.unique(a).size != a.size:
        raise _lib.InvalidArgumentError("ids must be distinct")
    return _tensors.to_device(a.astype(np.int64), torch.int64, device)


def record_input(records, n: int, record_bytes: int, device) -> torch.Tensor:
    """uint8 records (CUDA or host tensor, numpy array) of n * record_bytes bytes -> CUDA [n, record_bytes]."""
    if isinstance(records, torch.Tensor):
        ok = records.dtype == torch.uint8 and records.numel() == n * record_bytes
    else:
        records = np.asarray(records)
        if not records.flags.writeable:           # e.g. np.frombuffer of bytes read from a file
            records = records.copy()
        ok = records.dtype == np.uint8 and records.size == n * record_bytes
    if not ok:
        raise _lib.InvalidArgumentError("records must be uint8 [%d, %d], got %s %r" % (n, record_bytes, records.dtype,
                                                                                     tuple(records.shape)))
    return _tensors.to_device(records, torch.uint8, device).reshape(n, record_bytes)


def raise_rejected(ids: torch.Tensor, status: torch.Tensor):
    st = _tensors.to_host(status)
    bad = np.nonzero(st)[0]
    if bad.size:
        idv = _tensors.to_host(ids)
        raise _lib.InvalidArgumentError("%d record(s) rejected: %s" % (bad.size, "; ".join(
            "entry %d (id %d): %s" % (i, idv[i], _REJECTED.get(int(st[i]), "status %d" % st[i])) for i in bad[:16])))

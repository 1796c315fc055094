"""The serving loop of the reference (``HotwordDetector.start``, detector.py:148-212) for all the streams of a GPU.

``WaveServer`` is the host-side mirror of ``kws_server_*`` (include/kws_b200.h): the streams are split into waves,
each with its own stream object, CUDA stream, pinned ingest slots and a captured CUDA graph of the whole chunk
(H2D -> front end -> GRU -> decode/trigger -> D2H).  Producers write PCM into ``ingest_slot(wave)``; ``submit`` /
``wait`` (or ``serve`` for the steady-state loop) move the chunks; ``stats`` returns the per-chunk latency
percentiles the serving metric is defined on (SURVEY.md 8d).
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib, _tensors
from .rnn_ctc import DeployModel
from .streaming import raise_rejected, record_ids, record_input


class WaveServer:
    def __init__(self, model: DeployModel, n_streams: int, waves: int = 16, chunk_samples: int = None,
                 use_graphs: bool = True, window_chunks: int = None, vad_threshold: int = None,
                 decode_thres: float = None, keyword: str = None):
        cfg = model.config
        self.model = model
        self.device = model.device
        self.n_streams = int(n_streams)
        self.waves = int(waves)
        self.chunk_samples = int(chunk_samples if chunk_samples is not None else cfg.chunk_samples)
        self._lib = _lib.load()
        sc = _lib.ServerConfig()
        sc.n_streams = self.n_streams
        sc.waves = self.waves
        sc.chunk_samples = self.chunk_samples
        sc.use_graphs = 1 if use_graphs else 0
        sc.stream.window_chunks = int(window_chunks if window_chunks is not None else cfg.window_chunks)
        sc.stream.vad_threshold = int(vad_threshold if vad_threshold is not None else cfg.vad_threshold)
        sc.stream.decode_thres = float(decode_thres if decode_thres is not None else cfg.decode_thres)
        sc.stream.keyword = (keyword if keyword is not None else cfg.label_seqs).encode("ascii")
        handle = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.kws_server_create(model.handle, ctypes.byref(sc), ctypes.byref(handle)))
        self._handle = handle
        spw, w, g = ctypes.c_int64(0), ctypes.c_int32(0), ctypes.c_int32(0)
        _lib.check(self._lib.kws_server_info(handle, ctypes.byref(spw), ctypes.byref(w), ctypes.byref(g)))
        self.streams_per_wave = int(spw.value)
        self.graphs = bool(g.value)

    def close(self):
        if getattr(self, "_handle", None):
            self._lib.kws_server_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- ingest
    def ingest_slot(self, wave: int) -> np.ndarray:
        """The pinned host buffer ``[streams_per_wave, chunk_samples]`` int16 that the next ``submit(wave)`` sends
        (a numpy view, no copy)."""
        ptr = self._lib.kws_server_ingest_slot(self._handle, int(wave))
        if not ptr:
            raise _lib.InvalidArgumentError("wave %r out of range" % (wave,))
        n = self.streams_per_wave * self.chunk_samples
        buf = (ctypes.c_int16 * n).from_address(ptr)
        return np.frombuffer(buf, dtype=np.int16).reshape(self.streams_per_wave, self.chunk_samples)

    def submit(self, wave: int, chunk=None):
        """Enqueue the wave's chunk; ``chunk`` (``[streams_per_wave, chunk_samples]`` int16), if given, is copied into
        the ingest slot first."""
        if chunk is not None:
            src = chunk.cpu().numpy() if isinstance(chunk, torch.Tensor) else np.asarray(chunk)
            if src.shape != (self.streams_per_wave, self.chunk_samples) or src.dtype != np.int16:
                raise _lib.InvalidArgumentError("chunk must be int16 [%d, %d]" % (self.streams_per_wave, self.chunk_samples))
            self.ingest_slot(wave)[...] = src
        _lib.check(self._lib.kws_server_submit(self._handle, int(wave)))

    def wait(self, wave: int):
        """Block until the wave's oldest chunk in flight is done -> (trigger flags [streams_per_wave] int32 copy,
        latency in ms)."""
        ptr, ms = ctypes.c_void_p(), ctypes.c_double(0.0)
        _lib.check(self._lib.kws_server_wait(self._handle, int(wave), ctypes.byref(ptr), ctypes.byref(ms)))
        buf = (ctypes.c_int32 * self.streams_per_wave).from_address(ptr.value)
        return np.frombuffer(buf, dtype=np.int32).copy(), float(ms.value)

    def step(self, chunk) -> np.ndarray:
        """One chunk for EVERY stream (``[n_streams, chunk_samples]`` int16, host): all waves submitted, then waited
        for.  Returns the trigger flags ``[n_streams]``."""
        src = chunk.cpu().numpy() if isinstance(chunk, torch.Tensor) else np.asarray(chunk)
        if src.shape != (self.n_streams, self.chunk_samples):
            raise _lib.InvalidArgumentError("chunk must be int16 [%d, %d]" % (self.n_streams, self.chunk_samples))
        Sw = self.streams_per_wave
        for w in range(self.waves):
            self.submit(w, src[w * Sw:(w + 1) * Sw])
        return np.concatenate([self.wait(w)[0] for w in range(self.waves)])

    def serve(self, rounds: int, depth: int = 2):
        """``rounds`` chunks for every wave from the ingest slots as they are, at most ``depth`` waves in flight."""
        _lib.check(self._lib.kws_server_serve(self._handle, int(rounds), int(depth)))

    def stats(self, reset: bool = False) -> dict:
        p50, p99, mx = ctypes.c_double(0), ctypes.c_double(0), ctypes.c_double(0)
        n, trig = ctypes.c_int64(0), ctypes.c_int64(0)
        _lib.check(self._lib.kws_server_stats(self._handle, 1 if reset else 0, ctypes.byref(p50), ctypes.byref(p99),
                                              ctypes.byref(mx), ctypes.byref(n), ctypes.byref(trig)))
        return dict(unit="ms", p50=p50.value, p99=p99.value, max=mx.value, samples=int(n.value), triggers=int(trig.value))

    def set_copy_only(self, on: bool):
        _lib.check(self._lib.kws_server_set_copy_only(self._handle, 1 if on else 0))

    def reset(self):
        _lib.check(self._lib.kws_server_reset(self._handle))

    # -- inspection
    def state(self) -> torch.Tensor:
        """Carried GRU state of every stream ``[layers, n_streams, H]`` (CUDA tensor)."""
        cfg = self.model.config
        Sw = self.streams_per_wave
        out = torch.empty((cfg.num_layers, self.n_streams, cfg.hidden_size), dtype=torch.float32, device=self.device)
        part = torch.empty((cfg.num_layers, Sw, cfg.hidden_size), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            for w in range(self.waves):
                st = self._lib.kws_server_wave_stream(self._handle, w)
                torch.cuda.synchronize(self.device)
                _lib.check(self._lib.kws_stream_copy_state(st, _tensors.ptr(part), _tensors.stream_ptr(self.device)))
                out[:, w * Sw:(w + 1) * Sw] = part
        return out

    def window_labels(self, max_labels: int = 64):
        """Window decode of every stream as of its last chunk -> (labels [n_streams, max_labels], counts) numpy."""
        Sw = self.streams_per_wave
        labels = torch.empty((self.n_streams, max_labels), dtype=torch.int32, device=self.device)
        counts = torch.empty(self.n_streams, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            torch.cuda.synchronize(self.device)
            for w in range(self.waves):
                st = self._lib.kws_server_wave_stream(self._handle, w)
                _lib.check(self._lib.kws_stream_labels(st, labels[w * Sw:].data_ptr(), max_labels,
                                                       counts[w * Sw:].data_ptr(), _tensors.stream_ptr(self.device)))
            torch.cuda.synchronize(self.device)
        return _tensors.to_host(labels), _tensors.to_host(counts)

    # -- per-stream records over global stream ids (kws_server_export / kws_server_import)
    @property
    def record_bytes(self) -> int:
        """Bytes of one stream's record (the layout of ``StreamingDetector.export_streams``)."""
        return int(self._lib.kws_stream_record_bytes(self._lib.kws_server_wave_stream(self._handle, 0)))

    def export_streams(self, ids) -> torch.Tensor:
        """Records of global streams ``ids`` -> ``torch.uint8`` CUDA ``[n, record_bytes]``.  Nothing may be in
        flight; returns when the records are written."""
        idx = record_ids(ids, self.n_streams, self.device, distinct=False)
        out = torch.empty((idx.numel(), self.record_bytes), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.kws_server_export(self._handle, _tensors.ptr(idx), idx.numel(), _tensors.ptr(out),
                                                   _tensors.stream_ptr(self.device)))
        return out

    def import_streams(self, ids, records):
        """Make global streams ``ids`` continue from ``records`` (host or device); the next ``submit`` sees them.
        Nothing may be in flight.  Raises ``InvalidArgumentError`` naming every rejected record."""
        idx = record_ids(ids, self.n_streams, self.device, distinct=True)
        recs = record_input(records, idx.numel(), self.record_bytes, self.device)
        status = torch.empty(idx.numel(), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.kws_server_import(self._handle, _tensors.ptr(idx), idx.numel(), _tensors.ptr(recs),
                                                   _tensors.ptr(status), _tensors.stream_ptr(self.device)))
        raise_rejected(idx, status)

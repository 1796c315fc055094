"""Offline evaluation harness: the validation branch of the reference's driver (main.py:263-314, and the
in-training copy :169-217) on the GPU path.

For every batch: softmax of the utterances -> ``ctc_decode`` per utterance (main.py:290) ->
``ctc_predict(seq, label_seqs)`` (:291) -> ``evaluate(result, correctness)`` (:303-304) accumulated into the
miss / false-accept counts the reference prints (:311-314).  Decoding and the keyword test run on the device
for the whole batch (``kws_ctc_decode``); nothing here falls back to the CPU.
"""
from __future__ import annotations

from typing import Iterable, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib, _tensors
from .utils import prediction


class ValidationResult(dict):
    """miss / target / false_accept / total counts with the reference's two printed rates."""

    @property
    def miss_rate(self):
        return self["miss"] / self["target"] if self["target"] else 0.0

    @property
    def false_accept_rate(self):
        neg = self["total"] - self["target"]
        return self["false_accept"] / neg if neg else 0.0

    def report(self) -> str:                               # main.py:311-314
        return ("--------------------------------\nmiss rate: %d/%d\nflase_accept_rate: %d/%d"
                % (self["miss"], self["target"], self["false_accept"], self["total"] - self["target"]))


def evaluate_softmax(softmax, correctness, lens=None, label_seqs: str = "1233", device=None):
    """One validation batch given its posteriors.

    softmax ``[B, T, C]`` (numpy or CUDA tensor), correctness ``[B]`` 0/1, lens ``[B]`` valid frames or None.
    Returns (miss, target, false_accept, result[B]) exactly as main.py:290-304 computes them.
    """
    _, _, trig = prediction.decode_batch(softmax, lens=lens, mode=prediction.MODE_CTC_DECODE, keyword=label_seqs,
                                         device=device, want_labels=False)
    trig_t = trig if isinstance(trig, torch.Tensor) else torch.from_numpy(np.asarray(trig))
    if isinstance(correctness, torch.Tensor):
        tgt = correctness.to(device=trig_t.device, dtype=torch.int32)
    else:
        tgt = torch.from_numpy(np.asarray(correctness, np.int32)).to(trig_t.device)
    if tgt.shape != trig_t.shape:
        raise _lib.InvalidArgumentError("correctness must have one entry per utterance")
    xor = tgt ^ trig_t                                     # utils/prediction.py:203-210
    miss = int((xor & tgt).sum())
    false_accept = int((xor & trig_t).sum())
    return miss, int(tgt.sum()), false_accept, trig_t.cpu().numpy()


def validate(model, batches: Iterable[Tuple], label_seqs: Optional[str] = None,
             sample_lengths: bool = False) -> ValidationResult:
    """Run the validation set through ``model`` (a DeployModel or an AttentionDeployModel).

    ``batches`` yields ``(inputs, lens, correctness)``: inputs are mel frames ``[B, T, n_mel]`` (the valid
    queue's form, reader.py:282-305) or PCM ``[B, L]``; ``lens`` valid frames per utterance (or None).
    By default PCM rows are taken as equal-length utterances.  With ``sample_lengths``, the ``lens`` of PCM batches are
    valid samples per utterance: each model runs ``forward(..., lengths=lens)``, and the decoder takes its frame counts
    (``frame_counts(lens)``; ``output_lengths`` of those for the attention model).  For the attention model the
    ``lens`` of mel batches are mel frames: they run with them, and the decoder takes ``output_lengths(lens)``.
    """
    from .attention_ctc import AttentionDeployModel
    label_seqs = label_seqs or model.config.label_seqs
    res = ValidationResult(miss=0, target=0, false_accept=0, total=0)
    for inputs, lens, correctness in batches:
        x = inputs if isinstance(inputs, torch.Tensor) else np.asarray(inputs)
        B = x.shape[0]
        attention = isinstance(model, AttentionDeployModel)
        if x.ndim == 3:
            mel = _tensors.to_device(x, torch.float32, model.device)
        else:
            is_i16 = x.dtype in (np.int16, torch.int16)
            pcm = _tensors.to_device(x, torch.int16 if is_i16 else torch.float32, model.device)
        by_samples = sample_lengths and x.ndim != 3 and lens is not None
        if attention and by_samples:
            probs = model(pcm, lengths=lens)
            dec_lens = model.output_lengths(model.frame_counts(lens))
        elif attention:
            probs = model.run_mel(mel, lens=lens) if x.ndim == 3 else model(pcm)
            dec_lens = None if lens is None else model.output_lengths(lens)
        else:
            state = torch.zeros((model.config.num_layers, B, model.config.hidden_size), dtype=torch.float32, device=model.device)
            if by_samples:
                probs, _ = model(pcm, state, lengths=lens)
                dec_lens = model.frame_counts(lens)
            else:
                probs, _ = model.run_mel(mel, state, seq_len=lens) if x.ndim == 3 else model(pcm, state)
                dec_lens = lens
        miss, target, fa, _ = evaluate_softmax(probs, correctness, lens=dec_lens, label_seqs=label_seqs)
        res["miss"] += miss
        res["target"] += target
        res["false_accept"] += fa
        res["total"] += B
    return res

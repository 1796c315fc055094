"""CPU reference for variable-length attention_ctc batches: every utterance alone through oracle.attention.

The deployment graph (models/attention_ctc.py:215-274) has no padding mask and is run one utterance at a time
(batch-1 sess.run), so the reference for utterance b of a padded batch is the graph on mel[b, :lens[b]] alone.
"""
import numpy as np

from oracle import attention as oa


def mel_forward_lens(mel, lens, w, dtype=np.float32, use_relu=True, combine=oa.COMBINE):
    """mel [B, T, M], lens [B] valid frames -> (softmax, logits) [B, T', C], T' = T // combine + 1 (the oracle's
    padding rule).  Row block b is oa.mel_forward(mel[b, :lens[b]]); rows past that utterance's T'_b are zero."""
    mel = np.asarray(mel)
    B, T, _ = mel.shape
    C = np.asarray(w.w_out).shape[1]
    Tp = T // combine + 1
    probs = np.zeros((B, Tp, C), dtype)
    logits = np.zeros((B, Tp, C), dtype)
    for b in range(B):
        p, l = oa.mel_forward(mel[b:b + 1, :int(lens[b])], w, dtype, use_relu=use_relu, combine=combine)
        probs[b, :p.shape[1]] = p[0]
        logits[b, :l.shape[1]] = l[0]
    return probs, logits

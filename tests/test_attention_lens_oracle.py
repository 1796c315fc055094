"""CPU: the per-utterance reference for variable-length attention_ctc batches."""
import numpy as np

from oracle import attention as oa
from tests._attention_lens import mel_forward_lens


def _weights():
    return oa.init_weights(seed=7, n_mel=20, layers=1, ffn=64)


def test_mel_forward_lens_equals_mel_forward_at_full_length():
    w = _weights()
    mel = np.abs(np.random.default_rng(0).standard_normal((3, 9, 20))).astype(np.float32)
    got, lgot = mel_forward_lens(mel, [9, 9, 9], w)
    want, lwant = oa.mel_forward(mel, w)
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(lgot, lwant)


def test_mel_forward_lens_is_each_utterance_alone_and_ignores_padding():
    w = _weights()
    rng = np.random.default_rng(1)
    lens = [1, 2, 5, 6, 12]
    mel = np.abs(rng.standard_normal((5, 12, 20))).astype(np.float32)
    for b, n in enumerate(lens):
        mel[b, n:] = np.nan                        # frames past an utterance's length never count
    got, lgot = mel_forward_lens(mel, lens, w, np.float64)
    assert got.shape == (5, 12 // 2 + 1, 6)
    for b, n in enumerate(lens):
        want, lwant = oa.mel_forward(mel[b:b + 1, :n], w, np.float64)
        Tb = n // 2 + 1                            # odd n: the last group holds one frame and zeros
        assert want.shape[1] == Tb
        np.testing.assert_array_equal(got[b, :Tb], want[0])
        np.testing.assert_array_equal(lgot[b, :Tb], lwant[0])
        assert not got[b, Tb:].any() and not lgot[b, Tb:].any()
    # padding to the longest utterance instead changes the short ones: padded frames are keys and enter the layer norms
    pad = np.where(np.isnan(mel), 0.0, mel)
    padded, _ = oa.mel_forward(pad[2:3], w, np.float64)
    assert np.abs(padded[0, :3] - got[2, :3]).max() > 1e-6

"""Host-only: the frame and carried-tail rules of any analysis frame, the parametrised references of
tests/_frontend_ref.py (at 400/160 they are the oracle's own functions), the record size rule, and loading a frozen
graph whose mel basis belongs to another fft_size."""
import numpy as np
import pytest

from oracle import model as om
from oracle import streaming as ost
from tests import _frontend_ref as R


@pytest.mark.parametrize("cfg", R.ALL, ids=R.cfg_id)
def test_frame_and_tail_rules_agree(cfg):
    """A stream fed in chunks of any size frames exactly the samples one call on the whole signal frames: the carried
    tail is total - frames * hop samples, never more than fft - 1, and chunked frame counts add up."""
    fft, hop = cfg
    rng = np.random.default_rng(fft + hop)
    for total in range(fft, fft + 3 * hop + 2):
        n = om.num_frames(total, fft, hop)
        keep = ost.residual_length(total, fft, hop)
        assert keep == total - n * hop and 0 <= keep < fft
    for _ in range(20):
        sizes = rng.integers(1, 3 * fft, 12)
        tail, frames = 0, 0
        for c in sizes:
            total = tail + int(c)
            n = max(0, om.num_frames(total, fft, hop))
            frames += n
            tail = ost.residual_length(total, fft, hop) if n else total
            assert tail < max(fft, total + 1)
        assert frames == max(0, om.num_frames(int(sizes.sum()), fft, hop))


@pytest.mark.parametrize("cfg", R.ALL, ids=R.cfg_id)
def test_reference_front_end_is_the_dft(cfg):
    """pcm_to_mel = |x W| basis with the explicit DFT matrix, in float64."""
    fft, hop = cfg
    rng = np.random.default_rng(3)
    x = rng.standard_normal((2, fft + 2 * hop + 5))
    basis = R.mel_basis(fft, 16).astype(np.float64)
    assert basis.shape == (fft // 2 + 1, 16)
    got = R.pcm_to_mel(x, basis, fft, hop, np.float64)
    k = np.arange(fft // 2 + 1)
    W = np.exp(-2j * np.pi * np.outer(np.arange(fft), k) / fft)
    frames = np.stack([x[:, f * hop:f * hop + fft] for f in range(om.num_frames(x.shape[1], fft, hop))], axis=1)
    want = np.abs(frames @ W) @ basis
    np.testing.assert_allclose(got, want, rtol=1e-10, atol=1e-9)


def test_references_at_400_160_are_the_oracle():
    rng = np.random.default_rng(8)
    ow = om.init_weights(seed=5, n_mel=40)
    pcm = om.pcm16_to_float(rng.integers(-3000, 3000, (3, 4321)).astype(np.int16))
    np.testing.assert_array_equal(R.pcm_to_mel(pcm, ow.mel_basis, 400, 160), om.pcm_to_mel(pcm, ow))
    st = np.zeros((2, 3, 128), np.float32)
    for a, b in zip(R.deploy_forward(pcm, st, ow, 400, 160), om.deploy_forward(pcm, st, ow)):
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(R.mel_basis(400, 40), ow.mel_basis)
    ref, orc = R.StreamRef(ow, 3, 400, 160), ost.StreamOracle(ow, 3)
    for n in (4800, 100, 399, 3600):
        blk = rng.integers(-3000, 3000, (3, n)).astype(np.int16)
        a, b = ref.step(blk), orc.step(blk)
        np.testing.assert_array_equal(a["softmax"], b["softmax"])
        np.testing.assert_array_equal(a["trigger"], b["trigger"])
        np.testing.assert_array_equal(ref.res, orc.res)
    x = om.pcm16_to_float(rng.integers(-3000, 3000, 9000).astype(np.int16))
    for a, b in zip(R.stream_vs_offline(x, ow, 400, 160), ost.stream_vs_offline(x, ow)):
        np.testing.assert_array_equal(a, b)


def test_hop_equal_to_fft_carries_no_tail():
    """512/512: a chunk of whole frames leaves nothing behind (the tail is empty, not the whole signal)."""
    ow = R.weights(512, 16)
    ref = R.StreamRef(ow, 2, 512, 512)
    ref.step(np.ones((2, 1024), np.int16))
    assert ref.res.shape == (2, 0)
    ref.step(np.ones((2, 700), np.int16))
    assert ref.res.shape == (2, 188)


def test_record_size_rule():
    """Records keep today's layout for every fft_size <= 400 (2,368 bytes at the default stream configuration); a
    wider frame widens only the tail section, to fft_size rounded up to 8 samples."""
    assert R.record_bytes(400) == 2368
    for fft in (16, 200, 256, 320, 399):
        assert R.tail_capacity(fft) == 400 and R.record_bytes(fft) == 2368
    assert R.tail_capacity(401) == 408 and R.tail_capacity(512) == 512 and R.tail_capacity(500) == 504
    assert R.record_bytes(512) == 2368 + 2 * (512 - 400)


def test_frozen_graph_with_a_257_bin_basis_loads_with_its_fft_size():
    pytest.importorskip("google.protobuf")
    from keyword_spotting_b200 import ModelWeights
    from keyword_spotting_b200.graph_pb import GraphFormatError
    from tests.test_graph_pb import _frozen_graph
    ow = R.weights(512, 40)
    data, _ = _frozen_graph(ow)
    w = ModelWeights.from_frozen_graph(data, fft_size=512)
    np.testing.assert_array_equal(w.mel_basis, ow.mel_basis)
    np.testing.assert_array_equal(w.fc_w, ow.fc_w)
    with pytest.raises(GraphFormatError, match=r"\[201, n_mel\] mel basis Const of fft_size = 400 was not found.*\[257, 40\]"):
        ModelWeights.from_frozen_graph(data)

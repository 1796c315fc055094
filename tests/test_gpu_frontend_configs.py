"""GPU: models trained with other analysis frames (fft_size 16..512, hop_size 1..fft_size) through every layer: model
creation, the general DFT front end (csrc/frontend_dft.cu) against float64 numpy, per-row lengths, the deployment call
at every precision, the streaming detector, per-stream records, the wave server and the attention model's PCM path.
400/160 runs through the same tests as the control (there the FFT front end serves)."""
import numpy as np
import pytest

from tests import _frontend_ref as R
from tests._util import synth_pcm16, to_product_weights

pytestmark = pytest.mark.gpu

TOL_MEL = 2e-5           # of each frame's peak: the bar of the 400-point kernels (DESIGN.md section 4)
TOL_FP32 = 1e-4
TOL_CONTRACT = 1e-3
TOL_QUANTUM = 3e-2       # octbit graph: one or a few flipped u8 codes (tests/test_gpu_octbit_model.py)

_MODELS = {}


def _model(fft, hop, n_mel=40, precision="fp32", gain=1.0, seed=1234):
    key = (fft, hop, n_mel, precision, gain, seed)
    if key not in _MODELS:
        from keyword_spotting_b200 import Config, DeployModel
        ow = R.weights(fft, n_mel, seed, gain)
        cfg = Config(n_mel=n_mel, fft_size=fft, hop_size=hop)
        _MODELS[key] = (ow, DeployModel(cfg, to_product_weights(ow), precision=precision))
    return _MODELS[key]


@pytest.fixture(scope="module", autouse=True)
def _close_models():
    yield
    for _, dm in _MODELS.values():
        dm.close()
    _MODELS.clear()


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _c_frontend(dm, x, L, lengths=None):
    """kws_frontend_mel_lens on the first L samples of the rows of the CUDA tensor x [S, ld]."""
    import torch
    from keyword_spotting_b200 import _lib
    S, ld = x.shape[0], x.stride(0)
    n = dm.num_frames(L)
    mel = torch.full((S, max(n, 0), dm.config.n_mel), 7.0, dtype=torch.float32, device="cuda")
    dt = _lib.PCM_I16 if x.dtype == torch.int16 else _lib.PCM_F32
    _lib.check(_lib.load().kws_frontend_mel_lens(dm.handle, x.data_ptr(), dt, S, L, ld,
                                                 None if lengths is None else lengths.data_ptr(), mel.data_ptr(),
                                                 _stream()))
    torch.cuda.synchronize()
    return mel.cpu().numpy()


def _dev(a, dtype=None):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a))
    return (t if dtype is None else t.to(dtype)).cuda()


# ================================================================ 1. model creation
@pytest.mark.parametrize("cfg", R.ALL, ids=R.cfg_id)
def test_model_accepts_the_frame_and_counts_frames_like_the_oracle(cfg):
    from oracle import model as om
    fft, hop = cfg
    _, dm = _model(fft, hop)
    for L in (0, 1, fft - 1, fft, fft + 1, fft + hop - 1, fft + hop, 4800, 16000, 160000):
        assert dm.num_frames(L) == om.num_frames(L, fft, hop), L


@pytest.mark.parametrize("fft,hop", [(513, 160), (15, 8), (512, 0), (320, 321), (400, -1)])
def test_model_rejects_frames_outside_the_range(fft, hop):
    from keyword_spotting_b200 import Config, DeployModel, InvalidArgumentError
    ow = R.weights(fft, 40)
    with pytest.raises(InvalidArgumentError, match=r"fft_size must be in \[16, 512\] and hop_size in \[1, fft_size\]"):
        DeployModel(Config(n_mel=40, fft_size=fft, hop_size=hop), to_product_weights(ow), precision="fp32")


# ================================================================ 2. kws_frontend_mel vs float64
def _signals(rng, S, L, kind):
    if kind == "full":
        return rng.integers(-32768, 32768, (S, L)).astype(np.int16)
    return rng.integers(-1, 2, (S, L)).astype(np.int16)            # 1 LSB: only the lo half of the split is non-zero


@pytest.mark.parametrize("n_mel", [16, 40, 60, 80, 128])
@pytest.mark.parametrize("cfg", R.ALL, ids=R.cfg_id)
def test_frontend_mel_matches_float64_numpy(cfg, n_mel):
    fft, hop = cfg
    ow, dm = _model(fft, hop, n_mel)
    rng = np.random.default_rng(fft * 1000 + hop + n_mel)
    for L in (fft - 1, fft, fft + hop - 1, 160000):
        S = 3 if L < 160000 else 2
        for kind in ("full", "lsb"):
            x16 = _signals(rng, S, L, kind)
            xf = (x16.astype(np.float32) / np.float32(32768.0))
            want = R.pcm_to_mel(xf.astype(np.float64), ow.mel_basis.astype(np.float64), fft, hop, np.float64)
            for x in (x16, xf):
                got = _c_frontend(dm, _dev(x), L)
                assert got.shape == want.shape, (L, got.shape, want.shape)
                if want.size == 0:
                    continue
                peak = np.abs(want).max(axis=-1, keepdims=True)
                err = np.abs(got - want)
                assert (err <= TOL_MEL * peak + 1e-12).all(), (L, kind, x.dtype, float((err / np.maximum(peak, 1e-30)).max()))


# ================================================================ 3. rows of their own lengths
@pytest.mark.parametrize("dtype", [np.int16, np.float32], ids=["int16", "float32"])
@pytest.mark.parametrize("cfg", R.ALL, ids=R.cfg_id)
def test_rows_of_their_own_lengths_equal_each_row_alone(cfg, dtype):
    """Every row bit for bit as the row alone; rows past n_b zero; samples past a row's length (loud garbage, NaN)
    reach no output -- in kws_frontend_mel_lens and kws_deploy_forward_lens."""
    import torch
    from oracle import model as om
    fft, hop = cfg
    _, dm = _model(fft, hop)
    rng = np.random.default_rng(7 + fft + hop)
    L = max(12000, 129 * hop + fft)                 # the 129-frame row spans two front-end tiles
    lens = np.array([0, fft - 1, fft, fft + hop - 1, fft + hop, 3, 5003, 7777, 128 * hop + fft, L - 1, L], np.int64)
    pcm16 = synth_pcm16(rng, len(lens), L, silent_frac=0.1)
    x = pcm16.copy() if dtype == np.int16 else pcm16.astype(np.float32) / np.float32(32768.0)
    for b, n in enumerate(lens):
        x[b, n:] = rng.integers(-32768, 32768, L - n) if dtype == np.int16 else np.nan
    got = _c_frontend(dm, _dev(x), L, _dev(lens, torch.int32))
    probs, state = dm.forward(x, np.zeros((2, len(lens), 128), np.float32), lengths=lens)
    for b, n in enumerate(lens):
        nb = max(0, om.num_frames(int(n), fft, hop))
        assert (got[b, nb:] == 0).all(), b
        assert (probs[b, nb:] == 0).all(), b
        if nb == 0:
            continue
        alone = _c_frontend(dm, _dev(x[b:b + 1, :n]), int(n))
        np.testing.assert_array_equal(got[b, :nb], alone[0], err_msg="row %d" % b)
        p1, s1 = dm.forward(x[b:b + 1, :n], np.zeros((2, 1, 128), np.float32))
        np.testing.assert_array_equal(probs[b, :nb], p1[0], err_msg="row %d" % b)
        np.testing.assert_array_equal(state[:, b], s1[:, 0], err_msg="row %d" % b)
    assert np.isfinite(got).all() and np.isfinite(probs).all()


# ================================================================ 4. the deployment call at every precision
@pytest.mark.parametrize("precision", ["fp32", "tc", "octbit"])
@pytest.mark.parametrize("cfg", R.ALL, ids=R.cfg_id)
def test_deploy_forward_matches_the_oracle(cfg, precision):
    from keyword_spotting_b200 import OctbitModelWeights
    from oracle import model as om
    fft, hop = cfg
    ow, dm = _model(fft, hop, precision="fp32" if precision == "fp32" else "tc", seed=4321)
    rng = np.random.default_rng(31 + fft)
    S, L = 6, 8000
    pcm = om.pcm16_to_float(synth_pcm16(rng, S, L, silent_frac=0.2))
    st = (rng.uniform(-1, 1, (2, S, 128)) * 0.5).astype(np.float32)
    if precision == "octbit":
        octw = om.octize_model(ow)
        dm.set_octbit(OctbitModelWeights.from_float(dm.weights))
        try:
            p_got, s_got = dm.forward(pcm, st)
        finally:
            dm.set_octbit(None)
        mel = R.pcm_to_mel(pcm, ow.mel_basis, fft, hop)
        p_want, s_want, _ = om.octbit_mel_forward(mel, st, ow, octw)
        assert np.abs(p_got - p_want).max() < TOL_QUANTUM and np.abs(s_got - s_want).max() < TOL_QUANTUM
        return
    p_want, s_want, _ = R.deploy_forward(pcm, st, ow, fft, hop)
    p_got, s_got = dm.forward(pcm, st)
    assert p_got.shape == p_want.shape
    tol = TOL_FP32 if precision == "fp32" else TOL_CONTRACT
    assert np.abs(p_got - p_want).max() < tol and np.abs(s_got - s_want).max() < tol


# ================================================================ 5. the streaming detector
def _chunk_lengths(fft, hop):
    """Below one frame, exactly one frame, odd sizes, the usual 4800 and a chunk of more than 128 frames (one front-end
    tile) per stream; max_chunk keeps a chunk under 255 frames."""
    big = min(16000, 254 * hop)
    return [4800, 37, fft - 1, 1, fft, 3600, 2 * hop + 1, big, 4800, 999, 4800, 4801, 2000, 4800]


@pytest.mark.parametrize("cfg", R.ALL, ids=R.cfg_id)
def test_streaming_detector_matches_the_detector_loop(cfg):
    from keyword_spotting_b200 import StreamingDetector
    fft, hop = cfg
    ow, dm = _model(fft, hop, gain=6.0)
    sizes = _chunk_lengths(fft, hop)
    S = 40
    rng = np.random.default_rng(5 + fft + hop)
    det = StreamingDetector(dm, S, max_chunk=max(sizes), keyword="1")
    ref = R.StreamRef(ow, S, fft, hop, label="1")
    n_trig = n_sil = 0
    for c, n in enumerate(sizes):
        blk = synth_pcm16(rng, S, n, silent_frac=0.0)
        quiet = rng.random(S) < 0.3
        blk[quiet] = rng.integers(-2, 3, (int(quiet.sum()), n))
        want = ref.step(blk)
        trig, probs, nfr = det.step(blk, want_probs=True)
        nf = want["softmax"].shape[1]
        assert (nfr == nf).all(), (c, n, nfr[:4], nf)
        if nf:
            assert np.abs(probs[:, :nf] - want["softmax"]).max() < TOL_FP32, c
        np.testing.assert_array_equal(trig, want["trigger"], err_msg="chunk %d" % c)
        assert np.abs(det.state().cpu().numpy() - want["state"]).max() < TOL_FP32, c
        labels, counts = det.window_labels()
        for s in range(S):
            if not want["trigger"][s]:
                np.testing.assert_array_equal(labels[s, :counts[s]], want["labels"][s])
        n_trig += int(trig.sum())
        n_sil += int((~want["speech"]).sum())
    assert n_trig > 0 and n_sil > 20, (n_trig, n_sil)
    det.close()


def test_stream_vs_offline_at_512_160():
    """The reference's self-check (detector.py:254-289) with the product: one utterance fed in 3600-sample pieces with
    carried tail and state gives the whole-utterance softmax."""
    from oracle import model as om
    from oracle import streaming as ost
    fft, hop = 512, 160
    ow, dm = _model(fft, hop)
    rng = np.random.default_rng(77)
    pcm = om.pcm16_to_float(synth_pcm16(rng, 1, 30000, silent_frac=0.0))[0]
    want, st_want = R.stream_vs_offline(pcm, ow, fft, hop)
    whole, st_whole = dm.forward(pcm[None, :len(pcm) - (len(pcm) - fft) % hop], np.zeros((2, 1, 128), np.float32))
    state, res, outs = np.zeros((2, 1, 128), np.float32), np.zeros(0, np.float32), []
    for i in range(len(pcm) // 3600 + 1):
        data = np.concatenate([res, pcm[i * 3600:(i + 1) * 3600]])
        if len(data) < fft:
            res = data
            continue
        res = data[len(data) - ost.residual_length(len(data), fft, hop):]
        sm, state = dm.forward(data[None, :len(data) - (len(data) - fft) % hop], state)
        outs.append(sm[0])
    streamed = np.concatenate(outs, axis=0)
    assert streamed.shape == want.shape == whole[0].shape
    assert np.abs(streamed - want).max() < TOL_FP32 and np.abs(streamed - whole[0]).max() < TOL_FP32
    assert np.abs(state - st_want).max() < TOL_FP32


# ================================================================ 6. per-stream records
@pytest.mark.parametrize("cfg", [(512, 160), (320, 160)], ids=R.cfg_id)
def test_records_round_trip_and_moved_streams_continue(cfg):
    import torch
    from keyword_spotting_b200 import InvalidArgumentError, StreamingDetector
    fft, hop = cfg
    _, dm = _model(fft, hop, gain=6.0)
    rng = np.random.default_rng(3)
    A = StreamingDetector(dm, 200, keyword="1")
    B = StreamingDetector(dm, 90, keyword="1")
    assert A.record_bytes == R.record_bytes(fft)
    for n in (4800, 4000, 3601):
        A.step(synth_pcm16(rng, 200, n, silent_frac=0.2))
        B.step(synth_pcm16(rng, 90, n, silent_frac=0.2))
    ids = rng.permutation(200)[:60].astype(np.int64)
    slots = rng.permutation(90)[:60].astype(np.int64)
    rec = A.export_streams(ids)
    B.import_streams(slots, rec)
    np.testing.assert_array_equal(B.export_streams(slots).cpu().numpy(), rec.cpu().numpy())
    for c, n in enumerate((4800, 3333, 4800)):
        pa = synth_pcm16(rng, 200, n, silent_frac=0.2)
        pb = synth_pcm16(rng, 90, n, silent_frac=0.2)
        pb[slots] = pa[ids]
        ta, pra, na = A.step(pa, want_probs=True)
        tb, prb, nb = B.step(pb, want_probs=True)
        np.testing.assert_array_equal(tb[slots], ta[ids])
        np.testing.assert_array_equal(nb[slots], na[ids])
        np.testing.assert_array_equal(prb[slots], pra[ids])
        assert torch.equal(B.state()[:, torch.as_tensor(slots)], A.state()[:, torch.as_tensor(ids)]), c
    # a record of the default frame has another tail capacity: header mismatch (status 2)
    _, d400 = _model(400, 160, gain=6.0)
    C = StreamingDetector(d400, 4, keyword="1")
    C.step(synth_pcm16(rng, 4, 4800, silent_frac=0.0))
    other = C.export_streams([0, 1])
    if fft > 400:
        assert C.record_bytes != A.record_bytes
        with pytest.raises(InvalidArgumentError):
            A.import_streams([0, 1], other.new_zeros((2, A.record_bytes)))
        cut = torch.zeros((2, A.record_bytes), dtype=torch.uint8, device=other.device)
        cut[:, :C.record_bytes] = other
        with pytest.raises(InvalidArgumentError, match="header does not match"):
            A.import_streams([0, 1], cut)
    # tail_len = fft_size is malformed (status 3); fft_size - 1 is the longest tail a stream carries
    good = A.export_streams([5])
    bad = good.clone()
    bad[0, 32:36] = torch.tensor(np.frombuffer(np.int32(fft).tobytes(), np.uint8).copy(), device=bad.device)
    before = A.export_streams([7])
    with pytest.raises(InvalidArgumentError, match="malformed field"):
        A.import_streams([7], bad)
    np.testing.assert_array_equal(A.export_streams([7]).cpu().numpy(), before.cpu().numpy())
    C.close()
    A.close()
    B.close()


# ================================================================ 7. the wave server
@pytest.mark.parametrize("use_graphs", [True, False], ids=["graphs", "direct"])
def test_wave_server_at_512_160_matches_one_stream_object(use_graphs):
    import torch
    from keyword_spotting_b200 import StreamingDetector, WaveServer
    _, dm = _model(512, 160, precision="tc", gain=3.0, seed=21)
    W, Sw, chunks, n = 4, 96, 6, 4800
    S = W * Sw
    rng = np.random.default_rng(77)
    big = StreamingDetector(dm, S, keyword="1")
    srv = WaveServer(dm, S, waves=W, use_graphs=use_graphs, keyword="1")
    n_trig = 0
    for c in range(chunks):
        blk = synth_pcm16(rng, S, n, silent_frac=0.2)
        want = big.step(blk)
        got = srv.step(blk)
        np.testing.assert_array_equal(got, want, err_msg="chunk %d" % c)
        assert torch.equal(srv.state(), big.state()), c
        n_trig += int(want.sum())
    assert n_trig > 0
    srv.close()
    big.close()


# ================================================================ 8. the attention model's PCM path
def test_attention_forward_from_pcm_at_512_160():
    from keyword_spotting_b200 import AttentionConfig, AttentionDeployModel, AttentionWeights
    from oracle import attention as oa
    from oracle import model as om
    fft, hop = 512, 160
    ow = oa.init_weights(seed=4321, n_mel=60)
    ow.mel_basis = R.mel_basis(fft, 60)
    m = AttentionDeployModel(AttentionConfig(fft_size=fft, hop_size=hop), AttentionWeights.from_object(ow))
    rng = np.random.default_rng(9)
    pcm = om.pcm16_to_float(synth_pcm16(rng, 3, 16000, silent_frac=0.0))
    mel = R.pcm_to_mel(pcm, ow.mel_basis, fft, hop)
    want, _ = oa.mel_forward(mel, ow, np.float32)
    got = m.forward(pcm)
    got = got.cpu().numpy() if hasattr(got, "cpu") else np.asarray(got)
    assert got.shape == want.shape
    assert np.abs(got - want).max() < TOL_CONTRACT, np.abs(got - want).max()
    m.close()

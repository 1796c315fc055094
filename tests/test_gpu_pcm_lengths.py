"""GPU: the rnn_ctc front end and deployment call on batches of PCM rows of different lengths
(kws_frontend_mel_lens, kws_deploy_forward_lens, DeployModel.frontend / forward(lengths=)), and the attention model's
forward(lengths=) that now goes through the same front end.

Every row of a padded batch must come out exactly as a call on that row alone computes it, bit for bit, with zero rows
past its n_b frames; samples past its length (loud garbage for int16, NaN for float32) must never reach an output.
"""
import numpy as np
import pytest

from tests._util import make_config, synth_pcm16, to_product_weights

pytestmark = pytest.mark.gpu

FFT, HOP = 400, 160


def _n_frames(n):
    return max(0, 1 + (int(n) - FFT) // HOP)


def _lengths(L):
    """0, below / at / above one frame, the frame boundaries 559 / 560, odd n_b (the last valid frame's FFT partner
    lies past the end) and even n_b, n_b 30 / 31 (tensor-core front-end items) and 32 / 33 (FFT front-end items), odd
    lengths, lengths that are not multiples of 4 or 8, and the longest row equal to L."""
    lens = [0, 399, 400, 401, 559, 560, 880, 1041, 5040, 5201, 5360, 5521, 3, 7777, 1602, L - 1, L]
    assert _n_frames(401) % 2 == 1 and _n_frames(880) % 2 == 0
    assert [_n_frames(n) for n in (5040, 5201, 5360, 5521)] == [30, 31, 32, 33]
    return np.array(lens, np.int64)


def _pcm_batch(rng, lens, L, dtype, ld=None):
    """[S, ld] rows: real signal below each length, loud garbage (int16) or NaN (float32) from there on."""
    ld = ld or L
    pcm16 = synth_pcm16(rng, len(lens), ld, silent_frac=0.1)
    if dtype == np.int16:
        x = pcm16.copy()
        for b, n in enumerate(lens):
            x[b, n:] = rng.integers(-32768, 32768, ld - n)
        return x
    x = pcm16.astype(np.float32) / np.float32(32768.0)
    for b, n in enumerate(lens):
        x[b, n:] = np.nan
    return x


_MODELS = {}


def _model(precision="tc", frontend="fft", octbit=False):
    key = (precision, frontend, octbit)
    if key not in _MODELS:
        from keyword_spotting_b200 import DeployModel, OctbitModelWeights
        from oracle import model as om
        ow = om.init_weights(seed=1234, n_mel=40)
        dm = DeployModel(make_config(40), to_product_weights(ow), precision=precision, frontend=frontend)
        if octbit:
            dm.set_octbit(OctbitModelWeights.from_float(dm.weights))
        _MODELS[key] = (ow, dm)
    return _MODELS[key]


@pytest.fixture(scope="module", autouse=True)
def _close_models():
    yield
    for _, dm in _MODELS.values():
        dm.close()
    _MODELS.clear()


def _dev(a, dtype=None):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a))
    return (t if dtype is None else t.to(dtype)).cuda()


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _c_frontend(dm, x, L, lengths=None, legacy=False):
    """kws_frontend_mel(_lens) on the first L samples of the rows of the CUDA tensor x [S, ld]."""
    import torch
    from keyword_spotting_b200 import _lib
    lib = _lib.load()
    S, ld = x.shape[0], x.stride(0)
    n = dm.num_frames(L)
    mel = torch.full((S, n, dm.config.n_mel), 7.0, dtype=torch.float32, device="cuda")   # stale values must go
    dt = _lib.PCM_I16 if x.dtype == torch.int16 else _lib.PCM_F32
    if legacy:
        rc = lib.kws_frontend_mel(dm.handle, x.data_ptr(), dt, S, L, ld, mel.data_ptr(), _stream())
    else:
        rc = lib.kws_frontend_mel_lens(dm.handle, x.data_ptr(), dt, S, L, ld, None if lengths is None else lengths.data_ptr(),
                                       mel.data_ptr(), _stream())
    _lib.check(rc)
    torch.cuda.synchronize()
    return mel.cpu().numpy()


def _c_deploy(dm, x, L, state, lengths=None, legacy=False):
    import torch
    from keyword_spotting_b200 import _lib
    lib = _lib.load()
    S, ld = x.shape[0], x.stride(0)
    n, C = dm.num_frames(L), dm.config.num_classes
    probs = torch.full((S, n, C), 7.0, dtype=torch.float32, device="cuda")
    logits = torch.full((S, n, C), 7.0, dtype=torch.float32, device="cuda")
    st_out = torch.empty_like(state)
    dt = _lib.PCM_I16 if x.dtype == torch.int16 else _lib.PCM_F32
    if legacy:
        rc = lib.kws_deploy_forward(dm.handle, x.data_ptr(), dt, S, L, ld, state.data_ptr(), probs.data_ptr(),
                                    st_out.data_ptr(), logits.data_ptr(), _stream())
    else:
        rc = lib.kws_deploy_forward_lens(dm.handle, x.data_ptr(), dt, S, L, ld, None if lengths is None else lengths.data_ptr(),
                                         state.data_ptr(), probs.data_ptr(), st_out.data_ptr(), logits.data_ptr(), _stream())
    _lib.check(rc)
    torch.cuda.synchronize()
    return probs.cpu().numpy(), st_out.cpu().numpy(), logits.cpu().numpy()


# ================================================================ kws_frontend_mel_lens
FRONTEND_CASES = [("fft", np.int16, 10240), ("fft", np.float32, 10240), ("tc", np.int16, 10240),
                  ("fft", np.int16, 10243), ("fft", np.float32, 10243), ("tc", np.int16, 10243)]


@pytest.mark.parametrize("frontend,dtype,ld", FRONTEND_CASES, ids=lambda v: getattr(v, "__name__", str(v)))
def test_frontend_rows_equal_each_row_alone(frontend, dtype, ld):
    """Each row bit for bit as kws_frontend_mel on the row alone; rows past n_b exactly zero.  ld = 10243: odd row
    stride (element-wise int16 staging); ld = 10240: aligned rows whose lengths cut through vector loads."""
    import torch
    _, dm = _model("tc", frontend)
    rng = np.random.default_rng(11 + ld)
    L = 10240
    lens = _lengths(L)
    x = _pcm_batch(rng, lens, L, dtype, ld=ld)
    got = _c_frontend(dm, _dev(x), L, _dev(lens, torch.int32))
    n = dm.num_frames(L)
    assert got.shape == (len(lens), n, 40)
    for b, ln in enumerate(lens):
        nb = _n_frames(ln)
        if nb:
            alone = _c_frontend(dm, _dev(x[b:b + 1, :ln]), int(ln))
            assert alone.shape[1] == nb
            assert np.array_equal(got[b, :nb], alone[0]), (b, int(ln), float(np.abs(got[b, :nb] - alone[0]).max()))
        assert not got[b, nb:].any(), (b, int(ln))
        assert np.isfinite(got[b]).all()


@pytest.mark.parametrize("frontend,dtype", [("fft", np.int16), ("fft", np.float32), ("tc", np.int16)])
def test_frontend_null_and_full_lengths_equal_kws_frontend_mel(frontend, dtype):
    import torch
    _, dm = _model("tc", frontend)
    rng = np.random.default_rng(12)
    S, L = 37, 9601
    x = _dev(_pcm_batch(rng, [L] * S, L, dtype))
    want = _c_frontend(dm, x, L, legacy=True)
    np.testing.assert_array_equal(_c_frontend(dm, x, L, None), want)
    np.testing.assert_array_equal(_c_frontend(dm, x, L, torch.full((S,), L, dtype=torch.int32, device="cuda")), want)


def test_frontend_device_lengths_are_clamped():
    import torch
    _, dm = _model("tc", "fft")
    rng = np.random.default_rng(13)
    L = 4000
    raw = np.array([-7, -1 << 30, 0, L + 1, 1 << 30, 2000, L], np.int64)
    clamped = np.clip(raw, 0, L)
    x = _dev(_pcm_batch(rng, clamped, L, np.int16))
    got = _c_frontend(dm, x, L, _dev(raw, torch.int32))
    want = _c_frontend(dm, x, L, _dev(clamped, torch.int32))
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(got[3], _c_frontend(dm, x[3:4], L, legacy=True)[0])
    assert not got[:3].any()


# ================================================================ kws_deploy_forward_lens
DEPLOY_CASES = [("tc", "fft", False, np.int16), ("tc", "fft", False, np.float32), ("tc", "tc", False, np.int16),
                ("fp32", "fft", False, np.int16), ("fp32", "fft", False, np.float32), ("fp32", "tc", False, np.int16),
                ("fp32", "fft", True, np.int16), ("fp32", "fft", True, np.float32)]


def _check_deploy_rows(dm, ow, x, lens, L, st, oracle_tol=None):
    """x: host [S, ld >= L] rows; the batch call reads the first L samples of each row with row stride ld."""
    import torch
    probs, s_out, logits = _c_deploy(dm, _dev(x)[:, :L], L, _dev(st), _dev(lens, torch.int32))
    worst = 0.0
    for b, ln in enumerate(lens):
        nb = _n_frames(ln)
        if ln >= FFT:
            pa, sa, la = _c_deploy(dm, _dev(x[b:b + 1, :ln]), int(ln), _dev(st[:, b:b + 1]))
            assert pa.shape[1] == nb
            assert np.array_equal(probs[b, :nb], pa[0]), (b, int(ln), float(np.abs(probs[b, :nb] - pa[0]).max()))
            assert np.array_equal(logits[b, :nb], la[0]), (b, int(ln))
            assert np.array_equal(s_out[:, b], sa[:, 0]), (b, int(ln), float(np.abs(s_out[:, b] - sa[:, 0]).max()))
            if oracle_tol is not None:
                from oracle import model as om
                xb = x[b:b + 1, :ln]
                xf = om.pcm16_to_float(xb) if xb.dtype == np.int16 else xb
                pw, sw, _ = om.deploy_forward(xf, st[:, b:b + 1], ow)
                worst = max(worst, float(np.abs(pa - pw).max()), float(np.abs(sa - sw).max()))
        if nb == 0:
            np.testing.assert_array_equal(s_out[:, b], st[:, b])       # length-0 rule: the state passes through
        assert not probs[b, nb:].any() and not logits[b, nb:].any(), (b, int(ln))
        assert np.isfinite(probs[b]).all() and np.isfinite(s_out[:, b]).all()
    if oracle_tol is not None:
        assert worst < oracle_tol, worst
    return worst


@pytest.mark.parametrize("precision,frontend,octbit,dtype", DEPLOY_CASES,
                         ids=lambda v: getattr(v, "__name__", str(v)))
def test_deploy_rows_equal_each_row_alone(precision, frontend, octbit, dtype):
    """probs, logits and state_out of each row bit for bit as kws_deploy_forward on the row alone, with a nonzero
    incoming state; rows past n_b zero; n_b = 0 passes the state through; the float graphs against the CPU oracle."""
    ow, dm = _model(precision, frontend, octbit)
    rng = np.random.default_rng(21)
    L = 10240
    lens = _lengths(L)
    x = _pcm_batch(rng, lens, L, dtype)
    st = (rng.uniform(-1, 1, (2, len(lens), 128)) * 0.7).astype(np.float32)
    tol = None if octbit else (1e-3 if precision == "tc" else 1e-4)
    worst = _check_deploy_rows(dm, ow, x, lens, L, st, oracle_tol=tol)
    print("%s/%s%s: worst |row - oracle| %.3g" % (precision, frontend, "/octbit" if octbit else "", worst))


@pytest.mark.parametrize("precision,frontend", [("tc", "fft"), ("tc", "tc")])
def test_deploy_small_batch_pipelined_layers(precision, frontend):
    """A small batch of long rows takes the two-stream layer pipeline of the tensor-core recurrence (n >= 128 frames,
    under 32,768 utterances); rows alone of fewer than 128 frames do not.  Odd row stride on top."""
    ow, dm = _model(precision, frontend)
    rng = np.random.default_rng(22)
    L = 24000
    assert dm.num_frames(L) >= 128
    lens = np.array([L, 401, 20721, 5521, 0, 12345, 23999, 5040], np.int64)
    x = _pcm_batch(rng, lens, L, np.int16, ld=L + 1)
    st = (rng.uniform(-1, 1, (2, len(lens), 128)) * 0.5).astype(np.float32)
    _check_deploy_rows(dm, ow, x, lens, L, st)


@pytest.mark.parametrize("precision,octbit", [("tc", False), ("fp32", False), ("fp32", True)])
def test_deploy_batch_not_a_multiple_of_128(precision, octbit):
    ow, dm = _model(precision, "fft", octbit)
    rng = np.random.default_rng(23)
    L, S = 4000, 130
    lens = rng.integers(0, L + 1, S)
    lens[:4] = [L, 0, 400, 401]
    x = _pcm_batch(rng, lens, L, np.int16)
    st = (rng.uniform(-1, 1, (2, S, 128)) * 0.5).astype(np.float32)
    _check_deploy_rows(dm, ow, x, lens, L, st)


@pytest.mark.parametrize("precision,frontend,octbit", [("tc", "fft", False), ("tc", "tc", False), ("fp32", "fft", True)])
def test_deploy_null_and_full_lengths_equal_kws_deploy_forward(precision, frontend, octbit):
    import torch
    _, dm = _model(precision, frontend, octbit)
    rng = np.random.default_rng(24)
    S, L = 70, 8000
    x = _dev(_pcm_batch(rng, [L] * S, L, np.int16))
    st = _dev((rng.uniform(-1, 1, (2, S, 128)) * 0.5).astype(np.float32))
    want = _c_deploy(dm, x, L, st, legacy=True)
    for lengths in (None, torch.full((S,), L, dtype=torch.int32, device="cuda")):
        got = _c_deploy(dm, x, L, st, lengths)
        for g, w in zip(got, want):
            np.testing.assert_array_equal(g, w)


def test_deploy_device_lengths_are_clamped():
    import torch
    _, dm = _model("tc", "fft")
    rng = np.random.default_rng(25)
    L = 3000
    raw = np.array([-3, L + 5, 1 << 30, 1234, -(1 << 30)], np.int64)
    clamped = np.clip(raw, 0, L)
    x = _dev(_pcm_batch(rng, clamped, L, np.int16))
    st = _dev((rng.uniform(-1, 1, (2, len(raw), 128)) * 0.5).astype(np.float32))
    got = _c_deploy(dm, x, L, st, _dev(raw, torch.int32))
    want = _c_deploy(dm, x, L, st, _dev(clamped, torch.int32))
    for g, w in zip(got, want):
        np.testing.assert_array_equal(g, w)


# ================================================================ Python
def test_python_forward_and_frontend_with_host_and_cuda_lengths():
    import torch
    _, dm = _model("tc", "fft")
    rng = np.random.default_rng(31)
    L = 6000
    lens = np.array([6000, 0, 401, 559, 4321], np.int64)
    x = _pcm_batch(rng, lens, L, np.int16)
    st = (rng.uniform(-1, 1, (2, len(lens), 128)) * 0.5).astype(np.float32)
    p_h, s_h, l_h = dm.forward(x, st, want_logits=True, lengths=lens)
    assert isinstance(p_h, np.ndarray) and p_h.shape == (5, dm.num_frames(L), 6)
    p_d, s_d, l_d = dm.forward(_dev(x), _dev(st), want_logits=True, lengths=_dev(lens))       # int64 CUDA lengths
    assert isinstance(p_d, torch.Tensor) and p_d.is_cuda
    for a, b in ((p_h, p_d), (s_h, s_d), (l_h, l_d)):
        np.testing.assert_array_equal(a, b.cpu().numpy())
    want = _c_deploy(dm, _dev(x), L, _dev(st), _dev(lens, torch.int32))
    for a, b in zip((p_h, s_h, l_h), want):
        np.testing.assert_array_equal(a, b)
    mel_h = dm.frontend(x, lengths=list(lens))
    mel_d = dm.frontend(_dev(x), lengths=_dev(lens, torch.int32))
    np.testing.assert_array_equal(mel_h, mel_d.cpu().numpy())
    np.testing.assert_array_equal(mel_h, _c_frontend(dm, _dev(x), L, _dev(lens, torch.int32)))
    for b, ln in enumerate(lens):
        nb = _n_frames(ln)
        if nb:
            np.testing.assert_array_equal(mel_h[b, :nb], dm.frontend(x[b, :ln])[0])
            p1, s1 = dm.forward(x[b, :ln], st[:, b:b + 1], lengths=None)
            np.testing.assert_array_equal(p_h[b, :nb], p1[0])
            np.testing.assert_array_equal(s_h[:, b], s1[:, 0])
        assert not mel_h[b, nb:].any() and not p_h[b, nb:].any()


def test_python_frame_counts_keep_the_container_type():
    import torch
    _, dm = _model("tc", "fft")
    lens = [0, 399, 400, 559, 560, 16000]
    want = [dm.num_frames(n) if n >= FFT else 0 for n in lens]
    assert dm.frame_counts(lens) == want and isinstance(dm.frame_counts(lens), list)
    assert dm.frame_counts(tuple(lens)) == tuple(want)
    assert dm.frame_counts(560) == 2 and dm.frame_counts(np.int64(399)) == 0
    a = dm.frame_counts(np.array(lens))
    assert isinstance(a, np.ndarray) and a.tolist() == want
    t = dm.frame_counts(torch.tensor(lens, dtype=torch.int32, device="cuda"))
    assert isinstance(t, torch.Tensor) and t.is_cuda and t.cpu().tolist() == want


def test_python_bad_lengths_raise():
    import torch
    from keyword_spotting_b200 import InvalidArgumentError
    _, dm = _model("tc", "fft")
    x = np.zeros((3, 1000), np.int16)
    st = np.zeros((2, 3, 128), np.float32)
    bad = ([400, 500], [-1, 400, 500], [400, 1001, 500], [400.0, 500.0, 600.0], np.zeros((3, 1), np.int32),
           torch.tensor([400, 500, 600], dtype=torch.float32, device="cuda"),
           torch.tensor([400, 500], dtype=torch.int32, device="cuda"),
           torch.tensor([True, False, True], device="cuda"))
    for b in bad:
        with pytest.raises(InvalidArgumentError):
            dm.forward(x, st, lengths=b)
        with pytest.raises(InvalidArgumentError):
            dm.frontend(x, lengths=b)


# ================================================================ attention_ctc from PCM
def test_attention_pcm_lengths_bit_for_bit():
    """forward(pcm, lengths=) row by row against forward(pcm[b, :L_b]), now bit for bit (host and CUDA lengths)."""
    import torch
    from keyword_spotting_b200 import AttentionDeployModel
    from tests._util import synth_pcm16
    m = AttentionDeployModel()
    try:
        rng = np.random.default_rng(5)
        L = 16000
        lengths = np.array([400, 401, 559, 560, 7999, 12345, L])
        pcm = synth_pcm16(rng, len(lengths), L).astype(np.float32) / 32768.0
        for b, n in enumerate(lengths):
            pcm[b, n:] = rng.standard_normal(L - n) * 3.0          # loud garbage past the end
        got = m.forward(pcm, lengths=lengths)
        got_d = m.forward(_dev(pcm), lengths=_dev(lengths, torch.int32)).cpu().numpy()
        np.testing.assert_array_equal(got, got_d)
        for b, n in enumerate(lengths):
            alone = m.forward(pcm[b, :n])
            Tb = alone.shape[1]
            assert Tb == m.output_lengths(m.frame_counts(int(n)))
            assert np.array_equal(got[b, :Tb], alone[0]), (b, int(n), float(np.abs(got[b, :Tb] - alone[0]).max()))
            assert not got[b, Tb:].any()
    finally:
        m.close()


# ================================================================ evaluation.validate(sample_lengths=True)
def _pcm_batches(rng, n_batches, B, L):
    out = []
    for _ in range(n_batches):
        lens = rng.integers(FFT, L + 1, B)
        lens[0] = L
        x = _pcm_batch(rng, lens, L, np.int16)
        out.append((x, lens, rng.integers(0, 2, B)))
    return out


def test_validate_sample_lengths_rnn_ctc():
    from keyword_spotting_b200 import evaluation
    _, dm = _model("tc", "fft")
    rng = np.random.default_rng(41)
    batches = _pcm_batches(rng, 3, 8, 8000)
    want = dict(miss=0, target=0, false_accept=0, total=0)
    for x, lens, corr in batches:
        for b in range(len(lens)):
            sm, _ = dm(x[b:b + 1, :lens[b]], dm.zero_state(1))
            mi, t, fa, _ = evaluation.evaluate_softmax(sm, corr[b:b + 1], label_seqs=dm.config.label_seqs)
            want["miss"] += mi
            want["target"] += t
            want["false_accept"] += fa
            want["total"] += 1
    assert dict(evaluation.validate(dm, batches, sample_lengths=True)) == want


def test_validate_sample_lengths_attention():
    from keyword_spotting_b200 import AttentionDeployModel, evaluation
    m = AttentionDeployModel()
    try:
        rng = np.random.default_rng(42)
        batches = _pcm_batches(rng, 3, 8, 8000)
        want = dict(miss=0, target=0, false_accept=0, total=0)
        for x, lens, corr in batches:
            for b in range(len(lens)):
                sm = m(x[b:b + 1, :lens[b]])
                mi, t, fa, _ = evaluation.evaluate_softmax(sm, corr[b:b + 1], label_seqs=m.config.label_seqs)
                want["miss"] += mi
                want["target"] += t
                want["false_accept"] += fa
                want["total"] += 1
        assert dict(evaluation.validate(m, batches, sample_lengths=True)) == want
    finally:
        m.close()

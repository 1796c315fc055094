"""GPU: attention_ctc on batches of utterances of different lengths (kws_attention_forward_lens, run_mel(lens=),
forward(lengths=)).

Every utterance of a variable-length batch must come out exactly as a call on that utterance alone computes it, bit
for bit, with zero rows past its T'_b; mel frames past its length (NaN here) must never reach an output.
"""

import numpy as np
import pytest

from tests._attention_lens import mel_forward_lens

pytestmark = pytest.mark.gpu

HEAD = 16
TC, FFMA = 0, 1


def _lib():
    from keyword_spotting_b200 import _lib as lib_mod
    return lib_mod, lib_mod.load()


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _model(*args, **kw):
    from tests.test_gpu_attention_kernels import _model as make
    return make(*args, **kw)


def _frames(T, combine):
    return T // combine + 1 if combine > 1 else T


def _lens_for(combine):
    """Mel frame counts whose T'_b hit the edges: 1 and 2 frames, odd and even counts (the fold's zero tail), 16 / 17
    keys (a key group), 128 / 129 and 256 / 257 queries (query tiles), 400 (the tcgen05 maximum), 401 and 501 (the
    FFMA core), mixed with short ones; the longest is T itself."""
    def t_for(tp, r=0):                     # a frame count with T' = tp
        return tp if combine == 1 else (tp - 1) * combine + r
    lens = [1, 2, 3, 4, t_for(16), t_for(17, combine - 1), t_for(128, 1 % combine), t_for(129), t_for(256),
            t_for(257, combine - 1), t_for(400), 5, t_for(401, 1 % combine), 9, t_for(501), t_for(40)]
    return [max(1, n) for n in lens]


def _mel_batch(rng, lens, n_mel, T=None):
    T = T or max(lens)
    mel = (np.abs(rng.standard_normal((len(lens), T, n_mel))) * rng.uniform(0.2, 3.0)).astype(np.float32)
    for b, n in enumerate(lens):
        mel[b, n:] = np.nan
    return mel


def _check_each_utterance_alone(m, mel, lens, got, lgot):
    c = m.config.combine_frame
    for b, n in enumerate(lens):
        alone, lalone = m.run_mel(mel[b:b + 1, :n], want_logits=True)
        Tb = _frames(n, c)
        assert alone.shape[1] == Tb
        assert np.array_equal(got[b, :Tb], alone[0]), ("utterance", b, "frames", n, np.abs(got[b, :Tb] - alone[0]).max())
        assert np.array_equal(lgot[b, :Tb], lalone[0]), ("utterance", b, "frames", n)
        assert not got[b, Tb:].any() and not lgot[b, Tb:].any(), ("padding rows not zero", b)


# (n_mel, combine, layers, ffn, classes, relu): the shipped config and the others kws_attention_create accepts
_CONFIGS = [(60, 2, 3, 512, 6, True), (60, 2, 1, 512, 6, True), (60, 2, 8, 512, 6, True), (60, 2, 3, 200, 6, True),
            (60, 2, 3, 512, 16, True), (60, 2, 3, 512, 6, False), (41, 3, 3, 512, 6, True), (60, 1, 3, 512, 6, True)]


@pytest.mark.parametrize("n_mel,combine,layers,ffn,classes,relu", _CONFIGS)
def test_lens_batch_is_each_utterance_alone(n_mel, combine, layers, ffn, classes, relu):
    """Bit for bit against single-utterance calls; against the float64 / float32 oracle except at combine 1, where
    nothing here settles whether the reference gives T or T + 1 rows."""
    ow, m = _model(n_mel, combine, layers, ffn, classes, relu, seed=n_mel + 10 * layers + ffn + classes)
    try:
        lens = _lens_for(combine)
        mel = _mel_batch(np.random.default_rng(combine * 100 + layers), lens, n_mel)
        got, lgot = m.run_mel(mel, want_logits=True, lens=np.asarray(lens))
        assert got.shape == (len(lens), _frames(max(lens), combine), classes)
        assert np.isfinite(got).all() and np.isfinite(lgot).all()
        _check_each_utterance_alone(m, mel, lens, got, lgot)
        if combine > 1:
            want64, _ = mel_forward_lens(mel, lens, ow, np.float64, use_relu=relu, combine=combine)
            want, lwant = mel_forward_lens(mel, lens, ow, np.float32, use_relu=relu, combine=combine)
            assert np.abs(got - want64).max() < 1e-3, np.abs(got - want64).max()
            assert np.abs(got - want).max() < 1e-4, np.abs(got - want).max()
            assert np.abs(lgot - lwant).max() < 1e-3, np.abs(lgot - lwant).max()
    finally:
        m.close()


@pytest.fixture(scope="module")
def default_model():
    ow, m = _model()
    yield ow, m
    m.close()


def _c_forward(m, x, B, T, lens_ptr, C, use_lens):
    import torch
    lib_mod, lib = _lib()
    Tp = m.frames(T)
    probs = torch.full((B, Tp, C), float("nan"), device="cuda")
    logits = torch.full((B, Tp, C), float("nan"), device="cuda")
    if use_lens:
        rc = lib.kws_attention_forward_lens(m._handle, x.data_ptr(), B, T, lens_ptr, probs.data_ptr(), logits.data_ptr(),
                                            _stream())
    else:
        rc = lib.kws_attention_forward(m._handle, x.data_ptr(), B, T, probs.data_ptr(), logits.data_ptr(), _stream())
    lib_mod.check(rc)
    return probs.cpu().numpy(), logits.cpu().numpy()


@pytest.mark.parametrize("T", [100, 799, 1000])
def test_null_lens_and_full_lens_equal_the_equal_length_forward(default_model, T):
    import torch
    _, m = default_model
    B = 5
    x = torch.from_numpy(np.abs(np.random.default_rng(T).standard_normal((B, T, 60))).astype(np.float32)).cuda()
    full = torch.full((B,), T, dtype=torch.int32, device="cuda")
    want = _c_forward(m, x, B, T, None, 6, False)
    for ptr in (None, full.data_ptr()):
        got = _c_forward(m, x, B, T, ptr, 6, True)
        np.testing.assert_array_equal(got[0], want[0])
        np.testing.assert_array_equal(got[1], want[1])


def test_device_lens_are_clamped(default_model):
    import torch
    _, m = default_model
    T = 300
    mel = np.abs(np.random.default_rng(4).standard_normal((4, T, 60))).astype(np.float32)
    raw = torch.tensor([0, -5, T + 7, 57], dtype=torch.int32, device="cuda")
    got = m.run_mel(mel, lens=raw)
    want = m.run_mel(mel, lens=np.array([1, 1, T, 57]))
    np.testing.assert_array_equal(got, want)


def test_stale_scratch_and_chunking(default_model):
    """A full-length call with large inputs leaves its activations in the scratch; the variable-length call after it
    must equal a fresh model's, also when MAX_ROWS_PER_CALL splits the batch (lens are sliced with it)."""
    from keyword_spotting_b200 import AttentionDeployModel, AttentionWeights
    ow, m = default_model
    rng = np.random.default_rng(9)
    lens = _lens_for(2)
    mel = _mel_batch(rng, lens, 60)
    big = (np.abs(rng.standard_normal(mel.shape)) * 300.0).astype(np.float32)
    m.run_mel(big)
    got = m.run_mel(mel, lens=lens)
    fresh = AttentionDeployModel(m.config, AttentionWeights.from_object(ow))
    try:
        np.testing.assert_array_equal(got, fresh.run_mel(mel, lens=lens))
    finally:
        fresh.close()
    Tp = got.shape[1]
    m.MAX_ROWS_PER_CALL = 3 * Tp + 7                               # 3 utterances per call
    try:
        chunked = m.run_mel(mel, lens=lens)
        import torch
        chunked_dev = m.run_mel(mel, lens=torch.tensor(lens, dtype=torch.int32, device="cuda"))
    finally:
        del m.MAX_ROWS_PER_CALL
    np.testing.assert_array_equal(chunked, got)
    np.testing.assert_array_equal(chunked_dev, got)


def test_output_lengths(default_model):
    import torch
    _, m = default_model
    assert m.output_lengths(7) == 4
    assert m.output_lengths([1, 2, 799, 800]) == [1, 2, 400, 401]
    assert m.output_lengths((3, 4)) == (2, 3)
    np.testing.assert_array_equal(m.output_lengths(np.array([1, 1000])), [1, 501])
    t = m.output_lengths(torch.tensor([5, 6], device="cuda"))
    assert t.is_cuda and t.tolist() == [3, 4]


def test_pcm_lengths(default_model):
    """forward(pcm, lengths) row by row against forward(pcm[b, :L_b]): frames below T_b read no sample past L_b.  Within
    1e-5, not bit for bit: the front end's mel frames of a padded row can differ from the row alone in the last bits
    (1.9e-7 at most in the probabilities on a B200)."""
    _, m = default_model
    from tests._util import synth_pcm16
    rng = np.random.default_rng(5)
    L = 16000
    lengths = np.array([400, 401, 559, 560, 7999, 12345, L])
    pcm = synth_pcm16(rng, len(lengths), L).astype(np.float32) / 32768.0
    for b, n in enumerate(lengths):
        pcm[b, n:] = rng.standard_normal(L - n) * 3.0          # loud garbage past the end
    got = m.forward(pcm, lengths=lengths)
    worst, exact = 0.0, True
    for b, n in enumerate(lengths):
        alone = m.forward(pcm[b, :n])
        Tb = alone.shape[1]
        assert Tb == m.output_lengths(1 + (int(n) - 400) // 160)
        worst = max(worst, float(np.abs(got[b, :Tb] - alone[0]).max()))
        exact = exact and np.array_equal(got[b, :Tb], alone[0])
        assert not got[b, Tb:].any()
    assert worst <= 1e-5, worst
    print("pcm lengths: max |diff| %.3g, bit-identical %s" % (worst, exact))


def test_bad_lengths_and_lens_raise(default_model):
    import torch
    from keyword_spotting_b200._lib import InvalidArgumentError
    _, m = default_model
    mel = np.zeros((3, 50, 60), np.float32)
    for bad in ([1, 2], [0, 5, 5], [5, 51, 5], np.array([1.0, 2.0, 3.0]), np.zeros((3, 1), np.int32)):
        with pytest.raises(InvalidArgumentError):
            m.run_mel(mel, lens=bad)
    with pytest.raises(InvalidArgumentError):
        m.run_mel(mel, lens=torch.ones(2, dtype=torch.int32, device="cuda"))
    pcm = np.zeros((2, 1000), np.float32)
    for bad in ([400], [399, 500], [500, 1001], [400.0, 500.0]):
        with pytest.raises(InvalidArgumentError):
            m.forward(pcm, lengths=bad)


def test_validate_takes_the_attention_model(default_model):
    """evaluation.validate on mel batches with lens counts what evaluate_softmax counts on per-utterance forwards."""
    from keyword_spotting_b200 import evaluation
    _, m = default_model
    rng = np.random.default_rng(6)
    batches, want = [], dict(miss=0, target=0, false_accept=0, total=0)
    for _ in range(3):
        lens = rng.integers(1, 300, 8)
        mel = _mel_batch(rng, list(lens), 60, T=300)
        corr = rng.integers(0, 2, 8)
        batches.append((mel, lens, corr))
        for b in range(8):
            sm = m.run_mel(mel[b:b + 1, :lens[b]])
            mi, t, fa, _ = evaluation.evaluate_softmax(sm, corr[b:b + 1], label_seqs=m.config.label_seqs)
            want["miss"] += mi
            want["target"] += t
            want["false_accept"] += fa
            want["total"] += 1
    res = evaluation.validate(m, batches)
    assert dict(res) == want


# ================================================================ single kernels through the _lens debug entry points
def _lens_dev(lens):
    import torch
    return torch.tensor(lens, dtype=torch.int32, device="cuda")


def _qkv_with_poisoned_padding(B, Tp, lens, heads, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    qkv = torch.randn((B, Tp, 3 * HEAD * heads), device="cuda", generator=g)
    for b, n in enumerate(lens):
        qkv[b, n:] = float("nan") if b % 3 == 0 else (1e4 if b % 3 == 1 else -1e4)
    return qkv


def _check_core_lens(path, lens, heads=8):
    import torch
    lib_mod, lib = _lib()
    B, Tp = len(lens), max(lens)
    qkv = _qkv_with_poisoned_padding(B, Tp, lens, heads, seed=path + 1)
    out = torch.full((B, Tp, HEAD * heads), 7.0, device="cuda")
    ln = _lens_dev(lens)
    lib_mod.check(lib.kws_debug_att_core_lens(qkv.data_ptr(), B, Tp, ln.data_ptr(), heads, path, out.data_ptr(), _stream()))
    for b, n in enumerate(lens):
        q1 = qkv[b:b + 1, :n].contiguous()
        o1 = torch.empty((1, n, HEAD * heads), device="cuda")
        lib_mod.check(lib.kws_debug_att_core(q1.data_ptr(), 1, n, heads, path, o1.data_ptr(), _stream()))
        assert torch.equal(out[b, :n], o1[0]), ("path", path, "T'_b", n)
        assert bool((out[b, n:] == 7.0).all()), ("rows past T'_b written", path, n)


def test_core_tc_lens_every_key_count():
    _check_core_lens(TC, list(range(1, 401)))


def test_core_ffma_lens():
    _check_core_lens(FFMA, sorted(set(range(1, 1001, 7)) | {127, 128, 129, 400, 401, 512, 513, 1000}))


def test_core_tc_lens_rejects_more_than_400_rows():
    import torch
    _, lib = _lib()
    qkv = torch.zeros((1, 401, 384), device="cuda")
    out = torch.zeros((1, 401, 128), device="cuda")
    ln = _lens_dev([5])
    assert lib.kws_debug_att_core_lens(qkv.data_ptr(), 1, 401, ln.data_ptr(), 8, TC, out.data_ptr(), _stream()) == -4


def test_layernorm_lens_both_paths():
    """Utterance by utterance against a call at Tp = T'_b (which picks the shared-memory path whenever it fits), for
    both paths of the batch call: the two paths do identical arithmetic."""
    import torch
    lib_mod, lib = _lib()
    N = 128
    lens = sorted(set(range(1, 401, 3)) | {16, 17, 128, 129, 399, 400})
    B, Tp = len(lens), 400
    g = torch.Generator(device="cuda").manual_seed(3)
    a = 1e3 + torch.randn((B, Tp, N), device="cuda", generator=g)
    bb = torch.randn((B, Tp, N), device="cuda", generator=g)
    for i, n in enumerate(lens):
        a[i, n:] = float("nan")
        bb[i, n:] = 1e4
    gamma = 1 + 0.3 * torch.randn(N, device="cuda", generator=g)
    beta = torch.randn(N, device="cuda", generator=g)
    ln = _lens_dev(lens)
    outs = []
    for in_smem in (1, 0):
        y = torch.full((B, Tp, N), 7.0, device="cuda")
        lib_mod.check(lib.kws_debug_att_add_layernorm_lens(a.data_ptr(), bb.data_ptr(), gamma.data_ptr(), beta.data_ptr(), B,
                                                           Tp, ln.data_ptr(), N, in_smem, y.data_ptr(), _stream()))
        outs.append(y)
    assert torch.equal(outs[0], outs[1])
    for i, n in enumerate(lens):
        a1, b1 = a[i:i + 1, :n].contiguous(), bb[i:i + 1, :n].contiguous()
        for in_smem in (1, 0):
            y1 = torch.empty((1, n, N), device="cuda")
            lib_mod.check(lib.kws_debug_att_add_layernorm(a1.data_ptr(), b1.data_ptr(), gamma.data_ptr(), beta.data_ptr(), 1,
                                                          n, N, in_smem, y1.data_ptr(), _stream()))
            assert torch.equal(outs[0][i, :n], y1[0]), ("T'_b", n, "in_smem", in_smem)
        assert bool((outs[0][i, n:] == 7.0).all())

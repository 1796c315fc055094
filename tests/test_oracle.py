"""CPU: pin the oracle against the reference's golden vectors / known-answer tests (SURVEY.md 8c)."""
import numpy as np
import pytest

from oracle import cref, model as om, octbit as ooct, posenc as ope, prediction as op, streaming as ost
from tests._util import golden, synth_pcm16, unpack


# ---------------------------------------------------------------- decoders (utils/prediction.py)
@pytest.mark.parametrize("key,fn", [("decode", lambda p: op.ctc_decode(p)),
                                    ("decode2", lambda p: op.ctc_decode2(p, 6)),
                                    ("strict", lambda p: op.ctc_decode_strict(p, 6))])
def test_decoders_match_reference_golden(key, fn):
    g = golden("decode_golden.npz")
    po = g["probs_off"]
    n_trig = 0
    for i in range(len(po) - 1):
        p = unpack(g["probs"], po, i, 6)
        want = unpack(g[key], g[key + "_off"], i)
        got = fn(p)
        assert got.dtype == np.int32
        np.testing.assert_array_equal(got, want)
        assert op.ctc_predict(got, "1233") == g[key + "_pred"][i]
        n_trig += int(g[key + "_pred"][i])
    assert n_trig > 0           # the fixture really exercises the trigger


def test_decoders_nondefault_params_match_reference_golden():
    g = golden("decode_golden.npz")
    eo = g["extra_probs_off"]
    for i in range(len(eo) - 1):
        p = unpack(g["extra_probs"], eo, i, 6)
        lo, th, ls = int(g["extra_lockout"][i]), float(g["extra_thres"][i]), float(g["extra_loose"][i])
        np.testing.assert_array_equal(op.ctc_decode(p, lo, th, ls), unpack(g["extra_decode"], g["extra_decode_off"], i))
        np.testing.assert_array_equal(op.ctc_decode2(p, 6, th), unpack(g["extra_decode2"], g["extra_decode2_off"], i))
        np.testing.assert_array_equal(op.ctc_decode_strict(p, 6, lo, th), unpack(g["extra_strict"], g["extra_strict_off"], i))


def test_predict_and_evaluate_match_reference_golden():
    g = golden("decode_golden.npz")
    off = g["predict_cases_off"]
    for i in range(len(off) - 1):
        seq = unpack(g["predict_cases"], off, i)
        assert op.ctc_predict(seq, "1233") == g["predict_out"][i]
        assert op.ctc_predict(seq, "123") == g["predict_out_123"][i]
    assert tuple(op.evaluate(g["eval_result"], g["eval_target"])) == tuple(int(v) for v in g["eval_out"])


def test_vad_and_queue_match_reference_golden():
    g = golden("vad_queue_golden.npz")
    so = g["sig_off"]
    for i in range(len(so) - 1):
        sig = unpack(g["sig"], so, i)
        assert ost.vad(sig, 30) == bool(g["vad"][i, 0])
        assert ost.vad(sig) == bool(g["vad"][i, 1])
    q = ost.SimpleQueue(15)
    for i, opv in enumerate(g["queue_ops"]):
        if opv < 0:
            q.clear()
        else:
            q.add(int(opv))
        snap = list(q.get_all()) + [-1] * (15 - len(q.get_all()))
        np.testing.assert_array_equal(np.asarray(snap, np.int32), g["queue_snap"][i])


def test_integer_vad_equals_float_vad_away_from_threshold():
    rng = np.random.default_rng(3)
    for amp in (1, 3, 100, 200, 210, 3000):
        pcm = rng.integers(-amp, amp + 1, size=(8, 4800)).astype(np.int16)
        f = np.array([ost.vad(om.pcm16_to_float(r), 30) for r in pcm])
        i = ost.vad_pcm16(pcm, 30)
        margin = np.abs(np.abs(pcm.astype(np.int64)).sum(axis=1) - 30 * 32768)
        ok = margin > 64          # fp32 pairwise-sum noise is far below 64 LSB here
        np.testing.assert_array_equal(f[ok], i[ok])


# ---------------------------------------------------------------- octbit (octbit_mat_mul_op.cc)
def test_octbit_reference_known_answers():
    # octbit/octbit_ops_test.py:24-34
    out = ooct.octbit_mat_mul(-np.ones((1, 64), np.float32), np.arange(64, dtype=np.int8)[None], scale=3.0,
                              bias=[127 * 2016.0])
    np.testing.assert_array_equal(out, [[-6048.0]])
    # octbit/octbit_ops_test.py:41-53
    w = np.stack([np.ones(64)] + [np.arange(64)] * 3).astype(np.int8)
    out = ooct.octbit_mat_mul(-np.ones((2, 64), np.float32), w, scale=2.0,
                              bias=[127 * 64.0, 127 * 2016.0, 127 * 2016.0, 127 * 2016.0])
    np.testing.assert_array_equal(out, [[-128.0, -4032.0, -4032.0, -4032.0]] * 2)


def _octbit_cases():
    g = golden("octbit_golden.npz")
    keys = sorted(k[:-2] for k in g.files if k.endswith("_x"))
    return g, keys


def test_octbit_numpy_and_c_match_reference_kernel_golden():
    g, keys = _octbit_cases()
    assert len(keys) >= 27
    for k in keys:
        x, w, bias, scale, want = g[k + "_x"], g[k + "_w"], g[k + "_bias"], float(g[k + "_scale"]), g[k + "_out"]
        got = ooct.octbit_mat_mul(x, w, scale=scale, bias=bias)
        assert got.tobytes() == want.tobytes(), k
        got_c = cref.c_octbit_matmul(x, w, bias, scale)
        assert got_c.tobytes() == want.tobytes(), k


def test_octbit_golden_contains_saturating_pairs():
    g, keys = _octbit_cases()
    n_sat = 0
    for k in keys:
        if not k.endswith("saturating"):
            continue
        q, _, _ = ooct.quantize_activations(g[k + "_x"])
        pair = (q.astype(np.int32)[:, None, :] * g[k + "_w"].astype(np.int32)[None]).reshape(q.shape[0], -1, q.shape[1] // 2, 2).sum(-1)
        n_sat += int((np.abs(pair) > 32767).sum())
    assert n_sat > 1000


@pytest.mark.skipif(not cref.have_ref(), reason="oracle/_ref not built (reference sources absent)")
def test_octbit_oracle_matches_live_reference_kernel():
    rng = np.random.default_rng(11)
    for (A, B, K) in [(1, 1, 64), (9, 33, 128), (4, 7, 576), (2, 3, 2048)]:
        x = rng.standard_normal((A, K)).astype(np.float32) * rng.uniform(0.1, 30)
        w = rng.integers(-128, 128, (B, K)).astype(np.int8)
        bias = rng.standard_normal(B).astype(np.float32) * 1000
        want = cref.ref_octbit_matmul(x, w, bias, 0.37)
        assert ooct.octbit_mat_mul(x, w, scale=0.37, bias=bias).tobytes() == want.tobytes()
        assert cref.c_octbit_matmul(x, w, bias, 0.37).tobytes() == want.tobytes()


def test_octbit_argument_checks_follow_the_op():
    x = np.zeros((1, 64), np.float32)
    w = np.zeros((1, 64), np.int8)
    with pytest.raises(ooct.InvalidArgument):
        ooct.octbit_mat_mul(x, w, scale=0.0, bias=[0])            # :46 scale > 0 (the wrapper's default!)
    with pytest.raises(ooct.InvalidArgument):
        ooct.octbit_mat_mul(x, w, transpose_b=False, scale=1.0)   # :41
    with pytest.raises(ooct.InvalidArgument):
        ooct.octbit_mat_mul(x, w, transpose_a=True, scale=1.0)    # :42
    with pytest.raises(ooct.InvalidArgument):
        ooct.octbit_mat_mul(x[:, :32], w[:, :32], scale=1.0)      # :65-67
    with pytest.raises(ooct.InvalidArgument):
        ooct.octbit_mat_mul(x, w[:, :32], scale=1.0)              # :61-63


def test_octize_recipe():
    rng = np.random.default_rng(5)
    w = (rng.standard_normal((256, 128)) * 0.07).astype(np.float32)
    wq, scale, bias = ooct.octize_weight_int8_signed(w)
    assert wq.shape == (128, 256) and wq.dtype == np.int8
    assert np.abs(wq).max() == 127
    np.testing.assert_allclose(scale, np.abs(w).max() / 127.0, rtol=1e-7)
    np.testing.assert_array_equal(bias, 127.0 * wq.astype(np.float64).sum(axis=1))
    np.testing.assert_allclose(wq.T * scale, w, atol=scale * 0.5001)
    assert ooct.default_octbit_matmul_name_check("model/drnn/multi_rnn_cell/cell_1/gru_cell/gates/MatMul")
    assert not ooct.default_octbit_matmul_name_check("model/drnn/multi_rnn_cell/cell_0/gru_cell/gates/MatMul")
    assert not ooct.default_octbit_matmul_name_check("model/linear/linear/MatMul")


# ---------------------------------------------------------------- positional encoding
def test_posenc_matches_reference_kernel_golden():
    g = golden("posenc_golden.npz")
    assert len(g.files) >= 7
    for key in g.files:
        _, mp, sz = key.split("_")
        want = g[key]
        assert ope.positional_encoding(int(mp), int(sz), fill=-9.0).tobytes() == want.tobytes(), key
        assert cref.c_positional_encoding(int(mp), int(sz), fill=-9.0).tobytes() == want.tobytes(), key


def test_posenc_odd_size_leaves_last_column():
    pe = ope.positional_encoding(4, 5, fill=-9.0)
    assert (pe[:, 4] == -9.0).all() and (pe[0, :4] == [0, 1, 0, 1]).all()


# ---------------------------------------------------------------- model path (parity unpinned: self-consistency)
def test_mel_basis_properties():
    for M in (40, 60):
        mb = om.slaney_mel_basis(n_mels=M)
        assert mb.shape == (M, 201)
        assert (mb >= 0).all()
        freqs = np.linspace(0, 8000, 201)
        assert (mb[:, freqs < 300].sum() == 0)
        assert (mb.sum(axis=1) > 0).all()
        peaks = mb.argmax(axis=1)
        assert (np.diff(peaks) > 0).all()


def test_mel_basis_matches_an_independent_slaney_implementation():
    """librosa is not installable here; `transformers.audio_utils.mel_filter_bank(norm='slaney', mel_scale='slaney')` is
    an independent third-party implementation of the same `librosa.filters.mel` definition the reference calls
    (models/rnn_ctc.py:139-144: sr=16000, n_fft=400, fmin=300, fmax=8000).  It pins row a6's constant."""
    audio_utils = pytest.importorskip("transformers.audio_utils")
    for M in (40, 60):
        fb = audio_utils.mel_filter_bank(num_frequency_bins=201, num_mel_filters=M, min_frequency=300.0,
                                         max_frequency=8000.0, sampling_rate=16000, norm="slaney", mel_scale="slaney")
        np.testing.assert_allclose(om.slaney_mel_basis(n_mels=M), fb.T, rtol=0, atol=1e-15)
        w = om.init_weights(seed=1, n_mel=M)
        np.testing.assert_array_equal(w.mel_basis, fb.astype(np.float32))     # [201, M] f32 constant, as the graph holds it


def test_framing_and_rfft_magnitude_match_numpy_stride_tricks():
    """Row a4/a5 against an independent formulation: frames by stride tricks (utils/stft.py:67-79 builds the same
    index grid), |rfft| by an explicit DFT matrix in float64."""
    rng = np.random.default_rng(3)
    x = rng.standard_normal((2, 2000))
    fr = np.lib.stride_tricks.sliding_window_view(x, 400, axis=1)[:, ::160]
    np.testing.assert_array_equal(om.frame(x), fr)
    n = np.arange(400)
    dft = np.exp(-2j * np.pi * np.outer(n, np.arange(201)) / 400)
    want = np.abs(fr @ dft)
    got = np.abs(np.fft.rfft(om.frame(x), n=400, axis=-1))
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-9)
    w = om.init_weights(seed=1, n_mel=40)
    mel = om.pcm_to_mel(x, w, np.float64)
    np.testing.assert_allclose(mel, want @ w.mel_basis.astype(np.float64), rtol=0, atol=1e-9)


def test_num_frames_and_framing():
    assert om.num_frames(4800) == 28 and om.num_frames(5120) == 30 and om.num_frames(48000) == 298
    assert om.num_frames(400) == 1 and om.num_frames(399) == 0
    x = np.arange(1000, dtype=np.float32)[None]
    fr = om.frame(x)
    assert fr.shape == (1, 4, 400)
    np.testing.assert_array_equal(fr[0, 3], np.arange(480, 880))


def test_gru_float32_tracks_float64_and_masks_lengths():
    w = om.init_weights(seed=7)
    rng = np.random.default_rng(8)
    mel = np.abs(rng.standard_normal((5, 40, 40))).astype(np.float32) * 3
    st = (rng.standard_normal((2, 5, 128)) * 0.3).astype(np.float32)
    p32, s32, _ = om.mel_forward(mel, st, w, dtype=np.float32)
    p64, s64, _ = om.mel_forward(mel, st, w, dtype=np.float64)
    assert np.abs(p32 - p64).max() < 2e-5 and np.abs(s32 - s64).max() < 2e-5
    np.testing.assert_allclose(p32.sum(-1), 1.0, atol=1e-5)
    lens = np.array([40, 17, 0, 1, 39])
    pm, sm, _ = om.mel_forward(mel, st, w, seq_len=lens, dtype=np.float32)
    for s, ln in enumerate(lens):
        ps, ss, _ = om.mel_forward(mel[s:s + 1, :ln], st[:, s:s + 1], w, dtype=np.float32)
        np.testing.assert_allclose(pm[s, :ln], ps[0], atol=1e-6)
        np.testing.assert_allclose(sm[:, s], ss[:, 0], atol=1e-6)
        if ln < 40:     # zero outputs -> softmax(bias)
            np.testing.assert_allclose(pm[s, ln:], om.softmax(w.fc_b[None])[0][None].repeat(40 - ln, 0), atol=1e-6)


def test_streaming_equals_offline_like_detector_test2():
    """detector.py:254-289: 3600-sample segments with carried tail/state == whole utterance."""
    w = om.init_weights(seed=2)
    rng = np.random.default_rng(9)
    pcm = (rng.standard_normal(16000) * 0.05).astype(np.float32)
    used = len(pcm) - (len(pcm) - 400) % 160
    whole, st_whole, _ = om.deploy_forward(pcm[:used], np.zeros((2, 1, 128), np.float32), w)
    streamed, st_stream = ost.stream_vs_offline(pcm, w, seg_len=3600)
    assert streamed.shape == whole[0].shape
    np.testing.assert_allclose(streamed, whole[0], atol=2e-5)
    np.testing.assert_allclose(st_stream, st_whole, atol=2e-5)


def test_stream_oracle_runs_and_resets():
    from tests._util import synth_pcm16
    w = om.init_weights(seed=1234)
    rng = np.random.default_rng(5678)
    so = ost.StreamOracle(w, 6)
    pcm = synth_pcm16(rng, 6, 4800 * 3, silent_frac=0.5)
    for c in range(3):
        r = so.step(pcm[:, c * 4800:(c + 1) * 4800])
        assert r["softmax"].shape == (6, 28 if c == 0 else 30, 6)
        for s in np.nonzero(~r["speech"])[0]:
            assert len(so.queues[s].get_all()) == 1     # cleared, then this chunk pushed
    assert so.res.shape[1] == 320


def _wer_golden():
    g = golden("wer_golden.npz")
    refs = [g["ref"][g["ref_off"][i]:g["ref_off"][i + 1]].tolist() for i in range(len(g["ref_off"]) - 1)]
    hyps = [g["hyp"][g["hyp_off"][i]:g["hyp_off"][i + 1]].tolist() for i in range(len(g["hyp_off"]) - 1)]
    return g, refs, hyps


def test_wer_oracle_matches_reference_golden():
    """oracle/wer.py against values produced by the reference's own utils/wer.py (tests/golden/make_wer_golden.py)."""
    from oracle import wer as ow
    g, refs, hyps = _wer_golden()
    got = np.asarray([ow.wer(r, h) for r, h in zip(refs, hyps)])
    np.testing.assert_array_equal(got, g["wer"])
    assert max(len(r) for r in refs) == 254          # the reference's uint8 limit is covered


def test_ambiguous_frames_cover_every_possible_token_flip():
    """oracle.streaming.ambiguous_frames: for any two softmax arrays within `tol` of each other the ctc_decode2 token
    (above-threshold winner of the label columns, else none) may differ ONLY at frames flagged ambiguous."""
    from oracle import streaming as ost
    rng = np.random.default_rng(11)
    tol, thres = 1e-3, 0.4
    n_flip = 0
    for trial in range(40):
        logits = rng.standard_normal((64, 30, 6)) * rng.uniform(0.5, 4.0)
        # crowd many frames around the threshold / around ties
        p = np.exp(logits) / np.exp(logits).sum(-1, keepdims=True)
        p[::3, :, 1] = thres + rng.uniform(-3 * tol, 3 * tol, p[::3, :, 1].shape)
        p[1::3, :, 2] = p[1::3, :, 1] + rng.uniform(-4 * tol, 4 * tol, p[1::3, :, 1].shape)
        p = p.astype(np.float32)
        q = (p + rng.uniform(-tol, tol, p.shape) * 0.999).astype(np.float32)

        def token(a):
            lab = a[..., 1:-1].astype(np.float64)
            return np.where(lab.max(-1) > thres, lab.argmax(-1), -1)

        flip = token(p) != token(q)
        amb = ost.ambiguous_frames(p, thres, tol)
        assert not (flip & ~amb).any()
        n_flip += int(flip.sum())
    assert n_flip > 100        # the construction really produces flips


def test_stream_oracle_decide_on_hook_only_changes_the_decision_window():
    from oracle import model as om, streaming as ost
    ow = om.init_weights(seed=1234, n_mel=40)
    ow.fc_w = (ow.fc_w * 6).astype(np.float32)
    rng = np.random.default_rng(5)
    pcm = synth_pcm16(rng, 6, 4800 * 3, silent_frac=0.0)
    a, b = ost.StreamOracle(ow, 6, label="1"), ost.StreamOracle(ow, 6, label="1")
    for c in range(3):
        blk = pcm[:, c * 4800:(c + 1) * 4800]
        ra = a.step(blk)
        rb = b.step(blk, decide_on=lambda sm: sm.copy())             # identity hook: identical run
        np.testing.assert_array_equal(ra["trigger"], rb["trigger"])
        np.testing.assert_array_equal(ra["softmax"], rb["softmax"])
    never = ost.StreamOracle(ow, 6, label="1")
    fired = 0
    for c in range(3):
        r = never.step(pcm[:, c * 4800:(c + 1) * 4800], decide_on=lambda sm: np.zeros_like(sm))
        fired += int(r["trigger"].sum())
        assert r["softmax"].max() > 0.1                              # the returned softmax stays the oracle's own
    assert fired == 0


# ---------------------------------------------------------------- attention_ctc oracle (oracle/attention.py)
_ATTENTION_DEFAULT_WEIGHTS_SHA256 = "5eb546514f69998ad00afa584478e85b367fbf16f5212b50f905e1e72032603d"


def test_attention_oracle_defaults_are_the_shipped_config_unchanged():
    """init_weights / mel_forward take the config as parameters; their defaults must keep giving the weights and outputs
    that the shipped-config tests were written against.  The weights are pinned bit for bit (sha256 of every array, in
    field order); the outputs of a fixed mel batch (default_rng(77), [2, 9, 60]) are pinned in float64 to 1e-12, which
    only leaves room for a BLAS that orders its sums differently."""
    import hashlib
    from oracle import attention as oa
    w = oa.init_weights()
    h = hashlib.sha256()
    for name in ("mel_basis", "w_in", "b_in", "w_qkv", "b_qkv", "ln1_g", "ln1_b", "w_ff1", "b_ff1", "w_ff2", "b_ff2",
                 "ln2_g", "ln2_b", "w_out", "b_out"):
        v = getattr(w, name)
        for a in (v if isinstance(v, list) else [v]):
            h.update(np.ascontiguousarray(a).tobytes())
    assert h.hexdigest() == _ATTENTION_DEFAULT_WEIGHTS_SHA256
    explicit = oa.init_weights(seed=4321, n_mel=60, combine=2, layers=3, ffn=512, classes=6)
    for name in ("w_in", "w_qkv", "w_ff1", "w_ff2", "b_ff2", "w_out", "b_out"):
        np.testing.assert_array_equal(np.asarray(getattr(w, name)), np.asarray(getattr(explicit, name)))
    mel = np.abs(np.random.default_rng(77).standard_normal((2, 9, 60))).astype(np.float32)
    g = golden("attention_oracle_golden.npz")
    probs, logits = oa.mel_forward(mel, w, np.float64)
    np.testing.assert_allclose(probs, g["probs"], rtol=1e-12, atol=0)
    np.testing.assert_allclose(logits, g["logits"], rtol=1e-12, atol=1e-15)
    p2, l2 = oa.mel_forward(mel, w, np.float64, use_relu=True, combine=2)
    np.testing.assert_array_equal(p2, probs)
    np.testing.assert_array_equal(l2, logits)


def test_attention_oracle_other_configs_have_their_shapes():
    from oracle import attention as oa
    w = oa.init_weights(seed=1, n_mel=41, combine=3, layers=2, ffn=200, classes=16)
    assert w.w_in.shape == (123, 128) and len(w.w_qkv) == 2 and w.w_ff1[1].shape == (128, 200)
    assert w.w_out.shape == (128, 16) and w.mel_basis.shape == (201, 41)
    mel = np.ones((2, 10, 41), np.float32)
    probs, logits = oa.mel_forward(mel, w, np.float64, use_relu=False, combine=3)
    assert probs.shape == logits.shape == (2, 10 // 3 + 1, 16)
    assert (logits < 0).any()                                   # no relu on the output layer
    np.testing.assert_allclose(probs.sum(-1), 1, rtol=1e-12)

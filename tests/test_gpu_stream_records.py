"""Per-stream records (kws_stream_export / kws_stream_import, kws_server_export / kws_server_import): a stream moved
to another slot, object, wave server or GPU continues bit for bit as it would have where it was; streams not moved
are untouched; records are canonical; malformed records are rejected without touching their target."""
import numpy as np
import pytest

from tests._util import make_config, synth_pcm16, to_product_weights

pytestmark = pytest.mark.gpu

LENS = (4800, 4000, 3600)


def _model(precision="tc", octbit=False, device=None, gain=3.0, seed=21):
    """FC gain 3 and keyword "1" (as test_gpu_server.py): triggers fire, so both reset branches run."""
    from keyword_spotting_b200 import DeployModel, OctbitModelWeights
    from oracle import model as om
    ow = om.init_weights(seed=seed, n_mel=40)
    ow.fc_w = (ow.fc_w * gain).astype(np.float32)
    dm = DeployModel(make_config(40), to_product_weights(ow), precision=precision, device=device)
    if octbit:
        dm.set_octbit(OctbitModelWeights.from_float(dm.weights))
    return dm


def _chunk(rng, S, n, quiet_frac=0.3):
    """[S, n] int16; about quiet_frac of the rows are below the VAD threshold."""
    pcm = synth_pcm16(rng, S, n, silent_frac=0.0)
    quiet = rng.random(S) < quiet_frac
    pcm[quiet] = rng.integers(-2, 3, (int(quiet.sum()), n))
    return pcm, quiet


def _run_until_trigger(det, rng, min_chunks, max_chunks=40):
    """Step `det` at varying chunk lengths for at least min_chunks chunks, until its last chunk raised a trigger."""
    for c in range(max_chunks):
        pcm, quiet = _chunk(rng, det.n_streams, int(rng.choice(LENS)))
        trig = det.step(pcm)
        if c + 1 >= min_chunks and trig.any():
            return trig, quiet
    raise AssertionError("no trigger in %d chunks" % max_chunks)


def _pick_ids(rng, S, trig, quiet, n=100):
    """About n distinct ids of an S-stream object: 0, S-1, streams that triggered and streams that were quiet in the
    last chunk, and the rest spread at random."""
    must = [0, S - 1] + list(np.nonzero(trig)[0][:20]) + list(np.nonzero(quiet)[0][:20])
    rest = rng.permutation(S)
    ids = list(dict.fromkeys(must + list(rest)))[:n]
    return np.array(ids, dtype=np.int64)


def _continue_both(src, dst, ids, slots, rng, chunks):
    """Step src and dst `chunks` times, dst's slots fed src's ids' PCM; every output of a moved stream must match."""
    import torch
    for c in range(chunks):
        n = int(rng.choice(LENS))
        pa, _ = _chunk(rng, src.n_streams, n)
        pb, _ = _chunk(rng, dst.n_streams, n)
        pb[slots] = pa[ids]
        ta, pra, na = src.step(pa, want_probs=True)
        tb, prb, nb = dst.step(pb, want_probs=True)
        np.testing.assert_array_equal(tb[slots], ta[ids], err_msg="chunk %d" % c)
        np.testing.assert_array_equal(nb[slots], na[ids], err_msg="chunk %d" % c)
        np.testing.assert_array_equal(prb[slots], pra[ids], err_msg="chunk %d" % c)
        assert torch.equal(dst.state()[:, torch.as_tensor(slots)], src.state()[:, torch.as_tensor(ids)]), c
        la, ca = src.window_labels()
        lb, cb = dst.window_labels()
        np.testing.assert_array_equal(cb[slots], ca[ids])
        np.testing.assert_array_equal(lb[slots], la[ids])


@pytest.mark.parametrize("variant", ["tc", "fp32", "octbit", "tc_host_bytes"])
def test_moved_streams_continue_bit_exact_and_others_are_untouched(variant):
    import torch
    from keyword_spotting_b200 import StreamingDetector
    dm = _model("fp32" if variant == "fp32" else "tc", octbit=variant == "octbit")
    rng = np.random.default_rng(101)
    A = StreamingDetector(dm, 640, keyword="1")
    B = StreamingDetector(dm, 300, keyword="1")
    trig, quiet = _run_until_trigger(A, rng, 20)             # the windows wrap (20 > 15 chunks)
    for _ in range(3):                                      # B's own streams carry state of their own
        B.step(_chunk(rng, 300, int(rng.choice(LENS)))[0])
    ids = _pick_ids(rng, 640, trig, quiet)
    slots = rng.permutation(300)[:ids.size]
    others = np.setdiff1d(np.arange(300), slots)
    state_before, (lab_before, cnt_before) = B.state(), B.window_labels()
    rec_before = B.export_streams(others)

    recs = A.export_streams(ids)
    assert recs.dtype == torch.uint8 and recs.is_cuda and tuple(recs.shape) == (ids.size, A.record_bytes)
    if variant == "tc_host_bytes":
        raw = recs.cpu().numpy().tobytes()
        B.import_streams(slots, np.frombuffer(raw, dtype=np.uint8).reshape(ids.size, -1))
    else:
        B.import_streams(slots, recs)
    assert torch.equal(B.export_streams(slots), recs)       # canonical: the same bytes from another object

    o = torch.as_tensor(others)
    assert torch.equal(B.state()[:, o], state_before[:, o])
    lab, cnt = B.window_labels()
    np.testing.assert_array_equal(cnt[others], cnt_before[others])
    np.testing.assert_array_equal(lab[others], lab_before[others])
    assert torch.equal(B.export_streams(others), rec_before)

    _continue_both(A, B, ids, slots, rng, 6)
    A.close()
    B.close()
    dm.close()


def test_records_are_canonical():
    import torch
    from keyword_spotting_b200 import StreamingDetector
    dm = _model("tc")
    rng = np.random.default_rng(7)
    A = StreamingDetector(dm, 256, keyword="1")
    fresh = StreamingDetector(dm, 40, keyword="1")
    zero_rec = fresh.export_streams(np.arange(40))
    assert torch.equal(zero_rec, zero_rec[:1].expand(40, -1))
    assert torch.equal(A.export_streams([0, 255]), zero_rec[:2])     # fresh objects of the same layout agree
    _run_until_trigger(A, rng, 17)
    ids = rng.permutation(256)[:150]
    recs = A.export_streams(ids)
    A.import_streams(ids, recs)                                       # the ring now starts at entry 0
    assert torch.equal(A.export_streams(ids), recs)
    assert not torch.equal(recs, zero_rec[:1].expand(150, -1))
    A.reset()
    assert torch.equal(A.export_streams(np.arange(256)), zero_rec[:1].expand(256, -1))
    A.close()
    fresh.close()
    dm.close()


@pytest.mark.parametrize("use_graphs", [True, False], ids=["graphs", "direct"])
def test_wave_server_import_export(use_graphs):
    import torch
    from keyword_spotting_b200 import InvalidArgumentError, StreamingDetector, WaveServer
    dm = _model("tc")
    rng = np.random.default_rng(33)
    CH = 4800
    D = StreamingDetector(dm, 640, keyword="1")
    srv = WaveServer(dm, 400, waves=4, use_graphs=use_graphs, keyword="1")
    assert srv.graphs == use_graphs and srv.record_bytes == D.record_bytes
    trig = None
    for c in range(6):
        pcm, quiet = _chunk(rng, 640, CH)
        trig = D.step(pcm)
    for c in range(3):                                     # odd: under graph replay every wave's tail half is 1
        srv.step(_chunk(rng, 400, CH)[0])
    ids = _pick_ids(rng, 640, trig, quiet, n=120)
    slots = rng.permutation(400)[:ids.size]
    assert len(set(slots // srv.streams_per_wave)) == 4
    others = np.setdiff1d(np.arange(400), slots)
    rec_others = srv.export_streams(others)
    srv.import_streams(slots, D.export_streams(ids))
    assert torch.equal(srv.export_streams(others), rec_others)

    def both(n_chunks):
        for c in range(n_chunks):
            pd, _ = _chunk(rng, 640, CH)
            ps, _ = _chunk(rng, 400, CH)
            ps[slots] = pd[ids]
            np.testing.assert_array_equal(srv.step(ps)[slots], D.step(pd)[ids], err_msg="chunk %d" % c)
            assert torch.equal(srv.state()[:, torch.as_tensor(slots)], D.state()[:, torch.as_tensor(ids)]), c
            ld, cd = D.window_labels(max_labels=64)
            ls, cs = srv.window_labels(max_labels=64)
            np.testing.assert_array_equal(cs[slots], cd[ids])
            np.testing.assert_array_equal(ls[slots], ld[ids])
        assert torch.equal(srv.export_streams(slots), D.export_streams(ids))

    both(5)
    srv.import_streams(slots, D.export_streams(ids))       # after an even count too (tail half 0 under replay)
    both(2)

    # server -> detector
    E = StreamingDetector(dm, 200, keyword="1")
    back = rng.permutation(200)[:ids.size]
    E.import_streams(back, srv.export_streams(slots))
    _continue_both(D, E, ids, back, rng, 3)

    srv.submit(0)
    with pytest.raises(InvalidArgumentError):
        srv.export_streams(slots)
    with pytest.raises(InvalidArgumentError):
        srv.import_streams(slots, D.export_streams(ids))
    srv.wait(0)
    srv.export_streams([0, 399])
    with pytest.raises(InvalidArgumentError):
        srv.export_streams([400])
    E.close()
    srv.close()
    D.close()
    dm.close()


def test_rejected_records_leave_their_stream_untouched():
    import torch
    from keyword_spotting_b200 import InvalidArgumentError, StreamingDetector
    dm = _model("tc")
    rng = np.random.default_rng(55)
    A = StreamingDetector(dm, 64, keyword="1")
    other = StreamingDetector(dm, 64, keyword="1", window_chunks=10)
    for _ in range(4):
        pcm = synth_pcm16(rng, 64, 4000, silent_frac=0.0)
        A.step(pcm)
        other.step(pcm)
    W, L, R = 15, 2, A.record_bytes
    recs = A.export_streams(np.arange(64)).cpu().numpy()
    words = recs.view(np.int32)
    slot0 = 48 + 512 * L + 800
    tok0 = slot0 + 16
    # a donor with a window entry whose first frame holds a token, and a tail
    donor = int(np.nonzero((words[:, 9] >= 1) & (recs[:, slot0] >= 1) & (words[:, 8] > 0))[0][0])
    good = recs[donor].copy()
    target, bystander = 7 if donor != 7 else 8, 20 if donor != 20 else 21

    def corrupt(fn):
        r = good.copy()
        fn(r, r.view(np.int32))
        return r

    from_other = np.zeros_like(good)                       # another window_chunks: another size, padded to this one
    rec_other = other.export_streams([donor]).cpu().numpy()[0]
    assert rec_other.size != R
    from_other[:rec_other.size] = rec_other
    cases = {
        "header does not match": [from_other, corrupt(lambda r, w: w.__setitem__(0, w[0] ^ 1))],
        "malformed field": [
            corrupt(lambda r, w: w.__setitem__(8, 400)),            # tail_len
            corrupt(lambda r, w: w.__setitem__(9, W + 1)),          # win_n
            corrupt(lambda r, w: r.__setitem__(slot0, A.max_frames + 1)),
            corrupt(lambda r, w: r.__setitem__(tok0, 9)),
        ],
    }
    with pytest.raises(InvalidArgumentError):
        A.import_streams([target], rec_other[None])         # the wrong size is refused before any launch
    for reason, bad_records in cases.items():
        for bad in bad_records:
            before = A.export_streams(np.arange(64))
            state = A.state()
            with pytest.raises(InvalidArgumentError, match="entry 0 \\(id %d\\): %s" % (target, reason)):
                A.import_streams([target, bystander], np.stack([bad, good]))
            after = A.export_streams(np.arange(64))
            keep = torch.as_tensor(np.setdiff1d(np.arange(64), [bystander]))
            assert torch.equal(after[keep], before[keep])
            assert torch.equal(A.state()[:, keep], state[:, keep])
            assert np.array_equal(after[bystander].cpu().numpy(), good)    # the valid record of the batch lands
            A.import_streams([bystander], before[bystander:bystander + 1])

    # ids: host ids are checked in Python, CUDA ids by the kernels
    with pytest.raises(InvalidArgumentError):
        A.import_streams([64], good[None])
    with pytest.raises(InvalidArgumentError):
        A.import_streams([3, 3], np.stack([good, good]))
    with pytest.raises(InvalidArgumentError):
        A.export_streams([-1])
    dev_ids = torch.tensor([64, -5], dtype=torch.int64, device=A.device)
    before = A.export_streams(np.arange(64))
    with pytest.raises(InvalidArgumentError, match="entry 1 \\(id -5\\): id out of range"):
        A.import_streams(dev_ids, np.stack([good, good]))
    assert torch.equal(A.export_streams(np.arange(64)), before)
    assert int(A.export_streams(dev_ids).sum()) == 0
    with pytest.raises(InvalidArgumentError, match="header does not match"):
        A.import_streams([5], A.export_streams(torch.tensor([99], device=A.device)))
    A.close()
    other.close()
    dm.close()


@pytest.mark.skipif("__import__('torch').cuda.device_count() < 2", reason="needs two visible GPUs")
def test_move_streams_between_gpus():
    from keyword_spotting_b200 import StreamingDetector
    dm0 = _model("tc", device=0)
    dm1 = _model("tc", device=1)
    rng = np.random.default_rng(9)
    A = StreamingDetector(dm0, 256, keyword="1")
    B = StreamingDetector(dm1, 128, keyword="1")
    trig, quiet = _run_until_trigger(A, rng, 16)
    ids = _pick_ids(rng, 256, trig, quiet, n=64)
    slots = rng.permutation(128)[:ids.size]
    B.import_streams(slots, A.export_streams(ids).to("cuda:1"))
    _continue_both(A, B, ids, slots, rng, 4)
    A.close()
    B.close()
    dm0.close()
    dm1.close()

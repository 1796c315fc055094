"""PCM rows of different lengths: kws_deploy_forward_lens (rnn_ctc) and AttentionDeployModel.forward(lengths=) against
what a user can do without them.

PCM resident in HBM (larger than the 126 MB L2 at the default sizes), one GPU.  Every variant is warmed up, the variants
of a case are alternated in one process and repeated to show the spread (CUDA events around --iters calls; median / min
/ max over --repeats):

  1  rnn_ctc, BASELINE config-2 shape: int16 utterances uniform over 1-3 s, probabilities then labels
     (kws_ctc_decode with the per-row frame counts), at --utterances and at --full (the GPU full):
       deploy_forward_lens  vs  deploy_forward padded to 3 s (rows past the end computed from padding)
       vs  one deploy_forward per distinct length (rows gathered by length beforehand, not timed)
  2  attention_ctc from float PCM, --att-utterances uniform over 1-8 s:
       forward(lengths=) through kws_frontend_mel_lens  vs  the earlier path (kws_frontend_mel on the padded batch, then
       kws_attention_forward_lens), and the front end alone (its share)
  3  equal lengths, no regression: lengths = NULL vs lengths = L for every row, rnn_ctc (3 s) and attention (8 s)

Audio-s/s counts valid audio only.  The card's name and power limit are read in the same run.

    python tools/pcm_lengths_bench.py [--utterances 4096] [--full 32768] [--att-utterances 1024] [--out results.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SR, FFT, HOP = 16000, 400, 160


def card(index):
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001 -- the measurement stands without it; say so
        q = "nvidia-smi unavailable (%s)" % e
    return dict(device=torch.cuda.get_device_name(index), nvidia_smi=q)


def frames(samples):
    return np.maximum(0, 1 + (np.asarray(samples) - FFT) // HOP)


def time_variants(variants, repeats, iters):
    """variants: name -> callable.  Warm every one up, then alternate them `repeats` times; ms per call each time."""
    for fn in variants.values():
        fn()
        fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in variants}
    for _ in range(repeats):
        for name, fn in variants.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                fn()
            b.record()
            b.synchronize()
            ms[name].append(a.elapsed_time(b) / iters)
    return ms


def summarize(case, ms, audio_s, extra=None):
    rows = []
    for name, v in ms.items():
        med = float(np.median(v))
        rows.append(dict(case=case, variant=name, ms_median=med, ms_min=float(min(v)), ms_max=float(max(v)),
                         valid_audio_s=audio_s, audio_s_per_s=audio_s / (med * 1e-3), **(extra or {})))
    return rows


class RnnRunner:
    """kws_deploy_forward(_lens) + kws_ctc_decode on device buffers, no host synchronisation."""

    def __init__(self, dm):
        from keyword_spotting_b200 import _lib
        from keyword_spotting_b200.utils import prediction
        self.dm, self.lib, self._lib, self.prediction = dm, dm._lib, _lib, prediction
        self.stream = torch.cuda.current_stream().cuda_stream

    def buffers(self, S, L):
        n, C = self.dm.num_frames(L), self.dm.config.num_classes
        st = torch.zeros((self.dm.config.num_layers, S, self.dm.config.hidden_size), device="cuda")
        return dict(probs=torch.empty((S, n, C), device="cuda"), st_in=st, st_out=torch.empty_like(st))

    def call(self, pcm, L, buf, lengths=None, nframes=None, use_lens=True):
        S, ld = pcm.shape[0], pcm.stride(0)
        args = (self.dm.handle, pcm.data_ptr(), self._lib.PCM_I16, S, L, ld)
        tail = (buf["st_in"].data_ptr(), buf["probs"].data_ptr(), buf["st_out"].data_ptr(), None, self.stream)
        if use_lens:
            self._lib.check(self.lib.kws_deploy_forward_lens(*args, None if lengths is None else lengths.data_ptr(), *tail))
        else:
            self._lib.check(self.lib.kws_deploy_forward(*args, *tail))
        self.prediction.decode_batch(buf["probs"], lens=nframes, want_labels=True)


def rnn_case(results, dm, S, repeats, iters, rng, label):
    run = RnnRunner(dm)
    L3 = 3 * SR
    samples = rng.integers(1 * SR, L3 + 1, S)
    samples[0] = L3
    pcm = torch.from_numpy(rng.integers(-3000, 3000, (S, L3), dtype=np.int16)).cuda()
    lengths = torch.from_numpy(samples.astype(np.int32)).cuda()
    nfr = torch.from_numpy(frames(samples).astype(np.int32)).cuda()
    buf = run.buffers(S, L3)
    groups = []
    for ln in np.unique(samples):
        idx = torch.from_numpy(np.flatnonzero(samples == ln)).cuda()
        groups.append((pcm[idx, :int(ln)].contiguous(), int(ln), run.buffers(len(idx), int(ln))))

    def per_length():
        for g, ln, b in groups:
            run.call(g, ln, b, use_lens=False)
    ms = time_variants({"deploy_forward_lens": lambda: run.call(pcm, L3, buf, lengths, nfr),
                        "padded deploy_forward (3 s)": lambda: run.call(pcm, L3, buf, use_lens=False),
                        "one deploy_forward per length": per_length}, repeats, iters)
    results["rows"] += summarize("1: rnn_ctc 1-3 s, %s" % label, ms, float(samples.sum()) / SR,
                                 dict(utterances=S, distinct_lengths=len(groups), pcm_MB=pcm.numel() * 2 / 1e6))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--utterances", type=int, default=4096)
    ap.add_argument("--full", type=int, default=32768)
    ap.add_argument("--att-utterances", type=int, default=1024)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None, help="write the results as JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pcm_lengths_bench needs a CUDA device")
    from keyword_spotting_b200 import AttentionDeployModel, DeployModel
    rng = np.random.default_rng(args.seed)
    results = dict(card=card(0), repeats=args.repeats, iters=args.iters, rows=[])
    dm = DeployModel(device=0)

    # ---- case 1: rnn_ctc, config-2 shape and the full GPU
    rnn_case(results, dm, args.utterances, args.repeats, args.iters, rng, "%d utterances" % args.utterances)
    torch.cuda.empty_cache()
    rnn_case(results, dm, args.full, 3, 1, rng, "%d utterances" % args.full)
    torch.cuda.empty_cache()

    # ---- case 2: attention from PCM, 1-8 s
    am = AttentionDeployModel(device=0)
    fe = am._frontend
    B, L8 = args.att_utterances, 8 * SR
    samples = rng.integers(1 * SR, L8 + 1, B)
    samples[0] = L8
    pcm = torch.from_numpy(rng.standard_normal((B, L8)).astype(np.float32) * 0.05).cuda()
    lengths = torch.from_numpy(samples.astype(np.int32)).cuda()
    lens = torch.from_numpy(frames(samples).astype(np.int32)).cuda()
    T = fe.num_frames(L8)
    mel = torch.empty((B, T, am.config.n_mel), device="cuda")
    probs = torch.empty((B, am.frames(T), am.config.num_classes), device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    from keyword_spotting_b200 import _lib

    def front(use_lens):
        _lib.check(fe._lib.kws_frontend_mel_lens(fe.handle, pcm.data_ptr(), _lib.PCM_F32, B, L8, L8,
                                                 lengths.data_ptr() if use_lens else None, mel.data_ptr(), stream))

    def att(use_lens):
        front(use_lens)
        _lib.check(am._lib.kws_attention_forward_lens(am._handle, mel.data_ptr(), B, T, lens.data_ptr(), probs.data_ptr(),
                                                      None, stream))
    ms = time_variants({"forward(lengths=), front end with lengths": lambda: att(True),
                        "earlier path, front end on the padded batch": lambda: att(False),
                        "front end with lengths alone": lambda: front(True),
                        "front end on the padded batch alone": lambda: front(False)}, args.repeats, args.iters)
    results["rows"] += summarize("2: attention 1-8 s", ms, float(samples.sum()) / SR,
                                 dict(utterances=B, pcm_MB=pcm.numel() * 4 / 1e6))

    # ---- case 3: equal lengths, NULL vs L
    run = RnnRunner(dm)
    S, L3 = args.utterances, 3 * SR
    pcm3 = torch.from_numpy(rng.integers(-3000, 3000, (S, L3), dtype=np.int16)).cuda()
    full3 = torch.full((S,), L3, dtype=torch.int32, device="cuda")
    buf = run.buffers(S, L3)
    ms = time_variants({"rnn_ctc lengths = NULL": lambda: run.call(pcm3, L3, buf),
                        "rnn_ctc lengths = L": lambda: run.call(pcm3, L3, buf, full3)}, args.repeats, args.iters)
    results["rows"] += summarize("3: rnn_ctc 3 s equal", ms, S * 3.0, dict(utterances=S))
    full8 = torch.full((B,), L8, dtype=torch.int32, device="cuda")
    T8 = torch.full((B,), T, dtype=torch.int32, device="cuda")

    def att_eq(use_lens):
        _lib.check(fe._lib.kws_frontend_mel_lens(fe.handle, pcm.data_ptr(), _lib.PCM_F32, B, L8, L8,
                                                 full8.data_ptr() if use_lens else None, mel.data_ptr(), stream))
        _lib.check(am._lib.kws_attention_forward_lens(am._handle, mel.data_ptr(), B, T, T8.data_ptr() if use_lens else None,
                                                      probs.data_ptr(), None, stream))
    ms = time_variants({"attention lengths = NULL": lambda: att_eq(False), "attention lengths = L": lambda: att_eq(True)},
                       args.repeats, args.iters)
    results["rows"] += summarize("3: attention 8 s equal", ms, B * 8.0, dict(utterances=B))

    print(json.dumps(results["card"]))
    print("| case | variant | ms / call (median, min-max) | valid audio-s/s |")
    print("|---|---|---|---|")
    for r in results["rows"]:
        print("| %s | %s | %.2f (%.2f-%.2f) | %.3g |" % (r["case"], r["variant"], r["ms_median"], r["ms_min"], r["ms_max"],
                                                        r["audio_s_per_s"]))
    for r in results["rows"]:
        print(json.dumps(r))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)
    am.close()
    dm.close()


if __name__ == "__main__":
    main()

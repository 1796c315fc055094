"""attention_ctc on variable-length batches: kws_attention_forward_lens against what a user can do without it.

Mel frames resident in HBM (larger than the 126 MB L2 at the default sizes), default config (BASELINE config 5), one
GPU.  Three cases, each variant warmed up, the variants of a case alternated in one process and repeated to show the
spread (CUDA events around --iters calls; median / min / max over --repeats):

  1  8 s utterances:                 kws_attention_forward  vs  kws_attention_forward_lens with every lens = T
  2  lengths uniform over 1-8 s:     forward_lens  vs  the equal-length forward padded to 8 s (wrong answers; the
                                     upper bound on work)  vs  one equal-length forward per distinct length
  3  as 2 with 2 % of the utterances at 10 s (T' = 501: the FFMA attention core)

Audio-s/s counts valid audio only: an utterance of L_b samples is L_b / 16000 s, T_b = 1 + (L_b - 400) // 160 frames.
The card's name and power limit are read in the same run.

    python tools/attention_lens_bench.py [--utterances 1024] [--repeats 5] [--iters 5] [--out results.json]
"""
import argparse
import json
import subprocess
import sys
import os

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
    return 1 + (samples - FFT) // HOP


class Runner:
    def __init__(self, am):
        from keyword_spotting_b200 import _lib
        self.am, self.lib, self._lib = am, am._lib, _lib
        self.stream = torch.cuda.current_stream().cuda_stream
        self.C = am.config.num_classes

    def out(self, B, T):
        return torch.empty((B, self.am.frames(T), self.C), device="cuda")

    def forward(self, mel, probs):
        B, T, _ = mel.shape
        self._lib.check(self.lib.kws_attention_forward(self.am._handle, mel.data_ptr(), B, T, probs.data_ptr(), None,
                                                       self.stream))

    def forward_lens(self, mel, lens, probs):
        B, T, _ = mel.shape
        self._lib.check(self.lib.kws_attention_forward_lens(self.am._handle, mel.data_ptr(), B, T,
                                                            None if lens is None else lens.data_ptr(), probs.data_ptr(),
                                                            None, self.stream))


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


def grouped(run, mel_host_lens, mel):
    """One equal-length forward per distinct length: utterances gathered by length beforehand (not timed)."""
    lens = mel_host_lens
    groups = []
    for t in np.unique(lens):
        idx = torch.from_numpy(np.flatnonzero(lens == t)).cuda()
        g = mel[idx, :int(t)].contiguous()
        groups.append((g, run.out(len(idx), int(t))))

    def fn():
        for g, p in groups:
            run.forward(g, p)
    return fn, len(groups)


def summarize(case, ms, audio_s, extra=None):
    rows = []
    for name, v in ms.items():
        med = float(np.median(v))
        rows.append(dict(case=case, variant=name, ms_median=med, ms_min=float(min(v)), ms_max=float(max(v)),
                         valid_audio_s=audio_s, audio_s_per_s=audio_s / (med * 1e-3), **(extra or {})))
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--utterances", type=int, default=1024)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None, help="write the results as JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attention_lens_bench needs a CUDA device")
    from keyword_spotting_b200 import AttentionConfig, AttentionDeployModel
    am = AttentionDeployModel(AttentionConfig(), device=0)
    run = Runner(am)
    B, M = args.utterances, am.config.n_mel
    rng = np.random.default_rng(args.seed)
    g = torch.Generator(device="cuda").manual_seed(args.seed)
    results = dict(card=card(0), utterances=B, repeats=args.repeats, iters=args.iters, rows=[])

    # ---- case 1: 8 s utterances, lens = NULL path vs lens = T
    L8 = 8 * SR
    T8 = frames(L8)
    mel8 = torch.rand((B, T8, M), device="cuda", generator=g) * 3.0
    p8 = run.out(B, T8)
    full = torch.full((B,), T8, dtype=torch.int32, device="cuda")
    ms = time_variants({"forward": lambda: run.forward(mel8, p8), "forward_lens(lens=T)": lambda: run.forward_lens(mel8, full, p8)},
                       args.repeats, args.iters)
    results["rows"] += summarize("1: 8 s", ms, B * L8 / SR, dict(mel_MB=mel8.numel() * 4 / 1e6))
    del mel8, p8

    # ---- cases 2 and 3: lengths uniform over 1-8 s, then 2 % of them at 10 s
    for case, n10 in (("2: 1-8 s", 0), ("3: 1-8 s + 2 % at 10 s", max(1, round(0.02 * B)))):
        samples = rng.integers(1 * SR, L8 + 1, B)
        if n10:
            samples[rng.choice(B, n10, replace=False)] = FFT + (1000 - 1) * HOP       # 1000 frames: T' = 501
        lens_h = frames(samples).astype(np.int32)
        T = int(lens_h.max())
        mel = torch.rand((B, T, M), device="cuda", generator=g) * 3.0
        lens = torch.from_numpy(lens_h).cuda()
        probs = run.out(B, T)
        gfn, ngroups = grouped(run, lens_h, mel)
        ms = time_variants({"forward_lens": lambda: run.forward_lens(mel, lens, probs),
                            "padded forward (wrong answers)": lambda: run.forward(mel, probs),
                            "one forward per length": gfn}, args.repeats, args.iters)
        Tp = np.where(lens_h > 0, lens_h // 2 + 1, 0)
        extra = dict(T=T, distinct_lengths=ngroups, mel_MB=mel.numel() * 4 / 1e6,
                     valid_row_share=float(Tp.sum() / (B * am.frames(T))),
                     core_work_share=float((Tp.astype(np.float64) ** 2).sum() / (B * am.frames(T) ** 2)))
        results["rows"] += summarize(case, ms, float(samples.sum()) / SR, extra)
        del mel, probs, gfn
        torch.cuda.empty_cache()

    print(json.dumps(results["card"]))
    print("| case | variant | ms / call (median, min-max) | valid audio-s/s | vs padded |")
    print("|---|---|---|---|---|")
    for r in results["rows"]:
        pad = [q for q in results["rows"] if q["case"] == r["case"] and q["variant"].startswith("padded")]
        rel = "%.2fx" % (r["ms_median"] / pad[0]["ms_median"]) if pad else ""
        print("| %s | %s | %.2f (%.2f-%.2f) | %.3g | %s |" % (r["case"], r["variant"], r["ms_median"], r["ms_min"],
                                                               r["ms_max"], r["audio_s_per_s"], rel))
    for r in results["rows"]:
        print(json.dumps(r))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)
    am.close()


if __name__ == "__main__":
    main()

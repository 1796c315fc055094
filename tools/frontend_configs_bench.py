"""Speed of models with analysis frames other than 400/160 (the general DFT front end, csrc/frontend_dft.cu).

On one GPU, with the card's name and power limit read in the same run:
  * the streaming step of 131,072 streams on 4,800-sample chunks, device-resident PCM (1.26 GB of chunks, rotated: more
    than L2), per part with kws_debug_step_timing (front end incl. pre-step | GRU | decode), and end to end from pinned
    host memory (kws_stream_step_host);
  * kws_frontend_mel on 4,096 x 3 s of int16 PCM (393 MB), with the default 400/160 FFT front end as the reference line;
  * the DFT kernel's share of the tensor bound: its three fp16 products (x_hi W_hi + x_lo W_hi + x_hi W_lo) at the
    data-sheet 2,250 TFLOP/s dense fp16 of a 1,000 W B200, over the measured front-end time.
Configurations alternate inside every repeat; medians are reported.  Prints one JSON document (and writes it to --out).

    python tools/frontend_configs_bench.py [--streams 131072] [--out results.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

CONFIGS = [(512, 160), (320, 160), (200, 80)]
PEAK_FP16 = 2250e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def dft_flops_per_frame(fft):
    hc = (fft + 1) // 2
    b = (hc + 15) // 16 * 16
    ncols = (b + hc + 15) // 16 * 16
    kpad = (fft + 31) // 32 * 32
    return 3 * 2 * ncols * kpad


def model(fft, hop, n_mel=40):
    from keyword_spotting_b200 import Config, DeployModel, ModelWeights
    cfg = Config(n_mel=n_mel, fft_size=fft, hop_size=hop)
    return DeployModel(cfg, ModelWeights.random_init(cfg), precision="tc")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=131072)
    ap.add_argument("--chunk", type=int, default=4800)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--mel-rows", type=int, default=4096)
    ap.add_argument("--mel-len", type=int, default=48000)
    ap.add_argument("--out", default=None, help="write the results as JSON here")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("frontend_configs_bench needs a CUDA device")
    from keyword_spotting_b200 import StreamingDetector, _lib
    lib = _lib.load()
    res = {"card": card(), "streams": a.streams, "chunk": a.chunk, "configs": {}}
    S, n = a.streams, a.chunk
    g = torch.Generator(device="cuda").manual_seed(1)
    chunks = [torch.randint(-3000, 3000, (S, n), dtype=torch.int16, device="cuda", generator=g) for _ in range(2)]
    pinned = chunks[0].cpu().pin_memory()
    mel_pcm = torch.randint(-3000, 3000, (a.mel_rows, a.mel_len), dtype=torch.int16, device="cuda", generator=g)
    st = torch.cuda.current_stream().cuda_stream
    models = {c: model(*c) for c in CONFIGS + [(400, 160)]}
    dets = {c: StreamingDetector(models[c], S) for c in CONFIGS}
    mels = {c: torch.empty((a.mel_rows, models[c].num_frames(a.mel_len), 40), dtype=torch.float32, device="cuda")
            for c in models}
    samples = {c: {"step": [], "parts": [], "e2e": [], "mel": []} for c in models}

    def run_mel(c, reps):
        m = models[c]
        for _ in range(reps):
            _lib.check(lib.kws_frontend_mel(m.handle, mel_pcm.data_ptr(), _lib.PCM_I16, a.mel_rows, a.mel_len,
                                            a.mel_len, mels[c].data_ptr(), st))

    for c in CONFIGS:                                 # warm every shape the timed windows use
        dets[c].step(chunks[0])
        dets[c].step_host(pinned)
    for c in models:
        run_mel(c, 2)
    torch.cuda.synchronize()
    for rep in range(a.repeats):
        for c in CONFIGS:
            d = dets[c]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(a.steps):
                d.step(chunks[i & 1])
            torch.cuda.synchronize()
            samples[c]["step"].append((time.perf_counter() - t0) * 1e3 / a.steps)
            lib.kws_debug_step_timing(1, None, None)
            for i in range(a.steps):
                d.step(chunks[i & 1])
            part = (ctypes.c_double * 3)()
            cnt = ctypes.c_longlong()
            lib.kws_debug_step_timing(0, part, ctypes.byref(cnt))
            samples[c]["parts"].append([p / max(1, cnt.value) for p in part])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(a.steps):
                d.step_host(pinned)
            torch.cuda.synchronize()
            samples[c]["e2e"].append((time.perf_counter() - t0) * 1e3 / a.steps)
        for c in models:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run_mel(c, a.steps)
            e1.record()
            torch.cuda.synchronize()
            samples[c]["mel"].append(e0.elapsed_time(e1) / a.steps)
    audio_s = S * n / 16000.0
    for c in models:
        fft, hop = c
        sm = samples[c]
        out = {"mel_ms": float(np.median(sm["mel"])), "mel_rows": a.mel_rows, "mel_len": a.mel_len}
        frames = a.mel_rows * models[c].num_frames(a.mel_len)
        if c != (400, 160):
            bound = frames * dft_flops_per_frame(fft) / PEAK_FP16 * 1e3
            out["mel_tensor_bound_ms"] = bound
            out["mel_share_of_tensor_bound"] = bound / out["mel_ms"]
            step = float(np.median(sm["step"]))
            parts = np.median(np.array(sm["parts"]), axis=0).tolist()
            fr_step = S * max(0, 1 + (n + (fft - hop) - fft) // hop)
            out.update(step_ms=step, parts_ms=dict(frontend=parts[0], gru=parts[1], decode=parts[2]),
                       step_audio_s_per_s=audio_s / (step * 1e-3),
                       e2e_ms=float(np.median(sm["e2e"])), e2e_audio_s_per_s=audio_s / (np.median(sm["e2e"]) * 1e-3),
                       frontend_tensor_bound_ms=fr_step * dft_flops_per_frame(fft) / PEAK_FP16 * 1e3,
                       host_link_bytes_per_step=S * n * 2)
        res["configs"]["%d/%d" % c] = out
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    for d in dets.values():
        d.close()
    for m in models.values():
        m.close()


if __name__ == "__main__":
    main()

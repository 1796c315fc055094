#!/usr/bin/env python
"""Headline benchmark: streamed audio-seconds per second of the 2-layer GRU-128 KWS path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): streaming serve of
S = 131,072 concurrent streams PER GPU with carried GRU state and VAD reset, 300 ms chunks of
synthetic 16 kHz int16 audio, random-init weights.  One "step" = one 300 ms chunk for every stream:
VAD -> tail carry -> framing/|rFFT|/mel -> 2x GRU(128) -> FC -> softmax -> window decode -> trigger.
Streams are independent, so N GPUs hold N*S streams with no collective on the hot path (weak scaling);
NCCL is used only for the max-over-ranks of the device time and the final trigger-count gather.

One JSON line on rank 0: `value` = whole-job audio-s/s with the chunk already resident in HBM,
`e2e` = the same through the wave server of the package (kws_server_*: pinned host PCM -> H2D -> step -> D2H
triggers, one CUDA-graph launch per wave and chunk, copies inside the timed region) next to the `copy_ceiling` of
the same buffers / streams / schedule with no kernels, `roofline` for the dominant kernel, `parity_check` = a sample
of the very streams being benchmarked held against the CPU oracle before the timed region, `ops` = BASELINE
configs[1], [3], [4] and the custom ops timed next to their CPU baselines (N=1 only), `cpu_baseline` = the CPU oracle
port timed on this box's host cores on a bounded sample.  `--impl reference` times that CPU port alone.

The FC layer of the random-init model is scaled by --fc-gain (3) and the keyword is --keyword ("1"): with the
reference's own initialisation no posterior ever crosses the 0.4 decode threshold and "1233" never fires, so the
emit / trigger / window-clear / state-reset branches would never execute inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CHUNK = 4800                      # 300 ms at 16 kHz (README.md:88, detector.py:150)
FRAMES = 30                       # steady state: 320 carried + 4800 new samples -> 30 frames
AUDIO_S_PER_CHUNK = CHUNK / 16000.0
METRIC = "streamed audio-sec/sec, 2L GRU-128 KWS"
UNIT = "audio-s/s"
# algorithmic work (SURVEY.md 8d): GRU 325,632 + FC 1,536 FLOP per frame
GRU_FLOP_PER_FRAME = 2 * (40 * 384 + 128 * 384 + 128 * 384 + 128 * 384) + 2 * 128 * 6
# front-end kernel, compulsory bytes per stream-chunk: 4800 int16 in, carried tail 320 samples read + written,
# 30 x 40 fp32 mel out, VAD flag + frame count + tail length
FE_BYTES_PER_STREAM_CHUNK = CHUNK * 2 + 2 * 320 * 2 + FRAMES * 40 * 4 + 9
# decode kernel (K4): 30 x 6 fp32 probabilities read, 30 tokens written, the 15 x 32 B token window re-read, slot frame
# counts (15), window head / size r+w (16), VAD flag, frame count, 2 trigger words
POST_BYTES_PER_STREAM_CHUNK = FRAMES * 6 * 4 + FRAMES + 15 * 32 + 15 + 16 + 1 + 4 + 8


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=131072, help="concurrent streams per GPU")
    ap.add_argument("--precision", default="tc", choices=["tc", "fp32"],
                    help="recurrent kernel: tc = tcgen05 fp16 operands / fp32 accumulate (default), fp32 = exact FFMA path")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--waves", type=int, default=32, help="e2e: the streams of a GPU are served in this many waves "
                    "(independent stream objects on their own CUDA streams) so copies overlap compute and a chunk's "
                    "latency is one wave's, not the whole batch's")
    ap.add_argument("--depth", type=int, default=2, help="e2e: waves in flight")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-ops", action="store_true", help="skip the `ops` block (configs 2/4/5 + custom ops, N=1 only)")
    ap.add_argument("--no-parity", action="store_true", help="skip the `parity_check` block")
    ap.add_argument("--no-graphs", action="store_true", help="e2e: enqueue copies and kernels directly instead of graph replay")
    ap.add_argument("--workload", default="streaming", choices=["streaming", "attention"],
                    help="streaming = BASELINE configs[2] (the headline, default); attention = configs[4]: attention_ctc, "
                         "n_mel 60, batched 8 s utterances sharded by utterance over the GPUs (no collective)")
    ap.add_argument("--utterances", type=int, default=512, help="--workload attention: 8 s utterances per GPU and step")
    ap.add_argument("--frontend", default="fft", choices=["fft", "tc"],
                    help="front-end formulation: fft = packed-real FFT on the CUDA cores (default), tc = hop-block DFTs on tcgen05")
    ap.add_argument("--fc-gain", type=float, default=3.0, help="scale of the random-init FC layer (see the docstring)")
    ap.add_argument("--keyword", default="1", help="keyword of the trigger test (reference default '1233')")
    ap.add_argument("--parity-streams", type=int, default=256)
    ap.add_argument("--parity-chunks", type=int, default=4)
    ap.add_argument("--no-bind", action="store_true", help="do not pin the rank to its GPU's NUMA-local cores")
    ap.add_argument("--cpu-streams", type=int, default=0, help="CPU sample: streams (default 64 per host core)")
    ap.add_argument("--cpu-chunks", type=int, default=0, help="CPU sample: chunks per step (default: calibrated)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (rank 0) as DIR/<name>.npy, "
                         "float32 / float64, at most 64 MB: streaming = the trigger flags of every stream and, for a fixed "
                         "seeded sample of streams, the carried GRU state and the window labels; attention = the softmax "
                         "of a fixed seeded sample of utterances (all of them up to 4096)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; --impl reference has none")
    return args


# ----------------------------------------------------------------------------- CPU port (oracle)
def _cpu_worker(args):
    """One process = one host core: the detector loop of the oracle for a block of streams."""
    seed, n_streams, n_chunks = args
    os.environ["OMP_NUM_THREADS"] = "1"
    try:
        from threadpoolctl import threadpool_limits
        limiter = threadpool_limits(limits=1)
    except Exception:       # pragma: no cover
        limiter = None
    import numpy as np
    from oracle import model as om, streaming as ost
    w = om.init_weights(seed=1234, n_mel=40)
    rng = np.random.default_rng(seed)
    pcm = np.clip(np.rint(rng.standard_normal((n_streams, CHUNK * (n_chunks + 1))) * 600), -32768, 32767).astype(np.int16)
    orc = ost.StreamOracle(w, n_streams)
    orc.step(pcm[:, :CHUNK])                        # warm-up chunk (fills the tail: steady state)
    t0 = time.perf_counter()
    trig = 0
    for c in range(1, n_chunks + 1):
        trig += int(orc.step(pcm[:, c * CHUNK:(c + 1) * CHUNK])["trigger"].sum())
    dt = time.perf_counter() - t0
    del limiter
    return dt, trig


def cpu_port_throughput(total_streams, n_chunks, procs=None):
    """audio-s/s of the oracle port using `procs` single-threaded processes over disjoint streams."""
    import multiprocessing as mp
    procs = procs or (os.cpu_count() or 1)
    procs = max(1, min(procs, total_streams))
    per = max(1, total_streams // procs)
    jobs = [(1000 + i, per, n_chunks) for i in range(procs)]
    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    with ctx.Pool(procs) as pool:
        res = pool.map(_cpu_worker, jobs)
    wall = time.perf_counter() - t0
    slowest = max(r[0] for r in res)                # the processes run concurrently
    audio = per * procs * n_chunks * AUDIO_S_PER_CHUNK
    return dict(value=audio / slowest, unit=UNIT, cores=procs, kind="port",
                sample="%d streams x %d chunks of 300 ms through the numpy oracle (detector loop), %d single-thread "
                       "processes; %.1f s wall incl. start-up" % (per * procs, n_chunks, procs, wall))


def cpu_sample_size(args, budget_s):
    """Pick the bounded CPU sample: 64 streams per core (the port is fastest around there); chunk count calibrated to ~budget_s per sample."""
    cores = os.cpu_count() or 1
    streams = args.cpu_streams or 64 * cores
    if args.cpu_chunks:
        return streams, args.cpu_chunks
    probe = cpu_port_throughput(streams, 2)
    t_chunk = streams * AUDIO_S_PER_CHUNK / probe["value"]
    return streams, int(max(2, min(400, budget_s / max(t_chunk, 1e-3))))


def run_reference_arm(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path.  TensorFlow/librosa are not
    installable here, so this is the oracle port (kind 'port') on all host cores."""
    if rank != 0:
        return
    streams, chunks = cpu_sample_size(args, budget_s=150.0 / max(1, args.warmup + args.steps))
    vals = []
    info = None
    for i in range(args.warmup + args.steps):       # every step = one bounded sample of the workload
        info = cpu_port_throughput(streams, chunks)
        if i >= args.warmup:
            vals.append(info["value"])
    value = statistics.median(vals)
    info["value"] = value
    args.cpu_streams, args.cpu_chunks = streams, chunks
    per_step_audio = args.cpu_streams * args.cpu_chunks * AUDIO_S_PER_CHUNK
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=len(vals), warmup=args.warmup,
                ms_per_step=1e3 * per_step_audio / value, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="f32", data="synthetic", impl="reference",
                config=dict(workload="streaming serve (BASELINE configs[2]): concurrent streams with carried GRU state and "
                                     "VAD reset, 300 ms chunks; bounded CPU sample", streams_per_step=args.cpu_streams,
                            chunk_samples=CHUNK),
                cpu_baseline=info,
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, power, reasons = [], [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    power_w_max=max(power) if power else None, samples=len(sm), reasons=sorted(reasons))


# ----------------------------------------------------------------------------- ours
def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=float(d["hbm_gbs"]), bf16=float(d["bf16_tflops"]), bf16_sustained=float(d["bf16_tflops_sustained"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def load_traffic(S):
    """Per-launch DRAM traffic (dram__bytes_read.sum + dram__bytes_write.sum) from the committed ncu --set full
    capture, scaled from the captured stream count to S; None when the capture file is absent."""
    path = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(path):
        return {}
    d = json.load(open(path))
    k = S / float(d["streams"])
    out = {name: (v["dram_bytes_read"] + v["dram_bytes_write"]) * k for name, v in d["kernels"].items()}
    out["_source"] = d["source"]
    return out


def make_chunks(torch, S, n_buf, device, seed):
    """n_buf distinct [S, 4800] int16 chunks on the device: per-stream noise level log-uniform in [30, 3000] LSB,
    ~30% of (stream, chunk) cells near-silent so the VAD reset fires (SURVEY.md 8d)."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    bufs = []
    for b in range(n_buf):
        sigma = torch.exp(torch.empty((S, 1), device=device).uniform_(3.4, 8.0, generator=g))
        x = torch.randn((S, CHUNK), device=device, generator=g) * sigma
        silent = torch.rand((S, 1), device=device, generator=g) < 0.3
        x = torch.where(silent, torch.randint(-2, 3, (S, CHUNK), device=device, generator=g).float(), x)
        bufs.append(x.clamp_(-32768, 32767).round_().to(torch.int16).contiguous())
        del x
    return bufs


def timed_loop(torch, fn, steps, stream, barrier):
    """EXACTLY `steps` calls bracketed by barrier + synchronize; device time via CUDA events on `stream`."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    barrier()
    torch.cuda.synchronize()
    ev[0].record(stream)
    for i in range(steps):
        fn(i)
        ev[i + 1].record(stream)
    torch.cuda.synchronize()
    barrier()
    per_step = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
    return ev[0].elapsed_time(ev[steps]), per_step


# ----------------------------------------------------------------------------- --dump-outputs
DUMP_LIMIT_BYTES = 64 << 20
DUMP_SAMPLE_STREAMS = 8192        # state 8 MB + labels 2 MB; the trigger flags of 6.9 M streams (the HBM limit) add 28 MB
DUMP_SAMPLE_UTTERANCES = 4096     # softmax [4096, 400, 6] fp32 = 39 MB


def dump_sample(n, limit, seed=2024):
    """Sorted indices of a fixed, seeded sample of min(n, limit) out of n items (all of them when n <= limit)."""
    import numpy as np
    if n <= limit:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, limit, replace=False))


def stream_outputs(torch, det, trig):
    """What the last kws_stream_step left for its caller: the trigger flags of every stream and, for a fixed seeded
    sample of streams, the carried GRU state and the labels of the decode window (max 64 entries, -1 padded)."""
    import numpy as np
    sample = dump_sample(det.n_streams, DUMP_SAMPLE_STREAMS)
    idx = torch.from_numpy(sample).to(trig.device)
    labels, counts = det.window_labels(max_labels=64)
    return dict(triggers=trig.cpu().numpy().astype(np.float32), sample_streams=sample.astype(np.float64),
                state=det.state()[:, idx].cpu().numpy(), window_labels=labels[sample].astype(np.float32),
                window_label_counts=counts[sample].astype(np.float32))


def write_outputs(out_dir, arrays):
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def boosted_weights(cfg, gain, seed=1234):
    """Random-init weights of the reference architecture with the FC layer scaled by `gain` (module docstring)."""
    import numpy as np
    from keyword_spotting_b200 import ModelWeights
    w = ModelWeights.random_init(cfg, seed=seed)
    w.fc_w = (w.fc_w * np.float32(gain)).astype(np.float32)
    return w


def parity_check(args, torch, model, weights, det, chunks, S):
    """A sample of the benchmarked streams (first tile, beyond 65,536, last tile, random) through `parity-chunks`
    chunks of the benchmark's own PCM, held against the CPU oracle's detector loop -- the CHECKER, outside every
    timed region.  Probabilities / state: max-abs against the contract (1e-3).  Triggers and window labels: must
    be bit-identical once the frames whose decision lies within 1e-3 of a threshold (oracle.streaming.
    ambiguous_frames) are taken from the GPU; `trigger_mismatches` / `label_mismatches` count violations."""
    import numpy as np
    from oracle import model as om, streaming as ost
    P = max(8, min(args.parity_streams, S))
    rng = np.random.default_rng(99)
    q = P // 4
    parts = [np.arange(0, min(q, S))]
    if S > 65536 + q:
        parts.append(np.arange(65536, 65536 + q))
    parts.append(np.arange(max(0, S - q), S))
    fixed = np.unique(np.concatenate(parts))
    rest = np.setdiff1d(np.arange(S), fixed)
    extra = rng.choice(rest, max(0, min(len(rest), P - len(fixed))), replace=False) if len(rest) else np.zeros(0, np.int64)
    sample = np.sort(np.concatenate([fixed, extra])).astype(np.int64)
    sample_d = torch.from_numpy(sample).to(chunks[0].device)
    ow = om.Weights(mel_basis=weights.mel_basis, gates_kernel=list(weights.gates_kernel), gates_bias=list(weights.gates_bias),
                    cand_kernel=list(weights.cand_kernel), cand_bias=list(weights.cand_bias), fc_w=weights.fc_w, fc_b=weights.fc_b)
    orc = ost.StreamOracle(ow, len(sample), label=args.keyword)
    tol, thres = 1e-3, 0.4
    det.reset()
    worst_p = worst_s = 0.0
    trig_bad = lab_bad = n_trig = n_trig_all = n_amb = n_frames = n_silent = n_labels = 0
    for c in range(args.parity_chunks):
        x = chunks[c % len(chunks)]
        trig, probs, nfr = det.step(x, want_probs=True)
        state = det.state()[:, sample_d].cpu().numpy()
        labels, counts = [a for a in det.window_labels(max_labels=64)]
        labels, counts = labels[sample], counts[sample]
        gp = probs[sample_d].cpu().numpy()
        gt = trig[sample_d].cpu().numpy()
        n_trig_all += int(trig.sum())

        def decide(sm):
            nonlocal n_amb, n_frames
            amb = ost.ambiguous_frames(sm, thres, tol)
            n_amb += int(amb.sum())
            n_frames += amb.size
            out = sm.copy()
            out[amb] = gp[:, :sm.shape[1]][amb]
            return out

        want = orc.step(x[sample_d].cpu().numpy(), decide_on=decide)
        n = want["softmax"].shape[1]
        worst_p = max(worst_p, float(np.abs(gp[:, :n] - want["softmax"]).max()))
        worst_s = max(worst_s, float(np.abs(state - want["state"]).max()))
        trig_bad += int((gt != want["trigger"]).sum())
        n_trig += int(want["trigger"].sum())
        n_silent += int((~want["speech"]).sum())
        for i in range(len(sample)):
            wl = want["labels"][i] if not want["trigger"][i] else np.zeros(1, np.int32)
            n_labels += len(wl) // 2
            k = min(len(wl), 64)
            if counts[i] != len(wl) or not np.array_equal(labels[i, :k], wl[:k]):
                lab_bad += 1
        del probs, trig
    det.reset()
    return dict(streams_sampled=int(len(sample)), sampled_beyond_65536=int((sample >= 65536).sum()), chunks=args.parity_chunks,
                oracle="oracle.streaming.StreamOracle (numpy fp32 detector loop) on the same PCM and weights",
                max_abs_probs=worst_p, max_abs_state=worst_s, tolerance=tol,
                within_tolerance=bool(worst_p < tol and worst_s < tol),
                trigger_mismatches=trig_bad, label_mismatches=lab_bad, triggers_in_sample=n_trig, labels_in_sample=n_labels,
                vad_resets_in_sample=n_silent, triggers_all_streams=n_trig_all,
                ambiguous_frames=n_amb, frames=n_frames,
                rule="triggers / window labels bit-identical to the fp32 oracle, frames whose winner is within 1e-3 of the "
                     "threshold (or whose runner-up is within 2e-3 of an above-threshold winner) taken from the GPU")


def ops_block(args, torch, device, peaks):
    """BASELINE configs[1] (offline 4096 x 3 s), [3] (octbit op at the model's shapes), [4] (attention_ctc, 8 s
    utterances) and the custom ops, each timed on the device with CUDA events next to its CPU baseline on a bounded
    sample: the UNMODIFIED reference kernels from oracle/_ref (single thread, as the reference runs them) for octbit
    and posenc, the numpy oracle port for the model graphs.  Also measures the int8 tensor peak (torch._int_mm,
    i.e. cuBLASLt) that the octbit tensor-core kernel is held against.  N=1 only."""
    import numpy as np
    from keyword_spotting_b200 import AttentionConfig, AttentionDeployModel, Config, DeployModel, ModelWeights
    from keyword_spotting_b200.octbit.octbit_graph import octize_weight_int8_signed
    from keyword_spotting_b200.octbit.octbit_ops import octbit_mat_mul
    from keyword_spotting_b200.positional_encoding.positional_encoding_op import positional_encoding
    from keyword_spotting_b200.utils import prediction
    from keyword_spotting_b200.rnn_ctc import INITIAL_STATES, INPUT_X, RNN_STATES, SOFTMAX

    def timeit(fn, iters=5, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    def cpu_time(fn, min_s=1.0):
        fn()
        n, t0 = 0, time.perf_counter()
        while True:
            fn()
            n += 1
            dt = time.perf_counter() - t0
            if dt >= min_s:
                return dt / n

    out = {}
    sampler = ClockSampler(device.index)
    sampler.start()
    g = torch.Generator(device=device).manual_seed(1)
    # ---- int8 tensor peak of this box (denominator of the octbit tensor-core kernel)
    try:
        n8 = 8192
        a8 = torch.randint(-128, 127, (n8, n8), device=device, dtype=torch.int8, generator=g)
        b8 = torch.randint(-128, 127, (n8, n8), device=device, dtype=torch.int8, generator=g)
        ms = timeit(lambda: torch._int_mm(a8, b8), iters=10, warm=3)
        int8_peak = 2.0 * n8 ** 3 / ms / 1e9
        out["int8_tensor_peak"] = dict(TOPs=int8_peak, how="torch._int_mm (cuBLASLt) 8192^3, mean of 10 back to back")
        del a8, b8
    except Exception as exc:        # pragma: no cover
        int8_peak = None
        out["int8_tensor_peak"] = dict(TOPs=None, how="torch._int_mm failed: %r" % (exc,))
    # ---- octbit: the three converted matmuls of the rnn_ctc graph (main.py:357-360) at A = 131072 streams x 30 frames
    from oracle import cref, octbit as ooct
    A = 131072 * 30
    rng = np.random.default_rng(0)
    for K, B in ((256, 256), (256, 128), (128, 6)):
        x = torch.randn((A, K), device=device, generator=g)
        wf = torch.randn((K, B), device=device, generator=g) * (2.0 / (K + B)) ** 0.5
        w, scale, bias = octize_weight_int8_signed(wf)
        ms = timeit(lambda: octbit_mat_mul(x, w, scale=scale, bias=bias), iters=5)
        nbytes = A * K * 4 + B * K + A * B * 4
        rec = dict(ms=ms, algorithmic_GBps=nbytes / ms / 1e6, hbm_frac=nbytes / ms / 1e6 / peaks["hbm"],
                   int8_TOPs=2.0 * A * B * K / ms / 1e9, rows_per_s=A / ms * 1e3)
        if int8_peak:
            rec["int8_frac"] = rec["int8_TOPs"] / int8_peak
        if cref.have_ref():
            Ac = 4096
            xc = x[:Ac].cpu().numpy()
            wc = (w.cpu().numpy() if isinstance(w, torch.Tensor) else np.asarray(w)).astype(np.int8)
            bc = (bias.cpu().numpy() if isinstance(bias, torch.Tensor) else np.asarray(bias)).astype(np.float32)
            t = cpu_time(lambda: cref.ref_octbit_matmul(xc, wc, bc, float(scale)))
            rec["cpu_baseline"] = dict(rows_per_s=Ac / t, kind="reference", cores=1,
                                       sample="%d rows through the unmodified octbit_mat_mul_op.cc (oracle/_ref, -O2 -msse4.1, "
                                              "single thread as the reference runs it)" % Ac)
            rec["speedup_vs_cpu"] = rec["rows_per_s"] / rec["cpu_baseline"]["rows_per_s"]
        out["octbit_A%d_K%d_B%d" % (A, K, B)] = rec
        del x
    # ---- posenc
    for T, N in ((400, 128), (65536, 512)):
        ms = timeit(lambda: positional_encoding(T, N), iters=20)
        rec = dict(ms=ms, GBps=T * N * 4 / ms / 1e6)
        if cref.have_ref():
            t = cpu_time(lambda: cref.ref_positional_encoding(T, N), min_s=0.5)
            rec["cpu_baseline"] = dict(ms=t * 1e3, kind="reference", cores=1,
                                       sample="the unmodified positional_encoding_op.cc (libm double sin/cos/pow), single thread")
            rec["speedup_vs_cpu"] = t * 1e3 / ms
        out["posenc_%dx%d" % (T, N)] = rec
    # ---- batch decode
    for S_, T in ((4096, 298), (131072, 450)):
        p_ = torch.rand((S_, T, 6), device=device, generator=g)
        p_ = p_ / p_.sum(-1, keepdim=True)
        for name, mode in (("ctc_decode", prediction.MODE_CTC_DECODE), ("ctc_decode2", prediction.MODE_CTC_DECODE2)):
            ms = timeit(lambda: prediction.decode_batch(p_, mode=mode, want_labels=False), iters=5)
            out["%s_%dx%d" % (name, S_, T)] = dict(ms=ms, GBps=S_ * T * 6 * 4 / ms / 1e6, hbm_frac=S_ * T * 6 * 4 / ms / 1e6 / peaks["hbm"])
        del p_
    # ---- BASELINE configs[1]: 4096 utterances x 3 s of int16 PCM in HBM -> labels + trigger (main.py:263-314)
    cfg = Config(n_mel=40)
    wts = ModelWeights.random_init(cfg, seed=1234)
    dm = DeployModel(cfg, wts, device=device)
    # ---- the two front-end formulations side by side: 131,072 streams x one steady-state chunk (5120 samples, 30 frames)
    pcm_fe = (torch.randn((131072, 5120), device=device, generator=g) * 800).clamp_(-32768, 32767).to(torch.int16)
    fe = {}
    for name in ("fft", "tc"):
        dm.set_frontend(name)
        fe[name + "_ms"] = timeit(lambda: dm.frontend(pcm_fe), iters=5)
    dm.set_frontend("fft")
    fe["workload"] = "kws_frontend_mel, 131072 x 5120 int16 samples -> [131072, 30, 40] mel (row-major, no fused pre-step)"
    out["frontend_fft_vs_tc"] = fe
    del pcm_fe
    S2 = 4096
    pcm16 = (torch.randn((S2, 48000), device=device, generator=g) * 800).clamp_(-32768, 32767).to(torch.int16)
    st0 = torch.zeros((2, S2, 128), device=device)

    def offline():
        probs, _ = dm.run([SOFTMAX, RNN_STATES], {INPUT_X: pcm16, INITIAL_STATES: st0})
        return prediction.decode_batch(probs, mode=prediction.MODE_CTC_DECODE, want_labels=True)

    ms = timeit(offline, iters=5)
    rec = dict(ms=ms, utterances_per_s=S2 / ms * 1e3, audio_s_per_s=3.0 * S2 / ms * 1e3,
               workload="configs[1]: 4096 x 3 s int16 PCM resident in HBM -> mel -> 2L GRU-128 -> softmax (298 frames) -> ctc_decode labels + trigger")
    from oracle import model as om, prediction as oprd
    ow = om.Weights(mel_basis=wts.mel_basis, gates_kernel=wts.gates_kernel, gates_bias=wts.gates_bias, cand_kernel=wts.cand_kernel,
                    cand_bias=wts.cand_bias, fc_w=wts.fc_w, fc_b=wts.fc_b)
    nb = 32
    pc = om.pcm16_to_float(pcm16[:nb].cpu().numpy())

    def offline_cpu():
        pr, _, _ = om.deploy_forward(pc, np.zeros((2, nb, 128), np.float32), ow)
        return [oprd.ctc_decode(pr[i]) for i in range(nb)]

    t = cpu_time(offline_cpu, min_s=2.0)
    rec["cpu_baseline"] = dict(utterances_per_s=nb / t, kind="port", cores="numpy default threads of %d" % (os.cpu_count() or 1),
                               sample="%d utterances x 3 s through the numpy oracle (batch forward + ctc_decode)" % nb)
    rec["speedup_vs_cpu"] = rec["utterances_per_s"] / rec["cpu_baseline"]["utterances_per_s"]
    out["offline_config2_S4096_3s"] = rec
    del pcm16, st0
    # ---- BASELINE configs[3] as a model: the octbit-rewritten graph (float cell_0, OctbitMatMul for cell_1 and the FC),
    # one 300 ms chunk for 131,072 streams, PCM resident in HBM; CPU: the oracle loop over the UNMODIFIED reference op
    from keyword_spotting_b200 import OctbitModelWeights
    dm.set_octbit(OctbitModelWeights.from_float(wts))
    S3 = 131072
    pcm3 = (torch.randn((S3, 5120), device=device, generator=g) * 800).clamp_(-32768, 32767).to(torch.int16)
    st3 = torch.zeros((2, S3, 128), device=device)
    ms = timeit(lambda: dm(pcm3, st3), iters=3, warm=1)
    rec = dict(ms=ms, audio_s_per_s=0.3 * S3 / ms * 1e3,
               workload="configs[3]: graph_octbit.pb forward, 131072 streams x one 300 ms chunk (30 frames), per-stream activation "
                        "ranges (the reference's batch-1 semantics)")
    octw = om.octize_model(ow)
    nb3 = 4
    pc3 = om.pcm16_to_float(pcm3[:nb3].cpu().numpy())
    t = cpu_time(lambda: om.octbit_deploy_forward(pc3, np.zeros((2, nb3, 128), np.float32), ow, octw), min_s=2.0)
    rec["cpu_baseline"] = dict(audio_s_per_s=0.3 * nb3 / t, kind="reference op inside the oracle loop", cores=1,
                               sample="%d streams x 30 frames: numpy graph around the unmodified octbit_mat_mul_op.cc (oracle/_ref)" % nb3)
    rec["speedup_vs_cpu"] = rec["audio_s_per_s"] / rec["cpu_baseline"]["audio_s_per_s"]
    out["octbit_graph_S131072_chunk"] = rec
    del pcm3, st3
    dm.close()
    # ---- BASELINE configs[4]: attention_ctc forward, batched 8 s utterances (mel [B, 798, 60] -> T' = 400)
    am = AttentionDeployModel(AttentionConfig(), device=device)
    Ba = 1024
    mel = torch.rand((Ba, 798, 60), device=device, generator=g) * 2
    ms = timeit(lambda: am.run_mel(mel), iters=3, warm=2)
    flop = Ba * (400 * 120 * 128 * 2 + 3 * (400 * 128 * 384 * 2 + 2 * 8 * 400 * 400 * 16 * 2 + 2 * 400 * 128 * 512 * 2) + 400 * 128 * 6 * 2)
    rec = dict(ms=ms, utterances_per_s=Ba / ms * 1e3, audio_s_per_s=8.0 * Ba / ms * 1e3, TFLOPs=flop / ms / 1e9,
               tensor_frac=flop / ms / 1e9 / peaks["bf16"],
               workload="configs[4]: 1024 x 8 s, n_mel 60, mel frames resident in HBM -> attention_ctc softmax [B, 400, 6]")
    from oracle import attention as oat
    aw = oat.init_weights(seed=4321, n_mel=60)
    mc = mel[:2].cpu().numpy()
    t = cpu_time(lambda: oat.mel_forward(mc, aw), min_s=2.0)
    rec["cpu_baseline"] = dict(utterances_per_s=2 / t, kind="port", cores="numpy default threads of %d" % (os.cpu_count() or 1),
                               sample="2 utterances x 8 s through the numpy oracle (oracle/attention.py)")
    rec["speedup_vs_cpu"] = rec["utterances_per_s"] / rec["cpu_baseline"]["utterances_per_s"]
    out["attention_mel_forward_B1024_8s"] = rec
    del mel
    am.close()
    out["clocks"] = sampler.stop()
    return out


def run_ours(args, rank, world, local_rank):
    import ctypes
    import numpy as np
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    barrier = (lambda: dist.barrier()) if world > 1 else (lambda: None)

    from keyword_spotting_b200 import Config, DeployModel, StreamingDetector, WaveServer, _lib, sharding

    host_binding = sharding.bind_host_to_gpu(local_rank) if not args.no_bind else {"bound": False, "why": "--no-bind"}
    cfg = Config(n_mel=40)
    weights = boosted_weights(cfg, args.fc_gain)
    model = DeployModel(cfg, weights, device=device, precision=args.precision, frontend=args.frontend)
    S = args.streams
    det = StreamingDetector(model, S, keyword=args.keyword)
    n_buf = 4 if S <= 262144 else 2                  # 4 x 1.26 GB of PCM >> 126 MB L2: every step reads HBM-cold input
    chunks = make_chunks(torch, S, n_buf, device, seed=5678 + rank)
    stream = torch.cuda.current_stream(device)
    trig_total = torch.zeros((), dtype=torch.int64, device=device)
    trig = torch.empty(S, dtype=torch.int32, device=device)
    lib = _lib.load()

    # ---- parity of the streams about to be benchmarked (checker, outside every timed region)
    parity = None
    if rank == 0 and not args.no_parity:
        parity = parity_check(args, torch, model, weights, det, chunks, S)
    barrier()

    def step_dev(i):
        x = chunks[i % n_buf]
        _lib.check(lib.kws_stream_step(det._handle, x.data_ptr(), CHUNK, x.stride(0), trig.data_ptr(), None, None,
                                       stream.cuda_stream))

    for i in range(max(args.warmup, 3)):
        step_dev(i)
        trig_total.add_(trig.sum())                  # (also warms the reduction the timed loop uses)
    trig_total.zero_()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                              # 50 ms samples over every timed region below

    def step_counted(i):
        step_dev(i)
        trig_total.add_(trig.sum())                  # result consumption on the device (no host sync)

    total_ms, per_step = timed_loop(torch, step_counted, args.steps, stream, barrier)
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, stream_outputs(torch, det, trig))
    total_ms_max = sharding.reduce_max_scalar(total_ms, device)
    ms_per_step = total_ms_max / args.steps
    value = world * S * AUDIO_S_PER_CHUNK * args.steps / (total_ms_max * 1e-3)
    triggers_device_region = int(trig_total.item())

    # ---- the parts of the production step (front end incl. fused VAD/tail | GRU layers | decode), CUDA events inside
    # kws_stream_step (debug hook: every step synchronises, so this runs after the timed region)
    lib.kws_debug_step_timing(1, None, None)
    for i in range(2):                               # first use of the hook: event creation, not measured
        step_dev(i)
    lib.kws_debug_step_timing(0, None, None)
    lib.kws_debug_step_timing(1, None, None)         # switching resets the sums
    for i in range(6):
        step_dev(i)
    torch.cuda.synchronize()
    part_ms = (ctypes.c_double * 3)()
    part_n = ctypes.c_longlong(0)
    lib.kws_debug_step_timing(0, part_ms, ctypes.byref(part_n))
    parts = [part_ms[i] / max(1, part_n.value) for i in range(3)]

    # ---- the same kernels alone through the public entry points (front end without the fused pre-step, GRU from
    # row-major mel) on the same data
    mel = torch.empty((S, FRAMES, cfg.n_mel), dtype=torch.float32, device=device)
    pcm_full = torch.cat([chunks[0][:, -320:], chunks[1]], dim=1).contiguous()      # a steady-state 5120-sample input
    _lib.check(lib.kws_frontend_mel(model.handle, pcm_full.data_ptr(), _lib.PCM_I16, S, 5120, pcm_full.stride(0),
                                    mel.data_ptr(), stream.cuda_stream))
    st = torch.zeros((2, S, 128), dtype=torch.float32, device=device)
    probs = torch.empty((S, FRAMES, 6), dtype=torch.float32, device=device)

    def gru_only(i):
        _lib.check(lib.kws_gru_forward(model.handle, mel.data_ptr(), S, FRAMES, None, st.data_ptr(), probs.data_ptr(),
                                       st.data_ptr(), None, stream.cuda_stream))

    def fe_only(i):
        _lib.check(lib.kws_frontend_mel(model.handle, pcm_full.data_ptr(), _lib.PCM_I16, S, 5120, pcm_full.stride(0),
                                        mel.data_ptr(), stream.cuda_stream))

    gru_only(0)
    k_iters = max(3, min(args.steps, 10))
    gru_ms, _ = timed_loop(torch, gru_only, k_iters, stream, lambda: None)
    fe_ms, _ = timed_loop(torch, fe_only, k_iters, stream, lambda: None)
    # roofline launch times: the kernels as they run inside the production step
    gru_launch_ms = parts[1] / cfg.num_layers
    fe_launch_ms = parts[0]
    peaks = load_peaks()
    flop_per_launch = S * FRAMES * GRU_FLOP_PER_FRAME / cfg.num_layers
    achieved_tf = flop_per_launch / (gru_launch_ms * 1e-3) / 1e12
    kname = "gru_tc_kernel" if args.precision == "tc" else "gru_layer_kernel"
    traffic = load_traffic(S) if args.precision == "tc" else {}
    gru_traffic = None
    if "gru_tc_kernel_layer0" in traffic:
        gru_traffic = 0.5 * (traffic["gru_tc_kernel_layer0"] + traffic["gru_tc_kernel_layer1"])   # mean of the two launches
    roof_gru = dict(kernel=kname, bound="tensor", achieved=achieved_tf, peak=peaks["bf16_sustained"],
                    unit="TFLOP/s", frac=achieved_tf / peaks["bf16_sustained"], frac_of_burst_peak=achieved_tf / peaks["bf16"],
                    traffic=gru_traffic, launch_ms=gru_launch_ms,
                    peak_source=peaks["source"] + ", sustained bf16 (kernel timed inside a long step); burst fraction alongside",
                    note=("tcgen05 kind::f16 (fp16 operands, fp32 accumulate); " if args.precision == "tc" else
                          "exact fp32 FFMA kernel measured against the tensor-pipe peak; ") +
                         "algorithmic FLOP = 327,168 per frame (GRU 325,632 + FC 1,536), one launch per layer")
    fe_gbs = S * FE_BYTES_PER_STREAM_CHUNK / (fe_launch_ms * 1e-3) / 1e9
    roof_fe = dict(kernel="frontend_kernel" if args.frontend == "fft" else "frontend_tc_kernel", bound="hbm", achieved=fe_gbs, peak=peaks["hbm"], unit="GB/s",
                   frac=fe_gbs / peaks["hbm"], traffic=traffic.get("frontend_kernel"), launch_ms=fe_launch_ms,
                   algorithmic_bytes=S * FE_BYTES_PER_STREAM_CHUNK, traffic_source=traffic.get("_source"),
                   peak_source=peaks["source"] + ", copy bandwidth",
                   note="algorithmic bytes = %d per stream-chunk (int16 PCM in, carried tail r+w, fp32 mel out, flags); "
                        "one launch per step; timed inside the production step (fused VAD/tail work included)" % FE_BYTES_PER_STREAM_CHUNK,
                   limiter=("HBM is the bound by contract (SURVEY.md 8d), not in fact: DRAM traffic equals the algorithmic bytes, and ncu shows the "
                            "400-point FFT's shared-memory transposition at 72 % of the LSU wavefront peak with 50 % of the issue slots in use "
                            "(profiles/r02_ncu_summary_v11.md); the tensor-core formulation of the same transform reaches the same time "
                            "(profiles/r02_frontend_tc.md)") if args.frontend == "fft" else
                           "TMEM capacity: one accumulator buffer, transforms and combination of consecutive items cannot overlap "
                           "(profiles/r02_frontend_tc.md)")
    post_gbs = S * POST_BYTES_PER_STREAM_CHUNK / (max(parts[2], 1e-6) * 1e-3) / 1e9
    roof_post = dict(kernel="stream_post_kernel", bound="hbm", achieved=post_gbs, peak=peaks["hbm"], unit="GB/s",
                     frac=post_gbs / peaks["hbm"], traffic=traffic.get("stream_post_kernel"), launch_ms=parts[2],
                     algorithmic_bytes=S * POST_BYTES_PER_STREAM_CHUNK, peak_source=peaks["source"] + ", copy bandwidth",
                     note="K4 (window decode + trigger + resets): algorithmic bytes = %d per stream-chunk (30x6 fp32 probabilities "
                          "read, 30 one-byte tokens written, the 15-chunk token window re-read, window / VAD / trigger bookkeeping)"
                          % POST_BYTES_PER_STREAM_CHUNK)
    # the roofline of the dominant kernel (largest launch time); the others alongside
    roofline, roofline_other = (roof_fe, [roof_gru, roof_post]) if fe_launch_ms >= gru_launch_ms else (roof_gru, [roof_fe, roof_post])
    del pcm_full, mel, probs, st
    torch.cuda.empty_cache()                         # the library allocates with cudaMalloc: hand torch's cached blocks back

    # ---- end to end through the package's wave server (kws_server_*): pinned host PCM -> H2D -> step -> D2H flags
    e2e = None
    latency = None
    copy_ceiling = None
    triggers_e2e = None
    if not args.no_e2e:
        det.close()                                  # the full-batch server is not needed any more
        del chunks[2:]
        W = max(1, min(args.waves, S // 128))
        assert S % W == 0, "--streams must be divisible by --waves"
        srv = WaveServer(model, S, waves=W, use_graphs=not args.no_graphs, keyword=args.keyword)
        Sw = srv.streams_per_wave
        for w in range(W):                           # fill both ingest slots of every wave, run them once (warm-up)
            for b in range(2):
                srv.ingest_slot(w)[...] = chunks[b][w * Sw:(w + 1) * Sw].cpu().numpy()
                srv.submit(w)
            srv.wait(w)
            srv.wait(w)
        srv.serve(max(args.warmup, 3), args.depth)
        torch.cuda.synchronize()

        def timed_serve():
            srv.stats(reset=True)
            barrier()
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            ev0.record(stream)
            srv.serve(args.steps, args.depth)        # returns when every chunk's trigger flags are on the host
            ev1.record(stream)
            torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) * 1e3
            barrier()
            ms = sharding.reduce_max_scalar(max(ev0.elapsed_time(ev1), 0.0), device)
            return ms, wall, srv.stats()

        # copy-only leg first: the link ceiling of this box for the same buffers, CUDA streams and schedule
        srv.set_copy_only(True)
        srv.serve(2, args.depth)
        c_ms, c_wall, c_stats = timed_serve()
        srv.set_copy_only(False)
        srv.serve(2, args.depth)
        e_ms, e_wall, e_stats = timed_serve()
        h2d = S * CHUNK * 2
        copy_ceiling = dict(value=world * S * AUDIO_S_PER_CHUNK * args.steps / (c_ms * 1e-3), unit=UNIT,
                            ms_per_step=c_ms / args.steps, h2d_GBps_per_gpu=h2d / (c_ms / args.steps * 1e-3) / 1e9,
                            chunk_latency_ms_p99=c_stats["p99"],
                            note="same pinned buffers, CUDA streams, graphs and schedule with NO kernels (kws_server_set_copy_only)")
        e2e = dict(value=world * S * AUDIO_S_PER_CHUNK * args.steps / (e_ms * 1e-3), unit=UNIT,
                   h2d_bytes_per_step=h2d, d2h_bytes_per_step=S * 4, ms_per_step=e_ms / args.steps,
                   wall_ms_per_step=e_wall / args.steps, waves=W, depth=args.depth, cuda_graphs=srv.graphs,
                   h2d_GBps_per_gpu=h2d / (e_ms / args.steps * 1e-3) / 1e9,
                   frac_of_copy_ceiling=(c_ms / e_ms) if e_ms > 0 else None,
                   note="keyword_spotting_b200.WaveServer (kws_server_serve): pinned host int16 PCM -> H2D -> front end -> GRU -> "
                        "decode/trigger -> D2H trigger flags for every stream every step; %d waves of %d streams, one CUDA-graph "
                        "launch per wave and chunk, %d waves in flight" % (W, Sw, args.depth))
        latency = dict(e_stats)
        latency["definition"] = ("host clock from kws_server_submit of a wave's 300 ms chunk (pinned host memory) until its trigger "
                                 "flags are visible on the host, every (wave, chunk) of the e2e timed region (includes queueing "
                                 "behind the %d wave(s) in flight)" % (args.depth - 1))
        triggers_e2e = e_stats["triggers"]
        srv.close()
    clocks = sampler.stop() if rank == 0 else None

    trig_sum = torch.tensor([triggers_device_region + (triggers_e2e or 0)], dtype=torch.int64, device=device)
    if world > 1:
        dist.all_reduce(trig_sum)                    # the final result gather (NCCL), off the hot path
    ops = None
    if rank == 0 and world == 1 and not args.no_ops:
        ops = ops_block(args, torch, device, peaks)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_port_throughput(*cpu_sample_size(args, budget_s=15.0))
    if rank == 0:
        per_sorted = sorted(per_step)
        state_bytes_per_stream = 24 * 1024
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
                    ms_per_step=ms_per_step, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="f16 operands / f32 accumulate+state" if args.precision == "tc" else "f32",
                    data="synthetic",
                    config=dict(workload="streaming serve (BASELINE configs[2]): %d concurrent streams per GPU with carried GRU "
                                         "state and VAD reset, 300 ms chunks, 2L GRU-128 n_mel=40 6 classes" % S,
                                streams_per_gpu=S, chunk_samples=CHUNK, frames_per_chunk=FRAMES, sharding="streams/dp%d" % world,
                                l2_policy="inputs larger than L2: %d rotating %.2f GB PCM buffers" % (n_buf, S * CHUNK * 2 / 1e9),
                                fc_gain=args.fc_gain, keyword=args.keyword,
                                weights="random init of the reference architecture (seed 1234), FC scaled by fc_gain so that "
                                        "labels, triggers and their resets occur (the reference default keyword is '1233')"),
                    streams_resident=world * S,
                    realtime_capacity=dict(device_resident=value, e2e=(e2e["value"] if e2e else None),
                                           hbm_state_limit_per_gpu=int(170e9 // state_bytes_per_stream),
                                           note="streams at real time = audio-s/s; a capacity derived from throughput, bounded by "
                                                "~24 KB of resident state per stream; only `streams_resident` were actually held"),
                    chunk_latency_ms_p99=(latency["p99"] if latency else None), chunk_latency=latency,
                    full_batch_step_ms_p99=per_sorted[min(len(per_sorted) - 1, int(0.99 * len(per_sorted)))],
                    kernels_ms=dict(frontend=parts[0], gru_2_layers=parts[1], decode=parts[2], step_total=ms_per_step,
                                    standalone_frontend_no_pre_step=fe_ms / k_iters, standalone_gru_row_major_mel=gru_ms / k_iters,
                                    note="frontend/gru_2_layers/decode: CUDA events inside kws_stream_step (debug hook), "
                                         "mean of 6 synchronised steps after the timed region"),
                    roofline=roofline, roofline_other=roofline_other, parity_check=parity, cpu_baseline=cpu, e2e=e2e,
                    copy_ceiling=copy_ceiling, ops=ops,
                    gpu_launches=4 * args.steps, clocks=clocks, host_binding=host_binding,
                    triggers=int(trig_sum.item()), triggers_device_region=triggers_device_region)
        print(json.dumps(line), flush=True)
    if args.no_e2e:
        det.close()
    model.close()
    if world > 1:
        dist.destroy_process_group()


def run_attention(args, rank, world, local_rank):
    """BASELINE configs[4]: attention_ctc (n_mel 60, combine_frame 2, 3 x {8-head attention, FFN 512}) on batched 8 s
    utterances, sharded by utterance across the GPUs with no collective.  One step = `--utterances` utterances per GPU:
    int16 PCM -> mel (K1) -> positional encoding (K6) -> attention forward -> softmax [B, 400, 6]."""
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    barrier = (lambda: dist.barrier()) if world > 1 else (lambda: None)
    from keyword_spotting_b200 import AttentionConfig, AttentionDeployModel, sharding
    am = AttentionDeployModel(AttentionConfig(), device=device)
    B, L = args.utterances, 128000
    g = torch.Generator(device=device).manual_seed(4321 + rank)
    pcm = [(torch.randn((B, L), device=device, generator=g) * 800).clamp_(-32768, 32767).to(torch.int16) for _ in range(2)]
    host = [p_.cpu().pin_memory() for p_ in pcm]
    stream = torch.cuda.current_stream(device)
    out = [None]

    def step_dev(i):
        out[0] = am(pcm[i % 2])

    staging = torch.empty_like(pcm[0])
    probs_host = torch.empty((B, am.frames(am._frontend.num_frames(L)), 6), dtype=torch.float32).pin_memory()

    def step_e2e(i):
        staging.copy_(host[i % 2], non_blocking=True)
        probs_host.copy_(am(staging), non_blocking=True)

    for i in range(max(args.warmup, 3)):
        step_dev(i)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    total_ms, _ = timed_loop(torch, step_dev, args.steps, stream, barrier)
    if args.dump_outputs and rank == 0:
        sample = dump_sample(B, DUMP_SAMPLE_UTTERANCES)
        write_outputs(args.dump_outputs, dict(softmax=out[0][torch.from_numpy(sample).to(device)].cpu().numpy(),
                                              sample_utterances=sample.astype("float64")))
    total_ms = sharding.reduce_max_scalar(total_ms, device)
    for i in range(2):
        step_e2e(i)
    e_ms, _ = timed_loop(torch, step_e2e, args.steps, stream, barrier)
    e_ms = sharding.reduce_max_scalar(e_ms, device)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        audio = world * B * 8.0 * args.steps
        Tp = int(probs_host.shape[1])
        flop = B * (Tp * 120 * 128 * 2 + 3 * (Tp * 128 * 384 * 2 + 2 * 8 * Tp * Tp * 16 * 2 + 2 * Tp * 128 * 512 * 2) + Tp * 128 * 6 * 2)
        peaks = load_peaks()
        line = dict(metric="attention_ctc audio-sec/sec (BASELINE configs[4])", value=audio / (total_ms * 1e-3), unit=UNIT,
                    n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=total_ms / args.steps,
                    higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                    config=dict(workload="attention_ctc forward (BASELINE configs[4]): %d x 8 s utterances per GPU, n_mel 60, int16 PCM "
                                         "resident in HBM -> mel -> PE -> 3 x {8-head attention, FFN 512} -> softmax [B, %d, 6]" % (B, Tp),
                                utterances_per_gpu=B, sharding="utterances/dp%d" % world,
                                l2_policy="inputs larger than L2: 2 rotating %.0f MB PCM buffers" % (B * L * 2 / 1e6)),
                    utterances_per_s=world * B * args.steps / (total_ms * 1e-3),
                    roofline=dict(kernel="att_linear_tc_kernel + att_core_tc_kernel (tcgen05 kind::f16, fp16 hi/lo operand splits)", bound="tensor",
                                  achieved=flop * args.steps / (total_ms * 1e-3) / 1e12, peak=peaks["bf16"], unit="TFLOP/s",
                                  frac=flop * args.steps / (total_ms * 1e-3) / 1e12 / peaks["bf16"], traffic=None,
                                  note="algorithmic 0.69 GFLOP per utterance over the whole step (front end, layer norm and softmax passes included); "
                                       "every contraction runs as three fp16 MMAs (x_hi w_hi + x_lo w_hi + x_hi w_lo) for fp32-grade results, "
                                       "so the tensor pipe executes 3x the algorithmic FLOP; see DESIGN.md"),
                    e2e=dict(value=audio / (e_ms * 1e-3), unit=UNIT, h2d_bytes_per_step=B * L * 2, d2h_bytes_per_step=B * Tp * 6 * 4,
                             ms_per_step=e_ms / args.steps,
                             note="pinned host int16 PCM -> H2D -> AttentionDeployModel call -> D2H softmax, every step"),
                    gpu_launches=26 * args.steps, clocks=clocks)
        print(json.dumps(line), flush=True)
    am.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if args.workload == "attention":
        run_attention(args, rank, world, local_rank)
        return
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()

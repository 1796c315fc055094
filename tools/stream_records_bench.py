"""Per-stream records: kws_stream_export / kws_stream_import on one stream object and kws_server_export /
kws_server_import on a wave server, all --streams streams per call, in a random order spread over the object.

The records (--streams x record bytes, 310 MB at the defaults) and the objects' state are larger than the 126 MB L2.
The four calls are warmed up, then alternated --repeats times (CUDA events around --iters calls; median / min / max).
The server calls synchronise their stream before returning, so their time includes the per-wave pointer table upload
and that synchronisation.  Record GB/s counts record bytes only (written by an export, read by an import); the object
side moves at most as many bytes again, so "hbm_upper_GBps" = 2 x record bytes / time bounds the HBM traffic.  The
card's name and power limit are read in the same run.

    python tools/stream_records_bench.py [--streams 131072] [--waves 32] [--out results.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM_DATASHEET_GBPS = 7700.0      # HGX B200 data sheet, one GPU


def card(index):
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001 -- the measurement stands without it; say so
        q = "nvidia-smi unavailable (%s)" % e
    return dict(device=torch.cuda.get_device_name(index), nvidia_smi=q)


def time_variants(variants, repeats, iters):
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=131072)
    ap.add_argument("--waves", type=int, default=32)
    ap.add_argument("--repeats", type=int, default=15)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("stream_records_bench needs a CUDA device")

    from keyword_spotting_b200 import Config, DeployModel, ModelWeights, StreamingDetector, WaveServer, _lib
    from oracle import model as om
    ow = om.init_weights(seed=3, n_mel=40)
    dm = DeployModel(Config(n_mel=40), ModelWeights.from_arrays(ow.mel_basis, ow.gates_kernel, ow.gates_bias,
                                                                ow.cand_kernel, ow.cand_bias, ow.fc_w, ow.fc_b))
    lib = _lib.load()
    S = args.streams
    rng = np.random.default_rng(0)
    det = StreamingDetector(dm, S)
    srv = WaveServer(dm, S, waves=args.waves)
    for _ in range(3):                                   # carried state that is not all zero
        det.step(torch.from_numpy(rng.integers(-3000, 3000, (S, 4800), dtype=np.int16)).cuda())
    R = det.record_bytes
    ids = torch.from_numpy(rng.permutation(S).astype(np.int64)).cuda()
    recs_det = det.export_streams(ids)
    srv.import_streams(ids, recs_det)                    # the server now carries the detector's state
    status = torch.empty(S, dtype=torch.int32, device="cuda")
    out = torch.empty_like(recs_det)
    sp = lambda: torch.cuda.current_stream().cuda_stream
    p = lambda t: t.data_ptr()

    def ok(rc):
        if rc != 0:
            raise RuntimeError(_lib.last_error())

    variants = {
        "stream_export": lambda: ok(lib.kws_stream_export(det._handle, p(ids), S, p(out), sp())),
        "stream_import": lambda: ok(lib.kws_stream_import(det._handle, p(ids), S, p(recs_det), p(status), sp())),
        "server_export": lambda: ok(lib.kws_server_export(srv._handle, p(ids), S, p(out), sp())),
        "server_import": lambda: ok(lib.kws_server_import(srv._handle, p(ids), S, p(recs_det), p(status), sp())),
    }
    ms = time_variants(variants, args.repeats, args.iters)
    assert int(status.abs().sum()) == 0
    assert torch.equal(det.export_streams(ids), recs_det) and torch.equal(srv.export_streams(ids), recs_det)
    rows = []
    for name, v in ms.items():
        med = float(np.median(v))
        gbps = S * R / (med * 1e-3) / 1e9
        rows.append(dict(call=name, streams=S, record_bytes=R, record_MB=S * R / 1e6, ms_median=med,
                         ms_min=float(min(v)), ms_max=float(max(v)), record_GBps=gbps, hbm_upper_GBps=2 * gbps,
                         hbm_datasheet_GBps=HBM_DATASHEET_GBPS))
    result = dict(card=card(torch.cuda.current_device()), waves=args.waves, repeats=args.repeats, iters=args.iters,
                  rows=rows)
    for r in rows:
        print("%-14s %8.3f ms (min %.3f, max %.3f)  %7.1f GB/s of records, <= %7.1f GB/s HBM"
              % (r["call"], r["ms_median"], r["ms_min"], r["ms_max"], r["record_GBps"], r["hbm_upper_GBps"]))
    print(json.dumps(result["card"]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    srv.close()
    det.close()
    dm.close()


if __name__ == "__main__":
    main()

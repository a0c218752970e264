#!/usr/bin/env python
"""Cost of moving stream state: wwb_stream_export / wwb_stream_import against a plain device copy of the same bytes.

    python tools/bench_stream_state.py [--calls 20] [--rounds 5] [--warmup 3]

A WaveNet tc context of 65 536 slots x 320 samples (a few dense pushes first, so the windows start at varied ring rows and
half of them wrap) exports and imports K random slots, K = 4096 and 65 536.  Per K:
  - export and import: time per call from CUDA events around `--calls` back-to-back C ABI calls on preallocated buffers
    (host work included: the id checks and the id table's copy), after warm-up; bytes per call = K records.
  - the yardstick: a device-to-device torch copy of the same byte count, timed the same way in the same rounds.
    GB/s counts the record bytes once, as for the copy (each reads and writes them once).
  - parking a session: the K records through page-locked host memory and back (device -> host, host -> device), and the
    whole park + resume: export, copy out, copy in, import.
Export, import and the copy alternate within each of `--rounds` rounds; the median and min..max over the rounds are
reported.  The import's status is checked after the timing.  Prints one JSON line with the GPU's name and power limit,
read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_stream_indexed import gpu_info  # noqa: E402


def timed(torch, fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n * 1e3   # us per call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--cap", type=int, default=65536)
    args = ap.parse_args()
    if args.calls < 1 or args.rounds < 1:
        ap.error("--calls and --rounds must be at least 1")
    import torch
    from wakeword_detection_b200 import _cabi, synth, weights as W
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    eng = _cabi.Engine(W.load_model_dir(os.path.join(ROOT, "weights", "Wavenet"), "Wavenet"), 0, "tc")
    n = 320
    eng.stream_alloc(args.cap, n)
    for k in range(5):
        eng.stream_push(synth.device_pcm(args.cap, n, seed=k, device=dev))
    nb = eng.stream_state_bytes()
    res = {"metric": "stream_state_export_import", "unit": "us per call", **gpu_info(), "model": "Wavenet", "precision": "tc",
           "slots": args.cap, "chunk_samples": n, "record_bytes": nb, "calls_per_figure": args.calls, "rounds": args.rounds}
    stream = eng._stream()
    lib, ctx = eng.lib, eng.ctx
    rng = np.random.default_rng(5)
    med = lambda x: float(np.median(x))
    for K in (4096, args.cap):
        ids = np.ascontiguousarray(rng.permutation(args.cap)[:K], np.int32)
        rec = torch.empty((K, nb), dtype=torch.uint8, device=dev)
        src, dst = torch.empty_like(rec), torch.empty_like(rec)
        status = torch.zeros(2, dtype=torch.int32, device=dev)
        host = torch.empty((K, nb), dtype=torch.uint8).pin_memory()
        fns = {
            "export": lambda: lib.wwb_stream_export(ctx, ids.ctypes.data, K, rec.data_ptr(), stream),
            "import": lambda: lib.wwb_stream_import(ctx, ids.ctypes.data, K, rec.data_ptr(), status.data_ptr(), stream),
            "copy": lambda: dst.copy_(src),
            "d2h": lambda: host.copy_(rec, non_blocking=True),
            "h2d": lambda: rec.copy_(host, non_blocking=True),
        }
        assert fns["export"]() == 0
        for _ in range(args.warmup):
            for f in fns.values():
                f()
        torch.cuda.synchronize()
        t = {k: [] for k in fns}
        for _ in range(args.rounds):
            for k, f in fns.items():
                t[k].append(timed(torch, f, args.calls))
        bad, why = status.cpu().tolist()
        if bad:
            raise SystemExit("import rejected record %d (reason %d)" % (bad - 1, why))
        before = rec.clone()
        fns["import"]()
        fns["export"]()
        assert torch.equal(rec, before), "export after import differs from the imported records"
        gb = K * nb / 1e9
        row = {"bytes_per_call": K * nb}
        for k in fns:
            row[k + "_us"] = round(med(t[k]), 1)
            row[k + "_spread_us"] = [round(min(t[k]), 1), round(max(t[k]), 1)]
            row[k + "_GBps"] = round(gb / (med(t[k]) * 1e-6), 1)
        row["export_over_copy_bw"] = round(med(t["copy"]) / med(t["export"]), 3)
        row["import_over_copy_bw"] = round(med(t["copy"]) / med(t["import"]), 3)
        row["park_and_resume_us"] = round(sum(med(t[k]) for k in ("export", "d2h", "h2d", "import")), 1)
        res["K_%d" % K] = row
        del rec, src, dst, host
        torch.cuda.empty_cache()
    eng.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()

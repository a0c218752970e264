#!/usr/bin/env python
"""Cost of indexed streaming pushes (wwb_stream_push_indexed) against dense pushes (wwb_stream_push).

    python tools/bench_stream_indexed.py [--pushes 48] [--rounds 5] [--warmup 8]

(a) the dense shape (BASELINE config 4: WaveNet tc, 4096 streams x 160 samples): stream_push against
    stream_push_indexed(ids=arange(4096)) on the same context.
(b) cost in proportion to the pushed streams: a context of 65 536 slots x 320 samples receives indexed pushes over 256
    and over 4096 random slots; each is compared with a dense push of as many streams on a context whose capacity is
    exactly that number.  CRNN and WaveNet, tc.

Each figure is the time per push from CUDA events around `--pushes` back-to-back pushes through the Python Engine (the
call a server makes, host work included), after warm-up.  A and B alternate within the run, `--rounds` times; the
median and the spread (min..max) over the rounds are reported.  Prints one JSON line with the GPU's name and power
limit, read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:  # the JSON line says so rather than guessing
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unavailable (%s)" % type(e).__name__}


def timed(torch, fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n * 1e3   # us per push


def compare(torch, fa, fb, args):
    for _ in range(args.warmup):
        fa()
        fb()
    torch.cuda.synchronize()
    ta, tb = [], []
    for _ in range(args.rounds):
        ta.append(timed(torch, fa, args.pushes))
        tb.append(timed(torch, fb, args.pushes))
    med = lambda x: float(np.median(x))
    return {"a_us": round(med(ta), 1), "a_spread_us": [round(min(ta), 1), round(max(ta), 1)],
            "b_us": round(med(tb), 1), "b_spread_us": [round(min(tb), 1), round(max(tb), 1)],
            "b_over_a": round(med(tb) / med(ta), 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pushes", type=int, default=48)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--cap", type=int, default=65536)
    args = ap.parse_args()
    if args.pushes < 48:
        ap.error("--pushes must be at least 48")
    import torch
    from wakeword_detection_b200 import _cabi, synth, weights as W
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    wts = {m: W.load_model_dir(os.path.join(ROOT, "weights", m), m) for m in ("CRNN", "Wavenet")}
    res = {"metric": "stream_push_indexed", "unit": "us per push", **gpu_info(),
           "pushes_per_figure": args.pushes, "rounds": args.rounds}

    # (a) config 4 shape on one context: A = dense push, B = indexed push over arange(S)
    S, n = 4096, 160
    eng = _cabi.Engine(wts["Wavenet"], 0, "tc")
    eng.stream_alloc(S, n)
    pcm = synth.device_pcm(S, n, seed=1, device=dev)
    flat, ids, lens = pcm.reshape(-1), np.arange(S, dtype=np.int32), np.full(S, n, np.int32)
    res["a_dense_shape_wavenet_tc_4096x160"] = compare(
        torch, lambda: eng.stream_push(pcm), lambda: eng.stream_push_indexed(ids, flat, lens), args)
    eng.close()

    # (b) A = dense push of K streams on a K-slot context, B = indexed push of K random slots of a cap-slot context
    n = 320
    rng = np.random.default_rng(5)
    for model in ("CRNN", "Wavenet"):
        big = _cabi.Engine(wts[model], 0, "tc")
        big.stream_alloc(args.cap, n)
        for K in (256, 4096):
            small = _cabi.Engine(wts[model], 0, "tc")
            small.stream_alloc(K, n)
            pcm = synth.device_pcm(K, n, seed=K, device=dev)
            flat = pcm.reshape(-1)
            slots = rng.permutation(args.cap)[:K].astype(np.int32)
            lens = np.full(K, n, np.int32)
            res["b_%s_tc_%d_of_%d" % (model.lower(), K, args.cap)] = compare(
                torch, lambda: small.stream_push(pcm), lambda: big.stream_push_indexed(slots, flat, lens), args)
            small.close()
        big.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()

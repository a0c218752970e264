#!/usr/bin/env python
"""CRNN encode + detect stage at several window lengths L (the shipped CRNN's weights with mel_length = L: the weights
do not depend on L), tc.

    python tools/bench_crnn_window_lengths.py [--lengths 97,151,201,256] [--iters 20] [--rounds 5] [--warmup 3]

(a) sliding: the bench shape, 512 streams x 10 s of mel (997 frames) at hop 2, one wwb_posteriors call;
(b) windows: 8192 independent [L, 40] windows, one wwb_posteriors call with n_frames == L.

Each figure is the time per call from CUDA events around `--iters` back-to-back calls after warm-up; the median and the
spread (min..max) over `--rounds` rounds are reported.  Inputs are uniform [0, 5) mel values made on the device (the
sliding mel is 82 MB, the windows 33..84 MB: both fit the L2, read from there after the first pass).  Algorithmic
FLOP per window: 422 912 T + 8 192 + 128 n_out (T = ceil(L / 8): conv 128 000, GRU-1 input projection 245 760, the two
recurrences 2 x 12 288 and the GRU-2 input projection 24 576 per step; detect), against a peak of 1390.4 TFLOP/s.  The
path the sliding call took (shared columns or per-window tiles) is read from its kernel launch count.  Prints one JSON
line with the GPU's name and power limit, read in the same run.
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

from bench_stream_indexed import gpu_info, timed  # noqa: E402

PEAK_TFLOPS = 1390.4
S, SECONDS, HOP, N_WIN = 512, 10.0, 2, 8192


def flop_per_window(L, n_out):
    return 422912 * (-(-L // 8)) + 8192 + 128 * n_out


def figure(torch, fn, n_win, flop, args):
    for _ in range(args.warmup):
        fn()
    torch.cuda.synchronize()
    ms = [timed(torch, fn, args.iters) / 1e3 for _ in range(args.rounds)]
    med = float(np.median(ms))
    return {"ms": round(med, 3), "spread_ms": [round(min(ms), 3), round(max(ms), 3)],
            "windows_per_s": round(n_win / (med / 1e3)),
            "tflops": round(n_win * flop / (med / 1e3) / 1e12, 1),
            "share_of_peak": round(n_win * flop / (med / 1e3) / 1e12 / PEAK_TFLOPS, 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lengths", default="97,151,201,256")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    import torch
    from wakeword_detection_b200 import _cabi, weights as W
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    base = W.load_model_dir(os.path.join(ROOT, "weights", "CRNN"), "CRNN")
    n_out = int(base["det2_w"].shape[0])
    F = int((SECONDS * 16000 - 512) // 160 + 1)
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    mel = torch.rand((S, F, 40), device=dev, generator=g) * 5
    res = {"metric": "crnn_stage_by_window_length", "unit": "ms per call", "precision": "tc", **gpu_info(),
           "sliding": "%d streams x %d frames, hop %d" % (S, F, HOP), "windows": N_WIN, "iters": args.iters,
           "rounds": args.rounds, "peak_tflops": PEAK_TFLOPS, "lengths": {}}
    for L in (int(x) for x in args.lengths.split(",")):
        eng = _cabi.Engine(dict(base, mel_length=np.int32(L)), 0, "tc")
        n_slide = S * ((F - L) // HOP + 1)
        n0 = eng.launch_count()
        eng.posteriors(mel, hop=HOP)
        launches = eng.launch_count() - n0
        wins = (torch.rand((N_WIN, L, 40), device=dev, generator=g) * 5).contiguous()
        fl = flop_per_window(L, n_out)
        res["lengths"][str(L)] = {
            "T": -(-L // 8), "flop_per_window": fl,
            "sliding_path": "per-window tiles" if launches == 4 else "shared columns (%d front launches)" % (launches - 3),
            "sliding": figure(torch, lambda: eng.posteriors(mel, hop=HOP), n_slide, fl, args),
            "windows": figure(torch, lambda: eng.posteriors(wins, hop=1), N_WIN, fl, args)}
        eng.close()
        del wins
    print(json.dumps(res))


if __name__ == "__main__":
    main()

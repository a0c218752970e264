#!/usr/bin/env python
"""Cost of a speech pipeline with several wake-word stages (wwb_context_step_chain) at 4096 streams x one 320-sample
frame per step, tc.

    python tools/bench_stream_chain.py [--steps 48] [--rounds 5] [--warmup 8]

(a) K = 1, 2, 3 stages (WaveNet, CRNN, CRNN_arik_original) in one chain step, against K independent one-stage
    pipelines (wwb_context_step on K contexts, which do not see each other's activations) over the same audio.
(b) the indexed form (wwb_context_step_chain_indexed) over a random half of the 4096 slots, K = 1, 2, 3.

Each figure is the time per step from CUDA events around `--steps` back-to-back steps through the Python Engine (host
work included), after warm-up; A and B alternate within the run `--rounds` times and the median and spread (min..max)
over the rounds are reported, with stream-steps per second from the median.  Prints one JSON line with the GPU's name
and power limit, read in the same run.
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

MODELS = ("Wavenet", "CRNN", "CRNN_arik_original")
S, N = 4096, 320


def compare(torch, fa, fb, args, streams_a, streams_b):
    for _ in range(args.warmup):
        fa()
        fb()
    torch.cuda.synchronize()
    ta, tb = [], []
    for _ in range(args.rounds):
        ta.append(timed(torch, fa, args.steps) / 1e3)   # ms per step
        tb.append(timed(torch, fb, args.steps) / 1e3)
    med = lambda x: float(np.median(x))
    fig = lambda x, n: {"ms": round(med(x), 3), "spread_ms": [round(min(x), 3), round(max(x), 3)],
                        "stream_steps_per_s": round(n / (med(x) / 1e3))}
    return {"a": fig(ta, streams_a), "b": fig(tb, streams_b), "b_over_a": round(med(tb) / med(ta), 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=48)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=8)
    args = ap.parse_args()
    import torch
    from wakeword_detection_b200 import _cabi, synth, weights as W
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"metric": "context_step_chain", "unit": "ms per step", "streams": S, "frame_samples": N, **gpu_info(),
           "steps_per_figure": args.steps, "rounds": args.rounds}

    def engine(model, pipeline):
        typ = "Wavenet" if model == "Wavenet" else "CRNN"
        e = _cabi.Engine(W.load_model_dir(os.path.join(ROOT, "weights", model), typ), 0, "tc")
        e.stream_alloc(S, N)
        if pipeline:
            e.context_alloc()
        return e

    chain = [engine(m, i == 0) for i, m in enumerate(MODELS)]
    solo = [chain[0]] + [engine(m, True) for m in MODELS[1:]]
    pcm = synth.device_pcm(S, N, seed=3, device=dev)
    vad = torch.ones(S, dtype=torch.uint8, device=dev)
    half = np.sort(np.random.default_rng(7).permutation(S)[:S // 2]).astype(np.int32)
    np.random.default_rng(8).shuffle(half)
    flat, lens = pcm[:S // 2].reshape(-1), np.full(S // 2, N, np.int32)
    vad_half = vad[:S // 2]
    for K in (1, 2, 3):
        # A: K independent one-stage pipelines; B: one chain step with K stages
        res["a_vs_b_K%d" % K] = compare(
            torch, lambda: [e.context_step(pcm, vad) for e in solo[:K]],
            lambda: chain[0].context_step_chain(chain[1:K], pcm, vad), args, S, S)
    for K in (1, 2, 3):
        # A: the dense chain step over all 4096 streams; B: the indexed chain step over a random half of the slots
        res["dense_vs_half_indexed_K%d" % K] = compare(
            torch, lambda: chain[0].context_step_chain(chain[1:K], pcm, vad),
            lambda: chain[0].context_step_chain_indexed(chain[1:K], half, flat, lens, vad_half), args, S, S // 2)
    for e in chain + solo[1:]:
        e.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Cost of per-slot trigger options (wwb_stream_set_options) on 4096 streams x one 320-sample frame per step, tc.

    python tools/bench_stream_options.py [--steps 48] [--rounds 5] [--warmup 8] [--no-chain]
                                         [--parent DIR [--ab-rounds 2] [--ab bench_stream_chain,bench_stream_indexed,bench_py]]

(1) A dense chain step of K = 4 shipped models (WaveNet, CRNN, CRNN_arik_original, CRNN_arik_nosilence):
    - every stream listening to every stage;
    - each stream listening to exactly one stage, stream s to stage s % 4;
    - one-stage MultiStreamPipeline steps (wwb_context_step) of each of the four models, for scale.
    Every threshold is +inf, so that no activation makes a stage skip frames.
    Time per step from CUDA events around `--steps` back-to-back steps through the Python Engine (host work included),
    after warm-up; the cases alternate within the run `--rounds` times, median and spread (min..max) over the rounds.
(2) With --parent DIR (a checkout of the parent commit with its library built): tools/bench_stream_chain.py,
    tools/bench_stream_indexed.py and bench.py (extra.configs.config4_wavenet_streaming: the stream_push leg), none of
    which sets options, run from DIR and from this tree in turn, `--ab-rounds` times, in this one call (`--ab` picks
    which of the three).

Prints one JSON line with the GPU's name and power limit, read in the same run.
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
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_stream_indexed import gpu_info, timed  # noqa: E402

MODELS = ("Wavenet", "CRNN", "CRNN_arik_original", "CRNN_arik_nosilence")
S, N = 4096, 320


def chain_figures(args):
    import torch
    from wakeword_detection_b200 import _cabi, synth, weights as W
    dev = torch.device("cuda", 0)
    K = len(MODELS)

    def engine(model, pipeline):
        e = _cabi.Engine(W.load_model_dir(os.path.join(ROOT, "weights", model), "Wavenet" if model == "Wavenet" else
                                          "CRNN"), 0, "tc")
        e.stream_alloc(S, N)
        if pipeline:
            e.context_alloc()
        return e

    every = [engine(m, k == 0) for k, m in enumerate(MODELS)]
    single = [engine(m, k == 0) for k, m in enumerate(MODELS)]
    solo = [engine(m, True) for m in MODELS]
    # slot thresholds of +inf: no stream ever triggers, so a listening stage analyses every frame of every step (an
    # activation would make the later stages skip their chunks and hide their cost)
    ids = np.arange(S, dtype=np.int32)
    for e in every:
        e.stream_set_options(ids, threshold=np.inf)
    for k, e in enumerate(single):
        e.stream_set_options(ids, threshold=np.inf, listening=(ids % K == k).astype(np.uint8))
    pcm = synth.device_pcm(S, N, seed=3, device=dev)
    vad = torch.ones(S, dtype=torch.uint8, device=dev)
    cases = {"every_stream_every_stage": lambda: every[0].context_step_chain(every[1:], pcm, vad),
             "each_stream_one_stage_round_robin": lambda: single[0].context_step_chain(single[1:], pcm, vad)}
    for m, e in zip(MODELS, solo):
        cases["one_stage_pipeline_%s" % m] = (lambda e=e: e.context_step(pcm, vad, threshold=np.inf))
    for _ in range(args.warmup):
        for fn in cases.values():
            fn()
    torch.cuda.synchronize()
    t = {name: [] for name in cases}
    for _ in range(args.rounds):
        for name, fn in cases.items():
            t[name].append(timed(torch, fn, args.steps) / 1e3)   # ms per step
    # encoder windows of one more step of each case (round robin: each stage runs a quarter of the streams)
    win = {name: int(fn()["n_post"].sum()) for name, fn in cases.items()}
    for e in every + single + solo:
        e.close()
    med = lambda x: float(np.median(x))
    out = {name: {"ms": round(med(x), 3), "spread_ms": [round(min(x), 3), round(max(x), 3)]} for name, x in t.items()}
    for name, n in win.items():
        out[name]["windows_per_step"] = n
    return out


def ab(args):
    """parent / branch runs of the unchanged benchmarks, alternated"""
    trees = {"parent": os.path.abspath(args.parent), "branch": ROOT}
    runs = {"bench_stream_chain": [sys.executable, "tools/bench_stream_chain.py"],
            "bench_stream_indexed": [sys.executable, "tools/bench_stream_indexed.py"],
            "bench_py": [sys.executable, "bench.py", "--gpus", "1", "--steps", "10", "--warmup", "3",
                         "--no-cpu-baseline"]}
    runs = {name: runs[name] for name in args.ab.split(",")}
    out = {name: {t: [] for t in trees} for name in runs}
    env = {k: v for k, v in os.environ.items() if k not in ("WWB200_LIB", "PYTHONPATH")}
    for _ in range(args.ab_rounds):
        for name, cmd in runs.items():
            for tree, path in trees.items():
                r = subprocess.run(cmd, cwd=path, env=env, capture_output=True, text=True)
                if r.returncode:
                    raise SystemExit("%s in %s failed:\n%s" % (name, tree, r.stderr[-3000:]))
                res = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
                if name == "bench_py":
                    res = {"config4_wavenet_streaming": res["extra"]["configs"]["config4_wavenet_streaming"],
                           "value": res.get("value"), "unit": res.get("unit")}
                out[name][tree].append(res)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=48)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--parent", default=None, help="checkout of the parent commit, library built")
    ap.add_argument("--ab-rounds", type=int, default=2)
    ap.add_argument("--ab", default="bench_stream_chain,bench_stream_indexed,bench_py")
    ap.add_argument("--no-chain", action="store_true", help="skip part (1)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"metric": "stream_set_options", "unit": "ms per step", "streams": S, "frame_samples": N, **gpu_info(),
           "steps_per_figure": args.steps, "rounds": args.rounds}
    if not args.no_chain:
        res["chain_K4"] = chain_figures(args)
    if args.parent:
        res["parent_vs_branch"] = ab(args)
    print(json.dumps(res))


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Benchmark of the filter -> encode -> detect hot path (BASELINE.json metric:
audio-hours/sec at 1/2/4/8 B200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload sweep|filter|crnn|wavenet]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # CPU restatement of the reference path, host cores
    python bench.py ... --dump-outputs DIR    # + what the last timed step computed, as DIR/<name>.npy

One "step" = one pass of the hot path over one batch of synthetic 16 kHz int16 PCM.
Default workload "sweep" (BASELINE config 5, one time-chunk of it): S streams x T s ->
fused filter kernel -> CRNN and WaveNet encode+detect over all hop-2 windows
(get_posterior semantics) -> FAR/FRR counters.  Per-GPU work is fixed (weak scaling);
streams shard over ranks and the only collective is one all-reduce of the int64 counters.
Every step sees different PCM (three rotating batches from counter-based seeds, a wake clip
spliced into some streams so that the counters are not all zero).
`value` = audio-hours of PCM all ranks processed per second with the PCM resident in
HBM; `e2e` = the same work through the library's host-buffer plugin call
(wwb_sweep_submit / wwb_sweep_wait over ctypes, numpy buffers in pinned host memory): H2D of
the PCM, kernels, D2H of the posteriors and counters, all inside the timed region.
`extra.parity` compares a sample of the step's posteriors / decisions / counters with the CPU
oracle (outside the timed region); `extra.configs` carries short measurements of BASELINE
configs 2, 3 and 4.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_WINDOW = {"CRNN": 8043648, "Wavenet": 20663552}     # BASELINE.md §2
BYTES_PER_FRAME = 480                                         # 320 B int16 in + 160 B mel out
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return {k: float(d[k]) for k in FALLBACK_PEAKS}, "measured"
        except Exception:
            pass
    return dict(FALLBACK_PEAKS), "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------- CPU arm
def _cpu_stream_worker(args):
    """One stream through the CPU restatement of the reference path (oracle), both models."""
    seed, n_samples, models = args
    from threadpoolctl import threadpool_limits
    from oracle import restated as R
    from wakeword_detection_b200 import synth, weights as W
    with threadpool_limits(limits=1):
        pcm = synth.stream_int16(n_samples, seed % synth.N_CLASSES, 11, seed)
        x = R.int16_to_float(pcm)
        n = 0
        for m in models:
            w = W.load_model_dir(os.path.join(ROOT, "weights", m), m)
            mel = R.mel_stream(x, w)
            L = int(w["mel_length"])
            nw = R.eval_windows(mel.shape[0], L)
            j = np.arange(nw)
            for i in range(0, nw, 64):
                jj = j[i:i + 64]
                R.posterior(mel[(2 * jj)[:, None] + np.arange(L)[None, :]], w)
            n += nw
    return n


def cpu_reference_rate(models, n_streams, seconds_per_stream, processes):
    """audio-hours/sec of the oracle on `processes` host processes (1 BLAS thread each)."""
    import multiprocessing as mp
    n_samples = int(seconds_per_stream * 16000)
    jobs = [(s, n_samples, models) for s in range(n_streams)]
    t0 = time.perf_counter()
    if processes == 1:
        for j in jobs:
            _cpu_stream_worker(j)
    else:
        with mp.get_context("spawn").Pool(processes) as pool:
            pool.map(_cpu_stream_worker, jobs)
    dt = time.perf_counter() - t0
    return n_streams * seconds_per_stream / 3600.0 / dt, dt


def measured_traffic(kernel, S, N):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture
    (profiles/r2_traffic.json, taken at 512 streams x 10 s; the traffic - per-frame snapshots and input-layer rows - is
    per stream, so it is scaled to the step's stream count); only valid for the stream length it was captured on."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json"))).get(kernel)
        if d and abs(d["seconds"] - N / 16000.0) < 1e-9 and (d["streams"] == S or d.get("scales_with") == "streams"):
            return int(round(d["bytes_per_launch"] * (S / float(d["streams"]))))
    except Exception:
        pass
    return None


def workload_models(workload):
    return {"sweep": ["CRNN", "Wavenet"], "crnn": ["CRNN"], "wavenet": ["Wavenet"], "filter": []}[workload]


def default_shape(workload, args):
    if workload == "filter":
        return args.streams or 100000, int((args.seconds or 2.0) * 16000)       # BASELINE config 2
    return args.streams or 2560, int((args.seconds or 10.0) * 16000)            # one time-chunk of config 5 per GPU


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    models = workload_models(args.workload) or ["CRNN"]
    cores = os.cpu_count() or 1
    sec = 30.0 if args.workload != "filter" else 300.0
    rates = []
    for i in range(args.warmup + args.steps):
        if args.workload == "filter":
            r, dt = cpu_filter_rate(cores, sec)
        else:
            r, dt = cpu_reference_rate(models, cores, sec, cores)
        if i >= args.warmup:
            rates.append((r, dt))
    value = float(np.mean([r for r, _ in rates]))
    ms = float(np.mean([dt for _, dt in rates]) * 1e3)
    sample = ("each step a bounded sample of the workload: %d streams x %.0f s, %d processes x 1 thread, numpy restatement "
              "of the TFLite graphs (TFLite itself is not installable here)" % (cores, sec, cores))
    S, N = default_shape(args.workload, args)
    line = {"impl": "reference", "metric": "audio_hours_per_sec", "value": value, "unit": "audio-h/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config_dict(args, S, N),
            "cpu_baseline": {"value": value, "unit": "audio-h/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "audio-h/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def _cpu_filter_worker(args):
    seed, n_samples = args
    from threadpoolctl import threadpool_limits
    from oracle import restated as R
    from wakeword_detection_b200 import synth, weights as W
    with threadpool_limits(limits=1):
        w = W.load_model_dir(os.path.join(ROOT, "weights", "CRNN"), "CRNN")
        pcm = synth.stream_int16(16000, seed % synth.N_CLASSES, 11, seed)
        pcm = np.tile(pcm, n_samples // 16000 + 1)[:n_samples]
        R.mel_stream(R.int16_to_float(pcm), w)
    return 1


def cpu_filter_rate(processes, seconds_per_stream):
    import multiprocessing as mp
    n_samples = int(seconds_per_stream * 16000)
    t0 = time.perf_counter()
    with mp.get_context("spawn").Pool(processes) as pool:
        pool.map(_cpu_filter_worker, [(s, n_samples) for s in range(processes)])
    dt = time.perf_counter() - t0
    return processes * seconds_per_stream / 3600.0 / dt, dt


DUMP_BUDGET = 60 << 20        # bytes of sampled rows over all dumped arrays (the rest stays far below 64 MB)


def dump_outputs(out_dir, outputs):
    """Writes {name: tensor} as out_dir/<name>.npy: floating point as float32, integer counters as float64 (exact
    below 2**53).  A [rows, ...] array larger than its share of DUMP_BUDGET keeps a fixed seeded sample of rows
    (streams), whose indices go to out_dir/<name>_rows.npy, so that two builds are compared on the same rows."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BUDGET // max(1, sum(t.dim() >= 2 for t in outputs.values()))
    for name, t in outputs.items():
        a = t.detach()
        if a.dim() >= 2 and a.numel() * 4 > share:
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], max(1, share // (a[0].numel() * 4)), replace=False))
            a = a[torch.as_tensor(rows, device=a.device)]
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
        a = a.cpu().numpy()
        a = a.astype(np.float32) if np.issubdtype(a.dtype, np.floating) else a.astype(np.float64)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def config_dict(args, S, N):
    names = {"sweep": "config5-step: FAR/FRR sweep time-chunk, filter->encode->detect, CRNN + WaveNet, hop-2 windows",
             "crnn": "filter->encode->detect, CRNN, hop-2 windows", "wavenet": "filter->encode->detect, WaveNet, hop-2 windows",
             "filter": "config2: mel filterbank extraction only"}
    c = {"workload": names[args.workload], "sample_rate": 16000, "pcm": "int16", "hop_frames": 2,
         "precision": args.precision, "l2": "inputs larger than L2 (PCM batch > 126 MB)" if S and S * N * 2 > 126e6
         else "L2 flushed between steps"}
    if S:
        c.update({"streams_per_gpu": S, "seconds_per_stream": N / 16000.0})
    return c


# --------------------------------------------------------------------------------------- GPU arm
def bind_to_gpu_numa_node(torch, local):
    """Pins this process (and so its page-locked buffers, first-touch) to the NUMA node of its GPU: with eight ranks
    feeding eight GPUs the host->device copies otherwise cross the socket interconnect."""
    try:
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def make_pcm(synth, wake, S, N, seed, dev, first_stream):
    """One batch of device-generated PCM with the wake clip of every model spliced into a few streams."""
    import torch
    pcm = synth.device_pcm(S, N, seed=seed, device=dev, first_stream=first_stream)
    k = 0
    for sidx in sorted({0, S // 3, S // 2, S - 1}):
        for name, clip in wake.items():
            at = (k * 16000) % max(1, N - clip.numel())
            n = min(clip.numel(), N - at)
            if sidx + (0 if name == "crnn" else 1) < S and n > 0:
                pcm[sidx + (0 if name == "crnn" else 1), at:at + n] = clip[:n]
            k += 1
    return pcm


def parity_report(engines, models, pcm, post, thr, S):
    """extra.parity: the step's posteriors, decisions and counters against the CPU oracle on streams that carry wake
    clips and on a noise stream (outside the timed region; oracle = numpy restatement of the TFLite graphs)."""
    from oracle import restated as R
    out = {"windows_checked": 0, "max_abs_err": 0.0, "decision_flips_outside_band": 0, "decisions_fired": 0,
           "counters_equal": True, "counter_thresholds_differing": 0, "tolerance": 1e-3, "streams": []}
    streams = sorted({0, 1, S // 2, S // 2 + 1, 2})[:4]
    out["streams"] = streams
    for m in models:
        e = engines[m]
        w = e.weights
        L = int(w["mel_length"])
        ref_rows = []
        for sidx in streams:
            mel = R.mel_stream(R.int16_to_float(pcm[sidx].cpu().numpy()), w)
            j = np.arange(R.eval_windows(mel.shape[0], L))
            ref = R.posterior(mel[(2 * j)[:, None] + np.arange(L)[None, :]], w).astype(np.float32)
            got = post[m][sidx].cpu().numpy()
            err = np.abs(got - ref)
            band = np.abs(ref - 0.5) <= 1e-3
            out["windows_checked"] += int(j.size)
            out["max_abs_err"] = max(out["max_abs_err"], float(err.max()))
            out["decision_flips_outside_band"] += int(((got > 0.5) != (ref > 0.5))[~band].sum())
            out["decisions_fired"] += int((ref > 0.5).sum())
            ref_rows.append(ref)
        # counters of the checked streams: GPU kernel on the GPU posteriors vs the oracle's loops on the oracle posteriors
        sub = np.stack([post[m][sidx].cpu().numpy() for sidx in streams])
        seg = np.arange(len(streams) + 1, dtype=np.int64) * sub.shape[1]
        far = e.eval_counts(sub, seg, thr, "far_edges").cpu().numpy()
        frr = e.eval_counts(sub, seg, thr, "frr_max").cpu().numpy()
        far_ref = sum(np.array([R.rising_edges(R.smooth_same(r), t) for t in thr]) for r in ref_rows)
        frr_ref = np.array([sum(1 for r in ref_rows if r.max() > t) for t in thr])
        diff = int((far != far_ref).sum() + (frr != frr_ref).sum())
        out["counter_thresholds_differing"] += diff
        out["counters_equal"] = out["counters_equal"] and diff == 0
        out[m + "_far_edges_at_0.5"] = int(far[0])
        out[m + "_accepts_at_0.5"] = int(frr[0])
    return out


def extra_configs(torch, engines, dev, pk, precision):
    """Short measurements of BASELINE configs 2, 3 and 4 (CUDA events, inputs resident, >= 3 warm-up passes)."""
    from wakeword_detection_b200 import synth
    ev = lambda: torch.cuda.Event(enable_timing=True)
    out = {}

    def timed(fn, reps, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        a, b = ev(), ev()
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    crnn, wn = engines.get("CRNN"), engines.get("Wavenet")
    first = crnn or wn
    # config 2: mel filterbank extraction only, 100 000 clips x 2 s (6.4 GB of int16 PCM: larger than L2)
    S2, N2 = 100000, 32000
    pcm = synth.device_pcm(S2, N2, seed=77, device=dev)
    F2 = first.num_frames(N2)
    mel = torch.empty((S2, F2, 40), dtype=torch.float32, device=dev)
    ms = timed(lambda: first.filter(pcm, 0.0, out=mel), 5)
    gbs = S2 * F2 * BYTES_PER_FRAME / (ms / 1e3) / 1e9
    out["config2_filter"] = {"workload": "100000 clips x 2 s, mel extraction only", "ms_per_step": ms,
                             "audio_h_per_s": S2 * N2 / 16000.0 / 3600.0 / (ms / 1e3),
                             "roofline": {"bound": "hbm", "kernel": "filter_kernel", "achieved": gbs, "peak": pk["hbm_gbs"],
                                          "unit": "GB/s", "frac": gbs / pk["hbm_gbs"]},
                             "l2": "inputs larger than L2"}
    del pcm, mel
    torch.cuda.empty_cache()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    if crnn is not None:
        # config 3: 8192 independent [151, 40] windows per launch (per-window tiles: nothing is shared between windows)
        pcm3 = synth.device_pcm(64, 160 * 300 + 512, seed=3, device=dev)
        m3 = crnn.filter(pcm3)
        wins = m3.unfold(1, 151, 1).permute(0, 1, 3, 2)[:, :128].reshape(-1, 151, 40).contiguous()
        post3 = torch.empty((8192, 1), dtype=torch.float32, device=dev)

        def c3():
            flush.fill_(1)
            crnn.posteriors(wins, 1, out=post3)
        ms_all = timed(c3, 10)
        ms_flush = timed(lambda: flush.fill_(1), 10)
        ms = ms_all - ms_flush
        tf = 8192 * FLOP_PER_WINDOW["CRNN"] / (ms / 1e3) / 1e12
        out["config3_crnn_windows"] = {"workload": "8192 independent CRNN windows (wwb_posteriors, n_frames == L)", "ms_per_step": ms,
                                       "windows_per_s": 8192 / (ms / 1e3),
                                       "roofline": {"bound": "tensor", "kernel": "crnn encode+detect", "achieved": tf,
                                                    "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                                                    "frac": tf / pk["bf16_tflops_sustained"]},
                                       "l2": "flushed between steps (flush time subtracted)"}
    if wn is not None:
        # config 4: 4096 concurrent streams, every push brings 160 samples = one new mel frame per stream (hop 1) and
        # re-scores the stream's [182, 40] ring window; state (PCM tail, mel ring, posterior max) lives in HBM
        from wakeword_detection_b200 import _cabi
        e4 = _cabi.Engine(wn.weights, dev.index, precision)
        S4 = 4096
        e4.stream_alloc(S4, 160)
        pcm4 = synth.device_pcm(S4, 160 * 64, seed=9, device=dev)
        chunks = [pcm4[:, i * 160:(i + 1) * 160].contiguous() for i in range(64)]
        for c in chunks[:8]:
            e4.stream_push(c)
        state = {"i": 8}

        def c4():
            e4.stream_push(chunks[state["i"] % 64])
            state["i"] += 1
        ms = timed(c4, 48, warm=4)
        tf = S4 * FLOP_PER_WINDOW["Wavenet"] / (ms / 1e3) / 1e12
        out["config4_wavenet_streaming"] = {"workload": "4096 streams x 1 new frame per wwb_stream_push (hop 1)", "ms_per_step": ms,
                                            "pushes_per_s": 1e3 / ms, "stream_steps_per_s": S4 * 1e3 / ms,
                                            "audio_h_per_s": S4 * 0.01 / 3600.0 / (ms / 1e3),
                                            "roofline": {"bound": "tensor", "kernel": "wavenet encode+detect", "achieved": tf,
                                                         "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                                                         "frac": tf / pk["bf16_tflops_sustained"]},
                                            "l2": "working set 119 MB of mel rings + per-push PCM; no flush (streaming state is meant to stay hot)"}
        e4.close()
    return out


def cpu_config1_leg():
    """SURVEY 8(d) config 1, faithful call pattern: one 10 s stream pushed as 500 chunks of 320 samples through the
    WakewordTrigger state machine of the oracle, CRNN, batch 1, one thread: 997 mel frames -> 997 encode + detect."""
    from threadpoolctl import threadpool_limits
    from oracle import restated as R
    from wakeword_detection_b200 import synth, weights as W
    w = W.load_model_dir(os.path.join(ROOT, "weights", "CRNN"), "CRNN")
    pcm = synth.stream_int16(160000, 2, 11, 0)
    with threadpool_limits(limits=1):
        trig = R.TriggerOracle(w, threshold=2.0)
        t0 = time.perf_counter()
        for i in range(500):
            trig(pcm[i * 320:(i + 1) * 320], True)
        dt = time.perf_counter() - t0
    return {"audio_h_per_s": 10.0 / 3600.0 / dt, "seconds": dt, "invokes": len(trig.posteriors), "cores": 1, "kind": "port",
            "sample": "config 1: one 10 s stream, 500 x 320-sample frames through the trigger state machine, CRNN, batch 1"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="sweep", choices=["sweep", "filter", "crnn", "wavenet"])
    ap.add_argument("--streams", type=int, default=0, help="streams per GPU (0 = workload default)")
    ap.add_argument("--seconds", type=float, default=0.0, help="seconds per stream (0 = workload default)")
    ap.add_argument("--precision", default="tc", choices=["f32", "tc", "tc_fast"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip extra.configs / extra.parity (kernel work only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy; same arguments, same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        sys.stderr.write("bench.py: --warmup %d is below the 3 warm-up steps the timing rules require; using 3\n" % args.warmup)
        args.warmup = 3
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    from wakeword_detection_b200 import _cabi, weights as W, synth, dist as wdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(torch, local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    models = workload_models(args.workload)
    S, N = default_shape(args.workload, args)
    engines = {m: _cabi.Engine(W.load_model_dir(os.path.join(ROOT, "weights", m), m), local, args.precision)
               for m in (models or ["CRNN"])}
    first = next(iter(engines.values()))
    F = first.num_frames(N)
    nwin = {m: e.num_windows(F, 2) for m, e in engines.items()} if models else {}

    # three rotating batches: every step sees different PCM; wake clips make the counters non-zero
    wake = {k: torch.from_numpy(np.load(os.path.join(ROOT, "tests", "golden", "wake_%s_pcm.npy" % k))).to(dev)
            for k in ("crnn", "wavenet")} if models else {}
    NB = 3 if S * N * 2 <= 2e9 else 1
    pcm_dev = [make_pcm(synth, wake, S, N, 1234 + 7919 * i, dev, rank * S) for i in range(NB)]
    mel = torch.empty((S, F, 40), dtype=torch.float32, device=dev)
    post = {m: torch.empty((S, nwin[m]), dtype=torch.float32, device=dev) for m in models}
    thr = np.arange(0.5, 0.99999, 0.005)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if S * N * 2 <= 126e6 else None
    stage_ms = {"filter": 0.0, **{m: 0.0 for m in models}, "counts": 0.0}
    ev = lambda: torch.cuda.Event(enable_timing=True)
    step_no = {"i": 0}
    seg = {m: np.arange(S + 1, dtype=np.int64) * nwin[m] for m in models}

    def step(src, timed_stages=None):
        marks = [ev()]
        marks[0].record()
        first.filter(src, 0.0, out=mel)
        marks.append(ev()); marks[-1].record()
        counters = []
        for m in models:
            engines[m].posteriors(mel, 2, out=post[m])
            marks.append(ev()); marks[-1].record()
        for m in models:
            counters.append(engines[m].eval_counts(post[m], seg[m], thr, "far_edges"))
            counters.append(engines[m].eval_counts(post[m], seg[m], thr, "frr_max"))
        marks.append(ev()); marks[-1].record()
        if timed_stages is not None:
            timed_stages.append(marks)
        return counters

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(run, steps):
        sync_all()
        t0, t1 = ev(), ev()
        t0.record()
        for _ in range(steps):
            run()
        t1.record()
        sync_all()
        ms = torch.tensor([t0.elapsed_time(t1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    last_counters = {}

    def dev_step(stages=None):
        if flush is not None:
            flush.fill_(1)
        c = step(pcm_dev[step_no["i"] % NB], stages)
        step_no["i"] += 1
        if world > 1 and c:
            c = wdist.all_reduce_counters(*c)
        last_counters["c"] = c

    for _ in range(args.warmup):
        dev_step()
    launches0 = sum(e.launch_count() for e in engines.values())
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    stages = []
    try:
        total_ms = timed(lambda: dev_step(stages), args.steps)
    finally:
        clocks = sampler.stop() if rank == 0 else None       # never leave the nvidia-smi sampler running
    launches = sum(e.launch_count() for e in engines.values()) - launches0
    if args.dump_outputs and rank == 0:
        # before anything below reuses post / mel: posteriors and FAR / FRR counters per model (what
        # wwb_sweep_wait hands back), or the mel features of the filter-only workload
        outs = {m + "_posteriors": post[m] for m in models} if models else {"mel": mel}
        for k, m in enumerate(models):
            outs[m + "_far_edges"], outs[m + "_frr_accepts"] = last_counters["c"][2 * k:2 * k + 2]
        dump_outputs(args.dump_outputs, outs)
    for marks in stages:
        names = ["filter"] + models + ["counts"]
        for i, nme in enumerate(names):
            stage_ms[nme] += marks[i].elapsed_time(marks[i + 1])
    flush_ms = 0.0
    if flush is not None:      # the L2 flush is not part of the hot path: subtract its measured cost
        sync_all()
        a, b = ev(), ev()
        a.record()
        for _ in range(args.steps):
            flush.fill_(1)
        b.record()
        torch.cuda.synchronize()
        flush_ms = a.elapsed_time(b)
    ms_per_step = (total_ms - flush_ms) / args.steps
    audio_h = world * S * N / 16000.0 / 3600.0
    value = audio_h / (ms_per_step / 1e3)
    counters_dev = [int(x) for c in (last_counters.get("c") or []) for x in (c[0].item(), c[-1].item())]

    # ---------------- end to end through the host-buffer plugin call ----------------
    # PCM in page-locked numpy buffers (two, rotating) -> wwb_sweep_submit (ONE H2D copy + ONE filter pass feed every
    # model; two jobs in flight, so the copy of step k+1 overlaps the kernels of step k) -> wwb_sweep_wait (posteriors and
    # counters in host memory).  Timed with the host clock around the synchronous calls, barrier + device sync on both sides.
    elist = [engines[m] for m in models] or [first]
    e2e = None
    if models:
        host_pcm = []
        for i in range(2):
            h = _cabi.pinned_empty((S, N), np.int16)
            torch.from_numpy(h).copy_(pcm_dev[i % NB])
            host_pcm.append(h)
        recs = [None, None]

        def submit(i):
            recs[i % 2] = elist[0].sweep_submit(host_pcm[i % 2], 2, thr, others=elist[1:], out=recs[i % 2])

        def finish(i):
            elist[0].sweep_wait()
            r = recs[i % 2]
            if world > 1:
                t = torch.from_numpy(np.stack(r["far"] + r["frr"])).to(dev)
                dist.all_reduce(t)
                t.cpu()
            return r

        def e2e_run(steps):
            submit(0)
            for i in range(1, steps):
                submit(i)
                finish(i - 1)
            return finish(steps - 1)

        e2e_run(3)
        sync_all()
        t0 = time.perf_counter()
        last = e2e_run(args.steps)
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e_ms = float(dt.item()) * 1e3 / args.steps
        h2d = S * N * 2
        d2h = sum(S * nwin[m] * 4 for m in models) + len(models) * 2 * thr.size * 8
        # the host-call results of the last step equal the resident path's on the same PCM (same kernels)
        chk = step(pcm_dev[(args.steps - 1) % 2 % NB])
        torch.cuda.synchronize()
        same = all(np.array_equal(last["post"][k], post[m].cpu().numpy()) for k, m in enumerate(models))
        same = same and all(np.array_equal(last["far"][k], chk[2 * k].cpu().numpy()) and
                            np.array_equal(last["frr"][k], chk[2 * k + 1].cpu().numpy()) for k in range(len(models)))
        e2e = {"value": audio_h / (e2e_ms / 1e3), "unit": "audio-h/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "ms_per_step": e2e_ms, "api": "wwb_sweep_submit / wwb_sweep_wait (C ABI over ctypes, numpy host buffers, pinned)",
               "timer": "host clock around the synchronous calls, barrier + device sync on both sides, max over ranks",
               "equals_resident_path": bool(same), "numa_node": numa}
    else:
        # filter only: host PCM -> H2D -> filter -> first mel rows back (copy-bound: 6.4 GB of PCM per step)
        host = _cabi.pinned_empty((S, N), np.int16)
        torch.from_numpy(host).copy_(pcm_dev[0])
        stage = torch.empty_like(pcm_dev[0])
        th = torch.from_numpy(host)

        def fstep():
            stage.copy_(th, non_blocking=True)
            first.filter(stage, 0.0, out=mel)
            mel[:, :1].cpu()
        fstep()
        e2e_ms = timed(fstep, args.steps) / args.steps
        e2e = {"value": audio_h / (e2e_ms / 1e3), "unit": "audio-h/s", "h2d_bytes_per_step": S * N * 2,
               "d2h_bytes_per_step": S * 160, "ms_per_step": e2e_ms, "api": "Engine.filter on a staged copy", "numa_node": numa}

    pk, pk_src = peaks()
    per = {k: v / args.steps for k, v in stage_ms.items()}
    dom = max((k for k in per if k != "counts"), key=lambda k: per[k])
    if dom == "filter":
        ach = S * F * BYTES_PER_FRAME / (per[dom] / 1e3) / 1e9
        roof = {"bound": "hbm", "kernel": "filter_kernel", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": ach / pk["hbm_gbs"], "traffic": None}
    else:
        ach = S * nwin[dom] * FLOP_PER_WINDOW[dom] / (per[dom] / 1e3) / 1e12
        roof = {"bound": "tensor", "kernel": dom.lower() + " encode+detect", "achieved": ach,
                "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops_sustained"],
                "traffic": measured_traffic(dom.lower() + " encode+detect", S, N)}
    roof["peak_source"] = pk_src + (" (sustained bf16)" if dom != "filter" else " (copy)")
    extra = {"ms_per_stage": per,
             "filter_GBps": S * F * BYTES_PER_FRAME / (per["filter"] / 1e3) / 1e9,
             "filter_frac_of_hbm": S * F * BYTES_PER_FRAME / (per["filter"] / 1e3) / 1e9 / pk["hbm_gbs"],
             "pcm": "%d rotating device batches (counter-based seeds), wake clips spliced into 8 streams of each" % NB,
             "counters_first_last_threshold": counters_dev}
    for m in models:
        tf = S * nwin[m] * FLOP_PER_WINDOW[m] / (per[m] / 1e3) / 1e12
        extra[m + "_TFLOPs"] = tf
        extra[m + "_frac_of_tensor"] = tf / pk["bf16_tflops_sustained"]
        extra[m + "_windows_per_step"] = S * nwin[m]
    if "CRNN" in models and args.precision != "f32" and nwin["CRNN"] > 72:
        # Sliding windows share the conv + GRU-1 projection columns (crnn_tc.cu, CrnnShare): the figures above use the
        # ALGORITHMIC flops of the per-window formulation; these are the flops the kernels execute.
        q = 4                                                     # hop 2: position indices per conv step
        nsp = -(-((nwin["CRNN"] - 1 + 18 * q) // q + 1) // 126)   # strips of 126 conv steps per stream and phase
        cols = 3 * q * nsp * 126                                  # interior + two padded-column variants
        exe = cols * (2432000 + 4669440) / 19.0 / nwin["CRNN"] + 2 * 233472 + 466944 + 8320
        extra["CRNN_shared_columns"] = {"executed_flop_per_window": exe,
                                        "executed_TFLOPs": S * nwin["CRNN"] * exe / (per["CRNN"] / 1e3) / 1e12,
                                        "columns_per_window": cols / nwin["CRNN"]}
    if "Wavenet" in models and args.precision != "f32" and nwin["Wavenet"] >= 8:
        # Sliding windows take every activation outside the causal-padding cone from a stream-level pass
        # (wavenet_tc.cu): groups of 4 windows = 6 tiles of 128 time-major rows, tile i joins at the first block whose
        # padding-dependent prefix D(b) = sum 2*dilation reaches its first time step; the stream pass runs all 24 blocks
        # on chunks of 768 frames that advance by 588.  Fraction = executed rows x blocks / (182 x 24) per window.
        G, NT, L_wn = 4, 6, 182
        D = np.cumsum(2 * np.tile([1, 2, 4, 8], 6))
        tile_blocks = sum(24 - int(np.argmax(D > (128 * i) // G)) for i in range(NT))          # 76
        frac = (tile_blocks * 128.0 / G + (F / (NT * 128.0 - 180.0)) * NT * 24 * 128.0 / nwin["Wavenet"]) / (L_wn * 24.0)
        exe = FLOP_PER_WINDOW["Wavenet"] * frac
        extra["Wavenet_shared_activations"] = {"executed_fraction_of_row_blocks": frac,
                                               "executed_TFLOPs": S * nwin["Wavenet"] * exe / (per["Wavenet"] / 1e3) / 1e12}

    if rank == 0 and models and not args.no_extras:
        step(pcm_dev[0])                     # (no collective here: the other ranks are not in this branch)
        torch.cuda.synchronize()
        extra["parity"] = parity_report(engines, models, pcm_dev[0], post, thr, S)
    if rank == 0 and not args.no_extras and args.workload == "sweep":
        del pcm_dev
        torch.cuda.empty_cache()
        extra["configs"] = extra_configs(torch, engines, dev, pk, args.precision)

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline:
            cm = models or ["CRNN"]
            if args.workload == "filter":
                r, dt = cpu_filter_rate(1, 1800.0)
                cpu = {"value": r, "unit": "audio-h/s", "cores": 1, "kind": "port",
                       "sample": "1 stream x 1800 s, filter only, numpy restatement, 1 thread (%.1f s)" % dt}
            else:
                sec = 120.0 * (2.0 / len(cm)) if cm else 120.0
                r, dt = cpu_reference_rate(cm, 1, sec, 1)
                cpu = {"value": r, "unit": "audio-h/s", "cores": 1, "kind": "port",
                       "sample": "1 stream x %.0f s through %s, numpy restatement of the TFLite graphs, 1 thread (%.1f s)"
                                 % (sec, "+".join(cm), dt)}
                if not args.no_extras:
                    extra["cpu_config1_batch1"] = cpu_config1_leg()
        line = {"metric": "audio_hours_per_sec", "value": value, "unit": "audio-h/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32" if args.precision == "f32" else "f16x2->f32",
                "data": "synthetic", "config": config_dict(args, S, N), "clocks": clocks,
                "e2e": e2e, "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu, "extra": extra}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

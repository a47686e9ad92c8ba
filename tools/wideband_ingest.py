#!/usr/bin/env python
"""Many wideband captures through one channelizer: what batching the captures buys.

Usage: python tools/wideband_ingest.py OUT_DIR [--steps K] [--reps R] [--only a|b]

Writes OUT_DIR/wideband_ingest.jsonl, one JSON line per workload, each with the card name, power
limit and maximum SM clock read (nvidia-smi, read-only) in the same run. One step is 68 ms of
signal per capture: two 8192-sample blocks at 240 kS/s.

  (a) sites:   W in {1, 8, 32} captures of 24 MS/s, 100 carriers at 200 kHz, D = 100
  (b) dongles: W in {64, 256, 800} captures of 2.4 MS/s, 12 carriers at 200 kHz, D = 10,
               16 taps per phase, each tuned elsewhere: first carrier offset c0 alternates
               between -5.5 and -5.25 spacings (-5.0 would put carrier 11 on Nyquist)

Per workload:
  channelizer   the stage alone on one stream, device events: one multi-capture object
                (fmgpu_channelizer_process_multi) against W single-capture objects, alternated
                rep by rep; also the host time to enqueue one step through the Python wrapper
  full_step     pinned host [W][stride] -> device on a copy stream (torch copy_, double-buffered)
                -> process_multi -> fmgpu_process_batch_cf32 on W * C channels -> audio back to
                pinned host; ms per step, real-time factor, real-time captures per GPU, and H2D
                GB/s against a bare copy of the same buffers measured in the same run

Inputs are seeded random bytes generated on the device. Needs a CUDA device: without one it fails.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BLOCK, B = 8192, 2
SP = 200_000.0
WORKLOADS = [("a", "sites", w, 24_000_000, 100, 100, [-49.5]) for w in (1, 8, 32)] + \
            [("b", "dongles", w, 2_400_000, 10, 12, [-5.5, -5.25]) for w in (64, 256, 800)]


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    return {"nvidia_smi": out}


def ev():
    import torch
    return torch.cuda.Event(enable_timing=True)


def run_workload(fm, torch, kind, W, wide, D, Cn, c0s, steps, reps, seed):
    dev = torch.device("cuda", 0)
    n_in = B * BLOCK * D                       # pairs per capture per step
    stride = 2 * n_in
    n_dsp = B * BLOCK
    firsts = [c0s[w % len(c0s)] * SP for w in range(W)]
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    iq = torch.randint(0, 256, (W, stride), dtype=torch.uint8, device=dev, generator=g)
    s = torch.cuda.Stream()
    sp = s.cuda_stream
    zkw = dict(wide_rate=wide, decimation=D, n_channels=Cn, spacing_hz=SP, taps_per_phase=16,
               cutoff_hz=100_000.0)
    zm = fm.Channelizer(first_center_hz=firsts, **zkw)
    zs = [fm.Channelizer(first_center_hz=f, **zkw) for f in firsts]
    out_m = torch.zeros((W * Cn, n_dsp, 2), dtype=torch.float32, device=dev)
    out_s = torch.zeros_like(out_m)

    def multi():
        zm.process(iq.data_ptr(), n_in, out_m.data_ptr(), n_dsp, stream=sp, iq_stride_bytes=stride)

    def singles():
        for w, z in enumerate(zs):
            z.process(iq[w].data_ptr(), n_in, out_s[w * Cn].data_ptr(), n_dsp, stream=sp)

    def timed(fn):
        e0, e1 = ev(), ev()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record(s)
        for _ in range(steps):
            fn()
        t1 = time.perf_counter()
        e1.record(s)
        e1.synchronize()
        return e0.elapsed_time(e1) / steps, (t1 - t0) / steps * 1e6

    for _ in range(2):                          # warm-up; both sides see the same calls
        multi()
        singles()
    res = {"multi": [], "singles": []}
    for _ in range(reps):
        res["multi"].append(timed(multi))
        res["singles"].append(timed(singles))
    torch.cuda.synchronize()
    same = bool(torch.equal(out_m, out_s))
    del zs, out_s

    def summary(v):
        ms = [x[0] for x in v]
        us = [x[1] for x in v]
        return {"ms_per_step_median": statistics.median(ms), "ms_per_step_min": min(ms),
                "ms_per_step_max": max(ms), "host_enqueue_us_per_step_median": statistics.median(us)}

    chan = {"multi": summary(res["multi"]), "singles": summary(res["singles"]),
            "launches_per_step": {"multi": 2, "singles": 2 * W},
            "outputs_equal": same}
    chan["singles_over_multi"] = chan["singles"]["ms_per_step_median"] / chan["multi"]["ms_per_step_median"]

    # full step
    nch = W * Cn
    eng = fm.Engine(fm.make_config(iq_rate=240_000, decimation=1, max_blocks=B), nch, 0)
    acap = eng.audio_capacity(B)
    audio = torch.empty((nch, 2, acap), dtype=torch.float32, device=dev)
    n_audio = torch.zeros(nch, dtype=torch.int32, device=dev)
    status = torch.zeros((nch, B, 20), dtype=torch.uint8, device=dev)
    iq_host = torch.empty((W, stride), dtype=torch.uint8).pin_memory()
    iq_host.copy_(iq)
    audio_host = torch.empty((nch, 2, acap), dtype=torch.float32).pin_memory()
    n_audio_host = torch.zeros(nch, dtype=torch.int32).pin_memory()
    bufs = [iq, torch.empty_like(iq)]
    cs = torch.cuda.Stream()
    copied = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    h2d = [(ev(), ev()) for _ in range(steps)]

    def full(k, rec=None):
        i = k & 1
        with torch.cuda.stream(cs):
            cs.wait_event(consumed[i])
            if rec:
                rec[0].record(cs)
            bufs[i].copy_(iq_host, non_blocking=True)
            if rec:
                rec[1].record(cs)
            copied[i].record(cs)
        s.wait_event(copied[i])
        zm.process(bufs[i].data_ptr(), n_in, out_m.data_ptr(), n_dsp, stream=sp, iq_stride_bytes=stride)
        consumed[i].record(s)
        eng.process_batch_cf32(out_m.data_ptr(), n_dsp, B, audio.data_ptr(), acap, n_audio.data_ptr(),
                               None, B + 8, None, status.data_ptr(), sp)
        with torch.cuda.stream(s):
            audio_host.copy_(audio, non_blocking=True)
            n_audio_host.copy_(n_audio, non_blocking=True)

    for k in range(3):
        full(k)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(steps):
        full(k, h2d[k])
    torch.cuda.synchronize()
    step_ms = (time.perf_counter() - t0) / steps * 1e3
    h2d_ms = statistics.median(a.elapsed_time(b) for a, b in h2d)
    # bare copy of the same buffers, nothing else running
    e0, e1 = ev(), ev()
    with torch.cuda.stream(cs):
        e0.record(cs)
        for k in range(steps):
            bufs[k & 1].copy_(iq_host, non_blocking=True)
        e1.record(cs)
    torch.cuda.synchronize()
    bare_ms = e0.elapsed_time(e1) / steps
    eng.close()
    zm.close()
    sig_s = n_dsp / 240_000.0
    nbytes = W * stride
    rtf = sig_s / (step_ms * 1e-3)
    full_rec = {"ms_per_step": step_ms, "realtime_factor": rtf, "realtime_captures_per_gpu": W * rtf,
                "h2d_bytes_per_step": nbytes, "h2d_gbs_in_step": nbytes / (h2d_ms * 1e-3) / 1e9,
                "h2d_gbs_bare_copy": nbytes / (bare_ms * 1e-3) / 1e9}
    return {"workload": kind, "captures": W, "wide_rate": wide, "decimation": D, "carriers_per_capture": Cn,
            "c0": c0s, "taps": D * 16, "steps": steps, "reps": reps, "signal_ms_per_step": sig_s * 1e3,
            "channelizer": chan, "full_step": full_rec}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", choices=["a", "b"])
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("wideband_ingest: no CUDA device; this script only measures on the GPU")
    import fmtuner_sdr_b200 as fm
    info = card()
    os.makedirs(args.out_dir, exist_ok=True)
    path = os.path.join(args.out_dir, "wideband_ingest.jsonl")
    with open(path, "w") as f:
        for i, (tag, kind, W, wide, D, Cn, c0s) in enumerate(WORKLOADS):
            if args.only and tag != args.only:
                continue
            rec = run_workload(fm, torch, kind, W, wide, D, Cn, c0s, args.steps, args.reps, seed=1000 + i)
            rec["card"] = info
            line = json.dumps(rec)
            print(line, flush=True)
            f.write(line + "\n")
            f.flush()


if __name__ == "__main__":
    main()

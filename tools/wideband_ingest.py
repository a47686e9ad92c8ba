#!/usr/bin/env python
"""Many wideband captures through one channelizer: what batching the captures buys.

Usage: python tools/wideband_ingest.py OUT_DIR [--steps K] [--reps R] [--only a|b|formats|rational]

Writes OUT_DIR/wideband_ingest.jsonl, one JSON line per workload (the formats workload runs only
with --only formats and writes OUT_DIR/wideband_formats.jsonl; the rational workloads run only with
--only rational and write OUT_DIR/wideband_rational.jsonl), each with the card name, power
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

  (formats) 32 captures of 24 MS/s, 100 carriers, D = 100, as cu8, cs8 and cs16 objects
             (fmgpu_channelizer_create_format) on inputs of the same number of pairs (cs16: twice
             the bytes): the channelizer stage alone, formats alternated rep by rep, and the full
             step above for each format, reps alternated the same way, through one engine

  (rational) 32 captures each, through fmgpu_channelizer_create_rate / _process_stream, with the
             same 16384 output instants per step (the pairs per step vary where U > 1):
               20 MS/s cs8  -> 240 kS/s (U = 3, D = 250), 100 carriers
               24 MS/s cs8  -> 240 kS/s (U = 1, D = 100), 100 carriers
               10 MS/s cs16 -> 256 kS/s (U = 16, D = 625), 50 carriers
             the channelizer stage alone and the full step above, workloads alternated rep by rep

Inputs are seeded random samples generated on the device. Needs a CUDA device: without one it fails.
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

    eng = FullStep(fm, torch, W * Cn, s)
    full_rec = eng.run(zm, iq, n_in, out_m, steps)
    eng.close()
    zm.close()
    return {"workload": kind, "captures": W, "wide_rate": wide, "decimation": D, "carriers_per_capture": Cn,
            "c0": c0s, "taps": D * 16, "steps": steps, "reps": reps, "signal_ms_per_step": n_dsp / 240.0,
            "channelizer": chan, "full_step": full_rec}


class FullStep:
    """pinned host [W][stride] -> device (copy stream, double-buffered) -> channelizer -> engine of
    nch channels -> audio back to pinned host, on stream s."""

    def __init__(self, fm, torch, nch, s):
        self.torch, self.s, self.nch = torch, s, nch
        dev = torch.device("cuda", 0)
        self.eng = fm.Engine(fm.make_config(iq_rate=240_000, decimation=1, max_blocks=B), nch, 0)
        self.acap = self.eng.audio_capacity(B)
        self.audio = torch.empty((nch, 2, self.acap), dtype=torch.float32, device=dev)
        self.n_audio = torch.zeros(nch, dtype=torch.int32, device=dev)
        self.status = torch.zeros((nch, B, 20), dtype=torch.uint8, device=dev)
        self.audio_host = torch.empty((nch, 2, self.acap), dtype=torch.float32).pin_memory()
        self.n_audio_host = torch.zeros(nch, dtype=torch.int32).pin_memory()

    def close(self):
        self.eng.close()

    def run(self, zm, iq, n_in, out_m, steps):
        """iq [W][stride] on the device, the input of zm; its copy in pinned host memory is the source."""
        torch, s, eng = self.torch, self.s, self.eng
        sp = s.cuda_stream
        n_dsp = B * BLOCK
        W = iq.shape[0]
        stride = iq[0].numel() * iq.element_size()
        acap, audio, n_audio, status = self.acap, self.audio, self.n_audio, self.status
        audio_host, n_audio_host = self.audio_host, self.n_audio_host
        iq_host = torch.empty_like(iq, device="cpu").pin_memory()
        iq_host.copy_(iq)
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
        sig_s = n_dsp / 240_000.0
        nbytes = W * stride
        rtf = sig_s / (step_ms * 1e-3)
        return {"ms_per_step": step_ms, "realtime_factor": rtf, "realtime_captures_per_gpu": W * rtf,
                "h2d_bytes_per_step": nbytes, "h2d_gbs_in_step": nbytes / (h2d_ms * 1e-3) / 1e9,
                "h2d_gbs_bare_copy": nbytes / (bare_ms * 1e-3) / 1e9}


def run_formats(fm, torch, steps, reps, seed):
    """32 full-band sites as cu8, cs8 and cs16 captures of the same number of pairs."""
    W, wide, D, Cn = 32, 24_000_000, 100, 100
    dev = torch.device("cuda", 0)
    n_in = B * BLOCK * D
    n_dsp = B * BLOCK
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    iq = {"cu8": torch.randint(0, 256, (W, 2 * n_in), dtype=torch.uint8, device=dev, generator=g),
          "cs8": torch.randint(-128, 128, (W, 2 * n_in), dtype=torch.int8, device=dev, generator=g),
          "cs16": torch.randint(-32768, 32768, (W, 2 * n_in), dtype=torch.int16, device=dev, generator=g)}
    s = torch.cuda.Stream()
    sp = s.cuda_stream
    firsts = [-49.5 * SP] * W
    zs = {f: fm.Channelizer(first_center_hz=firsts, wide_rate=wide, decimation=D, n_channels=Cn, spacing_hz=SP,
                            taps_per_phase=16, cutoff_hz=100_000.0, sample_format=f) for f in iq}
    out = torch.zeros((W * Cn, n_dsp, 2), dtype=torch.float32, device=dev)

    def timed(f):
        z, x = zs[f], iq[f]
        e0, e1 = ev(), ev()
        torch.cuda.synchronize()
        e0.record(s)
        for _ in range(steps):
            z.process(x.data_ptr(), n_in, out.data_ptr(), n_dsp, stream=sp)
        e1.record(s)
        e1.synchronize()
        return e0.elapsed_time(e1) / steps

    for f in iq:                                # warm-up
        for _ in range(2):
            zs[f].process(iq[f].data_ptr(), n_in, out.data_ptr(), n_dsp, stream=sp)
    chan = {f: [] for f in iq}
    for _ in range(reps):
        for f in iq:
            chan[f].append(timed(f))
    eng = FullStep(fm, torch, W * Cn, s)
    full = {f: [] for f in iq}
    for _ in range(reps):
        for f in iq:
            full[f].append(eng.run(zs[f], iq[f], n_in, out, steps))
    eng.close()
    for z in zs.values():
        z.close()
    rec = {"workload": "formats", "captures": W, "wide_rate": wide, "decimation": D, "carriers_per_capture": Cn,
           "c0": [-49.5], "taps": D * 16, "form": "polyphase", "pairs_per_capture_per_step": n_in,
           "steps": steps, "reps": reps, "signal_ms_per_step": n_dsp / 240.0, "formats": {}}
    for f in iq:
        ms = chan[f]
        fs = sorted(full[f], key=lambda r: r["ms_per_step"])
        med = fs[len(fs) // 2]
        rec["formats"][f] = {
            "pair_bytes": iq[f].element_size() * 2,
            "channelizer": {"ms_per_step_median": statistics.median(ms), "ms_per_step_min": min(ms),
                            "ms_per_step_max": max(ms)},
            "full_step": dict(med, ms_per_step_min=fs[0]["ms_per_step"], ms_per_step_max=fs[-1]["ms_per_step"])}
    return rec


RATIONAL = [("20M_cs8_240k", 20_000_000, 240_000, 100, "cs8"), ("24M_cs8_240k", 24_000_000, 240_000, 100, "cs8"),
            ("10M_cs16_256k", 10_000_000, 256_000, 50, "cs16")]


class StreamSteps:
    """A rational-rate object behind FullStep's process() call: step k feeds the pairs that complete
    exactly B * BLOCK more outputs per row (fmgpu_channelizer_process_stream)."""

    def __init__(self, z):
        self.z, self.k = z, 0
        U, D, n_dsp = z.interpolation, z.decimation, B * BLOCK
        # smallest T with ceil(T U / D) >= m outputs: floor((m - 1) D / U) + 1
        self.need = lambda m: ((m - 1) * D) // U + 1
        self.max_in = max(self.need((k + 1) * n_dsp) - self.need(k * n_dsp) for k in range(1, 2 * U + 2))
        self.T = 0

    def process(self, iq_ptr, n_in, out_ptr, n_dsp, stream=None, iq_stride_bytes=None):
        n = self.need((self.k + 1) * n_dsp) - self.T
        got = self.z.process_stream(iq_ptr, n, out_ptr, n_dsp, stream=stream, iq_stride_bytes=iq_stride_bytes)
        assert got == n_dsp, (got, n_dsp)
        self.k += 1
        self.T += n


def run_rational(fm, torch, steps, reps, seed):
    W = 32
    dev = torch.device("cuda", 0)
    n_dsp = B * BLOCK
    s = torch.cuda.Stream()
    sp = s.cuda_stream
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    objs, iq = {}, {}
    for name, wide, out_rate, Cn, fmt in RATIONAL:
        c0 = -(Cn - 1) / 2.0
        z = fm.Channelizer(wide_rate=wide, output_rate=out_rate, n_channels=Cn, first_center_hz=[c0 * SP] * W,
                           spacing_hz=SP, taps_per_phase=16, cutoff_hz=100_000.0, sample_format=fmt)
        objs[name] = StreamSteps(z)
        row = 2 * objs[name].max_in
        iq[name] = (torch.randint(-128, 128, (W, row), dtype=torch.int8, device=dev, generator=g) if fmt == "cs8" else
                    torch.randint(-32768, 32768, (W, row), dtype=torch.int16, device=dev, generator=g))
    Cmax = max(r[3] for r in RATIONAL)
    out = torch.zeros((W * Cmax, n_dsp, 2), dtype=torch.float32, device=dev)

    def timed(name):
        st, x = objs[name], iq[name]
        stride = x[0].numel() * x.element_size()
        e0, e1 = ev(), ev()
        torch.cuda.synchronize()
        e0.record(s)
        for _ in range(steps):
            st.process(x.data_ptr(), None, out.data_ptr(), n_dsp, stream=sp, iq_stride_bytes=stride)
        e1.record(s)
        e1.synchronize()
        return e0.elapsed_time(e1) / steps

    for name in objs:                           # warm-up
        for _ in range(2):
            timed(name)
    chan = {name: [] for name in objs}
    for _ in range(reps):
        for name in objs:
            chan[name].append(timed(name))
    full = {name: [] for name in objs}
    engs = {Cn: FullStep(fm, torch, W * Cn, s) for Cn in sorted({r[3] for r in RATIONAL})}
    for _ in range(reps):
        for name, wide, out_rate, Cn, fmt in RATIONAL:
            full[name].append(engs[Cn].run(objs[name], iq[name], None, out, steps))
    for e in engs.values():
        e.close()
    rec = {"workload": "rational", "captures": W, "taps_per_phase": 16, "form": "polyphase", "steps": steps,
           "reps": reps, "outputs_per_row_per_step": n_dsp, "workloads": {}}
    for name, wide, out_rate, Cn, fmt in RATIONAL:
        z = objs[name].z
        U, D = z.interpolation, z.decimation
        Lin = -(-D * 16 // U)
        ms = chan[name]
        fs = sorted(full[name], key=lambda r: r["ms_per_step"])
        med = fs[len(fs) // 2]
        rtf = n_dsp / out_rate / (med["ms_per_step"] * 1e-3)    # FullStep assumes 240 kS/s
        rec["workloads"][name] = {
            "wide_rate": wide, "output_rate": out_rate, "U": U, "D": D, "carriers_per_capture": Cn,
            "sample_format": fmt, "P": int(wide // SP), "Lin": Lin, "pairs_per_capture_per_step": n_dsp * D / U,
            "signal_ms_per_step": n_dsp / out_rate * 1e3,
            "channelizer": {"ms_per_step_median": statistics.median(ms), "ms_per_step_min": min(ms),
                            "ms_per_step_max": max(ms)},
            "full_step": dict(med, realtime_factor=rtf, realtime_captures_per_gpu=W * rtf,
                              ms_per_step_min=fs[0]["ms_per_step"], ms_per_step_max=fs[-1]["ms_per_step"])}
        z.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", choices=["a", "b", "formats", "rational"])
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("wideband_ingest: no CUDA device; this script only measures on the GPU")
    import fmtuner_sdr_b200 as fm
    info = card()
    os.makedirs(args.out_dir, exist_ok=True)
    if args.only == "formats":
        rec = run_formats(fm, torch, args.steps, args.reps, seed=2000)
        rec["card"] = info
        line = json.dumps(rec)
        print(line, flush=True)
        with open(os.path.join(args.out_dir, "wideband_formats.jsonl"), "w") as f:
            f.write(line + "\n")
        return
    if args.only == "rational":
        rec = run_rational(fm, torch, args.steps, args.reps, seed=3000)
        rec["card"] = info
        line = json.dumps(rec)
        print(line, flush=True)
        with open(os.path.join(args.out_dir, "wideband_rational.jsonl"), "w") as f:
            f.write(line + "\n")
        return
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

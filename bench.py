#!/usr/bin/env python
"""bench.py — throughput of the IQ -> audio + RDS hot path on N B200s of one node.

Metric (BASELINE.json): aggregate IQ MS/s demodulated (stereo + RDS); real-time channel
count = value / 2.4. One "step" = one pass of the whole pipeline (decimate, discriminate,
pilot PLL + stereo matrix, 15 kHz low-pass, resample to 32 kHz, de-emphasis, RDS down to
groups) over `blocks` logical blocks (8192 samples @ 240 kHz each) of every channel.

Workload: BASELINE config 5 — the 10,000-channel weak-signal sweep — resident on ONE GPU
(it fits: 3.3 GB of IQ per step), weak-scaled to N GPUs (channels-per-GPU fixed, every rank a
differently seeded sweep): 2.4 MS/s uint8 IQ / 10 -> 240 kHz, SNR 10-40 dB, blend mode c%3,
dsp_agc fast, synthetic multiplexes generated on the device from per-channel seeds. Channels
are independent: they are sharded across ranks with no collective on the data path.

  value    IQ samples/s with inputs resident in HBM (CUDA events, max over ranks)
  e2e      same metric through the C-ABI host call (pinned host IQ in, audio/groups/status out),
           with h2d_roof_gbs: a bare concurrent cudaMemcpyAsync of the same pinned buffers on every
           rank, i.e. what the box's PCIe / host memory gives this many ranks at once
  roofline the dominant THROUGHPUT-bound kernel against the roof that binds it — the measured HBM
           copy bandwidth (MEASURED_PEAKS.json) or the FP32 FMA rate measured in this run
           (fmgpu_measure_fp32_tflops) — plus every stage's figures and the dominant latency-bound
           (one lane per channel) kernel, which has no roofline fraction (SURVEY 8(d))
  stage_ms every stage's kernels alone on one stream
  strong   the north-star split: 10,000 channels in total dealt over the N ranks, 4 blocks per step
  config4  BASELINE config 4: one 24 MS/s capture -> channelizer (this rank's channels) -> the
           complex-float batch path, 100 channels dealt over the N ranks
  cpu_baseline / --impl reference: the reference's own sources (oracle/_ref/libfmref.so: its
           unmodified FMDemod / StereoDecoder / AFPostProcessor / RDSDecoder / redsea code over
           the liquid shim) on the host cores, one channel per thread; kind "reference". Falls
           back to the restated oracle (kind "port") when that library was not built.
Multi-GPU runs give every rank NVML's ideal CPU affinity for its GPU before pinned host memory
is allocated; a rank that cannot pin its buffers takes the e2e leg off for all ranks.
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

# the engine drives up to 3 streams per pipeline group: give them their own hardware queues
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

IQ_RATE = 2_400_000
DECIM = 10
BLOCK = 8192
BYTES_PER_IQ_SAMPLE_ALG = 2.0 + 8.0 * 32000.0 / IQ_RATE   # SURVEY §8(d): 2.107 B
FLOP_PER_IQ_SAMPLE_ALG = 269.0                            # SURVEY §8(d)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--channels", type=int, default=10000, help="channels per GPU")
    ap.add_argument("--blocks", type=int, default=2, help="logical blocks per step")
    ap.add_argument("--groups", type=int, default=1, help="channel ranges with their own set of stage streams (1 or 2)")
    ap.add_argument("--sync-steps", action="store_true",
                    help="join every step on the caller's stream (fmgpu_process_batch) instead of "
                         "streaming the steps (fmgpu_process_batch_async + one fmgpu_join)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--decim-mode", default="tc", choices=["tc", "fp32"],
                    help="arithmetic: tc = the engine's fast forms (tcgen05 int8 decimator, "
                         "fmgpu_set_decimator_mode 1; de-emphasis / DC blocker as a warp-shuffle scan, "
                         "fmgpu_set_scan_mode 1; pilot band-pass and L/R low-pass as tcgen05 int8 "
                         "contractions, fmgpu_set_fir_mode 1; channel filter + discriminator fused into one "
                         "tensor-core kernel, AGC elided, fmgpu_set_demod_mode 1); fp32 = the reference's "
                         "summation order everywhere, "
                         "bit-identical to the CPU oracle (modes 0)")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the strong-scaling, config-4 and H2D-roof records")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (audio, frame and group counts, groups "
                         "and block status of a fixed sample of rank 0's channels) to DIR/<name>.npy")
    return ap.parse_args()


# --------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                clk, mx = float(f[1]), float(f[2])
            except ValueError:
                continue
            smax = mx
            if t0 - 0.05 <= ts <= t1 + 0.15:
                sm.append(clk)
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                      "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        if not sm:
            sm = [float(l.split(",")[1]) for _, l in self.lines[-3:] if len(l.split(",")) > 2] or [0.0]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------
# CPU arm: the oracle on the host cores (one channel per thread)
# --------------------------------------------------------------------------------------
def cpu_arm(iq_rows, n_blocks_per_pass: int, passes: int, threads: int):
    """Each thread decodes its own channel: `passes` passes over its n_blocks_per_pass blocks.
    Returns (IQ samples processed in total, wall seconds)."""
    from oracle import orc
    lib = orc.OracleLib(cpu_flavour())
    chans = [orc.Channel(lib, orc.make_config(iq_rate=IQ_RATE, decimation=DECIM, dsp_agc=1,
                                              stereo_blend=c % 3)) for c in range(threads)]

    def work(i):
        for _ in range(passes):
            chans[i].process(iq_rows[i % len(iq_rows)])

    ths = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
    t0 = time.perf_counter()
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    return threads * passes * n_blocks_per_pass * BLOCK * DECIM, dt


def cpu_flavour() -> str:
    """The reference's own code when oracle/_ref/libfmref.so exists, else the restated oracle."""
    from oracle import orc
    return "ref" if orc.OracleLib.have_ref("ref") else "libm"


def cpu_kind() -> dict:
    if cpu_flavour() == "ref":
        return {"kind": "reference",
                "note": "the reference's unmodified fm_demod / stereo_decoder / af_post_processor / "
                        "rds_decoder / redsea_port sources (oracle/_ref/libfmref.so, -O3 -mavx2 -mfma "
                        "-ffp-contract=off) over oracle/liquid_shim; liquid-dsp itself is not "
                        "installable here, its objects are the restatement in oracle/liquid_restated.hpp"}
    return {"kind": "port", "note": "restated reference pipeline (oracle, libm flavour): "
                                    "oracle/_ref/libfmref.so was not built"}


def host_signals(n_channels: int, n_blocks: int):
    """config-5-style channels from the oracle-side generator (CPU arm input)."""
    import numpy as np
    from oracle import orc
    rows = [None] * n_channels

    def gen(c):
        s = orc.config3_signal(c, fs_iq=IQ_RATE)
        s.snr_db = 10.0 + 30.0 * ((c * 37) % 100) / 100.0
        rows[c] = s.generate(n_blocks * BLOCK * DECIM)

    ths = [threading.Thread(target=gen, args=(c,)) for c in range(n_channels)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    return np.stack(rows)


def run_reference(args, rank: int):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    threads = cores
    iq = host_signals(min(threads, 16), args.blocks)
    # one step = every thread decodes PASSES x `blocks` logical blocks of its own channel (a
    # bounded sample of the 10,000-channel workload: one channel per host thread)
    passes = 8
    for _ in range(max(1, args.warmup)):
        cpu_arm(iq, args.blocks, 1, threads)
    samples, dt = 0, 0.0
    for _ in range(args.steps):
        s, d = cpu_arm(iq, args.blocks, passes, threads)   # d: the threads' decode time only (not the
        samples += s                                        # construction of the pipeline objects)
        dt += d
    value = samples / dt / 1e6
    sample_desc = (f"{threads} channels x {passes} passes x {args.blocks} blocks x {BLOCK * DECIM} IQ "
                   f"samples per step, {args.steps} steps, one channel per thread")
    line = {
        "impl": "reference", "metric": "aggregate IQ MS/s demodulated (stereo+RDS)", "value": value,
        "unit": "MS/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "realtime_channels": value * 1e6 / IQ_RATE,
        "config": workload_config(args, threads),
        "cpu_baseline": {"value": value, "unit": "MS/s", "cores": threads, "sample": sample_desc,
                         **cpu_kind()},
        "e2e": {"value": value, "unit": "MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, channels_this_arm: int) -> dict:
    return {
        "workload": "BASELINE config 5 (10,000-channel weak-signal sweep) per GPU, sharded by "
                    f"channel: {args.channels} channels/GPU, 2.4 MS/s uint8 IQ /10 -> 240 kHz, "
                    "SNR 10-40 dB, blend soft/normal/aggressive by c%3, dsp_agc fast, stereo + RDS",
        "channels_per_gpu": args.channels, "blocks_per_step": args.blocks,
        "pipeline_groups": args.groups,
        "arithmetic": ("fast forms where they exist: decimator = tcgen05 int8 contraction, TMA-fed, "
                       "accumulators in TMEM (decim_tc.cu, fmgpu_set_decimator_mode 1); de-emphasis + DC "
                       "blocker = warp-shuffle scan (fmgpu_set_scan_mode 1); pilot band-pass + L/R low-pass = "
                       "tcgen05 int8 contractions on 24-bit fixed-point samples, A operand in TMEM (fir_tc.cu, "
                       "fmgpu_set_fir_mode 1); channel filter + discriminator = one tcgen05 int8 kernel, the "
                       "pre-discriminator AGC (a positive real gain the discriminator cannot see) elided "
                       "(fmgpu_set_demod_mode 1); every other stage in "
                       "the reference's summation order" if args.decim_mode == "tc" else
                       "reference order everywhere: bit-identical to the CPU oracle (modes 0)"),
        "step_submission": "joined per step" if args.sync_steps else
                           "streamed (async steps, one join before the closing event)",
        "block_samples": BLOCK, "iq_rate": IQ_RATE, "decimation": DECIM,
        "channels_in_this_arm": channels_this_arm,
        "l2_policy": "inputs larger than L2 (no flush): "
                     f"{args.channels * args.blocks * BLOCK * DECIM * 2 / 1e6:.0f} MB of IQ per step per GPU",
        "parallelism": "channels sharded across ranks, no collective on the data path",
    }


# --------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------
def bind_host_to_gpu(local_rank: int):
    """Multi-GPU runs: give this rank the CPU cores next to ITS GPU (NVML's ideal affinity) before any
    host buffer exists, so that the pinned buffers of the end-to-end leg are first-touched on the
    GPU's own NUMA node and the H2D copies of the ranks do not all cross one socket link. (Not at
    N = 1: there the CPU baseline wants every core.)"""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        uuid = "GPU-" + str(torch.cuda.get_device_properties(local_rank).uuid)
        try:
            h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
        pynvml.nvmlDeviceSetCpuAffinity(h)
        cpus = sorted(os.sched_getaffinity(0))
        return {"count": len(cpus), "first": cpus[0], "last": cpus[-1]}
    except Exception as ex:  # affinity is an optimisation, never a requirement
        return {"error": str(ex)[:120]}


class Workload:
    """One engine + its synthetic IQ resident in HBM + device output buffers."""

    def __init__(self, fm, shard, args, rank, local_rank, world, channels, blocks, global_ids, seed):
        import numpy as np
        import torch
        self.fm, self.C, self.B = fm, channels, blocks
        self.dev = torch.device("cuda", local_rank)
        self.n_iq = blocks * BLOCK * DECIM
        self.stride = (2 * self.n_iq + 15) // 16 * 16
        self.eng = fm.Engine(fm.make_config(iq_rate=IQ_RATE, decimation=DECIM, max_blocks=blocks,
                                            dsp_agc=1), channels, local_rank)
        self.eng.set_pipeline_groups(args.groups)
        self.eng.set_decimator_mode(1 if args.decim_mode == "tc" else 0)
        self.eng.set_scan_mode(1 if args.decim_mode == "tc" else 0)
        self.eng.set_fir_mode(1 if args.decim_mode == "tc" else 0)
        self.eng.set_demod_mode(1 if args.decim_mode == "tc" else 0)
        for m in (0, 2):   # blend mode = global channel id % 3 (1 = normal is the engine default)
            for c, g in enumerate(global_ids):
                if g % 3 == m:
                    self.eng.set_blend_mode(m, c)
        self.iq = torch.empty((channels, self.stride), dtype=torch.uint8, device=self.dev)
        rng = np.random.default_rng(seed)
        params = []
        for g in global_ids:
            params.append(fm.SynthParams(
                float(rng.choice([22_500.0, 37_500.0, 50_000.0, 60_000.0, 75_000.0])),
                400.0 + 37.0 * (g % 200), 0.8, 700.0 + 53.0 * (g % 150), 0.8, 0.10, 0.04, 0.5,
                float(rng.uniform(10.0, 40.0)), g, 0x1000 + (g & 0xFFF), 0))
        fm.synth_iq(local_rank, params, IQ_RATE, self.n_iq, self.iq.data_ptr(), self.stride)
        torch.cuda.synchronize()
        self.acap = self.eng.audio_capacity(blocks)
        self.gcap = blocks + 8
        C, B = channels, blocks
        self.audio = torch.empty((C, 2, self.acap), dtype=torch.float32, device=self.dev)
        self.n_audio = torch.zeros(C, dtype=torch.int32, device=self.dev)
        self.groups = torch.zeros((C, self.gcap, 16), dtype=torch.uint8, device=self.dev)
        self.n_groups = torch.zeros(C, dtype=torch.int32, device=self.dev)
        self.status = torch.zeros((C, B, 20), dtype=torch.uint8, device=self.dev)

    def step(self, stream, joined: bool):
        f = self.eng.process_batch if joined else self.eng.process_batch_async
        f(self.iq.data_ptr(), self.stride, self.B, self.audio.data_ptr(), self.acap,
          self.n_audio.data_ptr(), self.groups.data_ptr(), self.gcap, self.n_groups.data_ptr(),
          self.status.data_ptr(), stream)

    def timed(self, stream, steps, warmup, joined, barrier):
        """`steps` steps between two CUDA events on `stream`; returns (this rank's ms, launches)."""
        import torch
        for _ in range(max(3, warmup)):
            self.step(stream, joined)
        self.eng.join(stream)
        barrier()
        l0 = self.eng.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(steps):
            self.step(stream, joined)
        self.eng.join(stream)
        ev1.record()
        barrier()
        return ev0.elapsed_time(ev1), self.eng.launch_count() - l0

    def dump_outputs(self, out_dir: str, max_bytes: int = 60 << 20):
        """What the last step returned, for comparing two builds output for output (the seeded inputs
        and the number of steps fix it): audio [k, 2, cap] (float32, zero past n_audio) and, as
        float64, n_audio [k], groups [k, gcap, 6] (a, b, c, d, errors, block_index; zero past
        n_groups), n_groups [k] and status [k, blocks, 5] (n_audio, stereo, pilot_tenths, clip_ratio,
        n_groups) of the channels listed in channels [k], a seeded sample when all of them would
        exceed max_bytes."""
        import numpy as np
        import torch
        C = self.C
        per_channel = 4 * 2 * self.acap + 8 * (2 + 6 * self.gcap + 5 * self.B + 1)
        k = min(C, max_bytes // per_channel)
        pick = np.sort(np.random.default_rng(0).choice(C, k, replace=False)) if k < C else np.arange(C)
        idx = torch.from_numpy(pick).to(self.dev)
        n_audio = self.n_audio.index_select(0, idx).cpu().numpy()
        n_groups = self.n_groups.index_select(0, idx).cpu().numpy()
        audio = self.audio.index_select(0, idx).cpu().numpy()
        audio = np.where(np.arange(self.acap)[None, None, :] < n_audio[:, None, None], audio, np.float32(0))
        g = self.groups.index_select(0, idx).cpu().numpy().view(self.fm.GROUP_DTYPE).reshape(k, self.gcap)
        groups = np.stack([g[f].astype(np.float64) for f in ("a", "b", "c", "d", "errors", "block_index")], -1)
        groups[np.arange(self.gcap)[None, :] >= n_groups[:, None]] = 0.0
        st = self.status.index_select(0, idx).cpu().numpy().view(self.fm.STATUS_DTYPE).reshape(k, self.B)
        status = np.stack([st[f].astype(np.float64) for f in self.fm.STATUS_DTYPE.names], -1)
        os.makedirs(out_dir, exist_ok=True)
        for name, a in (("channels", pick.astype(np.float64)), ("audio", audio),
                        ("n_audio", n_audio.astype(np.float64)), ("groups", groups),
                        ("n_groups", n_groups.astype(np.float64)), ("status", status)):
            np.save(os.path.join(out_dir, f"{name}.npy"), a)

    def stage_times(self, stream, reps=3):
        """Every stage's kernels alone: the block pipeline queued on ONE stream (overlap off)."""
        import torch
        self.eng.set_stage_overlap(False)
        for _ in range(2):
            self.step(stream, True)
        torch.cuda.synchronize()
        self.eng.enable_stage_timing(True)
        acc = {}
        for _ in range(reps):
            self.step(stream, True)
            torch.cuda.synchronize()
            for k, v in self.eng.stage_times().items():
                acc[k] = acc.get(k, 0.0) + v / reps
        self.eng.enable_stage_timing(False)
        self.eng.set_stage_overlap(True)
        return acc

    def host_buffers(self):
        """Pinned host copies of the IQ and two sets of host output buffers (RuntimeError if the
        box cannot pin them)."""
        import torch
        C, B = self.C, self.B
        iq_host = torch.empty((C, self.stride), dtype=torch.uint8).pin_memory()
        iq_host.copy_(self.iq)
        outs = []
        for _ in range(2):   # step k+1 is submitted before step k is waited for
            outs.append((torch.empty((C, 2, self.acap), dtype=torch.float32).pin_memory(),
                         torch.zeros(C, dtype=torch.int32).pin_memory(),
                         torch.zeros((C, self.gcap, 16), dtype=torch.uint8).pin_memory(),
                         torch.zeros(C, dtype=torch.int32).pin_memory(),
                         torch.zeros((C, B, 20), dtype=torch.uint8).pin_memory()))
        return iq_host, outs

    def e2e(self, iq_host, outs, steps, warmup, joined, barrier, shard, world):
        """Through fmgpu_submit_host / fmgpu_wait_host: every step copies its IQ from pinned host
        memory, runs the pipeline and copies audio / groups / status back; wall clock, max over
        ranks. Returns the e2e record."""
        import torch
        eng, B = self.eng, self.B

        def submit(k):
            a_h, na_h, g_h, ng_h, st_h = outs[k & 1]
            return eng.submit_host_raw(iq_host.data_ptr(), self.stride, B, a_h.data_ptr(), self.acap,
                                       na_h.data_ptr(), g_h.data_ptr(), self.gcap, ng_h.data_ptr(),
                                       st_h.data_ptr())

        def run(n):
            if joined:
                for k in range(n):
                    eng.wait_host(submit(k))
                return
            pending = submit(0)
            for k in range(1, n):
                nxt = submit(k)
                eng.wait_host(pending)
                pending = nxt
            eng.wait_host(pending)

        run(max(2, min(warmup, 3)))
        barrier()
        t0 = time.perf_counter()
        run(steps)
        torch.cuda.synchronize()
        dt = shard.max_over_ranks(time.perf_counter() - t0, self.dev)
        frames = int(outs[0][1].max().item())
        C = self.C
        total = shard.sum_over_ranks(C * self.n_iq, self.dev)   # IQ samples per step, all ranks
        return {"value": total * steps / dt / 1e6, "unit": "MS/s",
                "h2d_bytes_per_step": int(C * 2 * self.n_iq),
                "d2h_bytes_per_step": int(C * 2 * frames * 4 + C * self.gcap * 16 + C * B * 20 + 8 * C),
                "ms_per_step": dt / steps * 1e3,
                "realtime_channels": total * steps / dt / IQ_RATE}

    def h2d_roof(self, iq_host, barrier, shard, reps=4):
        """The box's roof for the e2e leg: every rank copies its pinned IQ buffer to its GPU with one
        bare cudaMemcpyAsync at the same time as all the others; GB/s per rank (min over ranks) and
        in total."""
        import torch
        dst = torch.empty_like(self.iq)
        s = torch.cuda.Stream(device=self.dev)
        worst = 0.0
        with torch.cuda.stream(s):
            dst.copy_(iq_host, non_blocking=True)
            s.synchronize()
            barrier()
            t0 = time.perf_counter()
            for _ in range(reps):
                dst.copy_(iq_host, non_blocking=True)
            s.synchronize()
            worst = shard.max_over_ranks(time.perf_counter() - t0, self.dev)
        per_rank = iq_host.numel() * reps / worst / 1e9
        total = shard.sum_over_ranks(iq_host.numel(), self.dev) * reps / worst / 1e9
        del dst
        return {"per_rank_gbs": per_rank, "total_gbs": total,
                "probe": f"{reps} x cudaMemcpyAsync of each rank's pinned IQ buffer "
                         f"({iq_host.numel() / 1e6:.0f} MB), all ranks at once, slowest rank's wall clock"}

    def close(self):
        self.eng.close()


def run_b200(args, rank: int, local_rank: int, world: int):
    import torch
    import torch.distributed as dist

    import fmtuner_sdr_b200 as fm
    from fmtuner_sdr_b200 import shard

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    host_cpus = bind_host_to_gpu(local_rank) if world > 1 else None
    C, B = args.channels, args.blocks
    joined = args.sync_steps

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream

    # ---- main record: weak scaling, C channels on every rank -----------------------------------
    wl = Workload(fm, shard, args, rank, local_rank, world, C, B,
                  list(shard.channels_of_rank(rank, world, C)), 1234 + rank)
    # Steps are streamed the way the reference's main loop runs block after block (main.cpp:992):
    # every stage orders itself after its own previous block, so one step's serial kernels overlap
    # the next step's FIR kernels; fmgpu_join puts all of it back on the caller's stream before the
    # closing event. --sync-steps joins after every step.
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.25)
    w0 = time.time()
    ms_rank, launches = wl.timed(stream, args.steps, args.warmup, joined, barrier)
    w1 = time.time()
    clocks = sampler.stop(w0, w1)
    ms = shard.max_over_ranks(ms_rank, dev)
    if args.dump_outputs and rank == 0:
        wl.dump_outputs(args.dump_outputs)   # before stage_times() runs further steps
    samples_per_step_rank = C * wl.n_iq
    value = shard.aggregate_throughput(samples_per_step_rank, args.steps, world, ms)  # MS/s, whole job

    # sanity: the run really decoded (stereo flags + RDS groups present)
    st_host = wl.status.cpu().numpy().view(fm.STATUS_DTYPE).reshape(C, B)
    decoded = {"stereo_channels": int(st_host["stereo"][:, -1].sum()),
               "groups_last_step": int(wl.n_groups.sum().item())}

    # ---- per-stage device times and the roofline records ---------------------------------------
    acc = wl.stage_times(stream)
    stage_ms = {k: round(v, 4) for k, v in acc.items()}
    fp32_peak = fm.measure_fp32_tflops(local_rank)
    roofline = roofline_record(acc, C, B, fp32_peak, args.decim_mode, ms / args.steps)
    # the RF level meter (SURVEY 8(f) row 2: 2 B in per IQ sample) is not part of the step: timed here
    sums = torch.zeros((C, B, 48), dtype=torch.uint8, device=dev)
    for _ in range(2):
        wl.eng.signal_level_batch(wl.iq.data_ptr(), wl.stride, B, sums.data_ptr(), stream)
    sl0, sl1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    sl0.record()
    for _ in range(5):
        wl.eng.signal_level_batch(wl.iq.data_ptr(), wl.stride, B, sums.data_ptr(), stream)
    sl1.record()
    torch.cuda.synchronize()
    sl_ms = sl0.elapsed_time(sl1) / 5
    sl_gbs = 2.0 * C * wl.n_iq / (sl_ms * 1e-3) / 1e9
    roofline["streaming_kernels"].append(
        {"kernel": "signal_level", "bytes_per_launch": 2.0 * C * wl.n_iq, "launch_ms": sl_ms,
         "achieved": sl_gbs, "unit": "GB/s", "frac": sl_gbs / roofline["hbm_peak_gbs"]})
    del sums

    # ---- end to end through the host-buffer C-ABI call -----------------------------------------
    e2e = None
    h2d = None
    e2e_ready = not args.no_e2e
    iq_host = outs = None
    if e2e_ready:
        # a rank that cannot pin its buffers takes the leg off for every rank (the timing
        # reduction is a collective)
        failed = 0.0
        try:
            iq_host, outs = wl.host_buffers()
        except RuntimeError as ex:
            print(f"rank {rank}: no pinned host buffers for the end-to-end leg: {ex}", file=sys.stderr)
            failed = 1.0
        e2e_ready = shard.max_over_ranks(failed, dev) == 0
    if e2e_ready:
        e2e = wl.e2e(iq_host, outs, args.steps, args.warmup, joined, barrier, shard, world)
        if not args.no_extras:
            h2d = wl.h2d_roof(iq_host, barrier, shard)
            e2e["h2d_roof_gbs"] = h2d["per_rank_gbs"]
            e2e["h2d_roof_total_gbs"] = h2d["total_gbs"]
            e2e["h2d_gbs"] = e2e["h2d_bytes_per_step"] / (e2e["ms_per_step"] * 1e-3) / 1e9
            e2e["frac_of_h2d_roof"] = e2e["h2d_gbs"] / h2d["per_rank_gbs"]
            e2e["h2d_roof_probe"] = h2d["probe"]
    iq_host = outs = None

    # ---- CPU baseline on this box's host cores (rank 0, N = 1 only) ----------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        rows = wl.iq[:min(cores, 16), :2 * wl.n_iq].cpu().numpy()
        cpu_arm(rows, B, 1, cores)                       # warm-up + calibration
        s1, d1 = cpu_arm(rows, B, 1, cores)
        passes = max(1, int(args.cpu_seconds / max(d1, 1e-3)))
        s, d = cpu_arm(rows, B, passes, cores)
        cpu_baseline = {"value": s / d / 1e6, "unit": "MS/s", "cores": cores,
                        "sample": f"{cores} channels (one per thread) x {passes} passes x {B} blocks "
                                  f"x {BLOCK * DECIM} IQ samples of the same synthetic workload",
                        "seconds": d, **cpu_kind()}
    wl.close()
    del wl
    torch.cuda.empty_cache()

    strong = config4 = None
    if not args.no_extras:
        strong = strong_record(fm, shard, args, rank, local_rank, world, stream, barrier)
        torch.cuda.empty_cache()
        config4 = config4_record(fm, shard, args, rank, local_rank, world, stream, barrier)

    if rank == 0:
        line = {
            "metric": "aggregate IQ MS/s demodulated (stereo+RDS)", "value": value, "unit": "MS/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "realtime_channels": value * 1e6 / IQ_RATE,
            "config": workload_config(args, world * C),
            "clocks": clocks, "gpu_launches": int(launches), "e2e": e2e, "roofline": roofline,
            "cpu_baseline": cpu_baseline, "stage_ms": stage_ms, "decoded": decoded,
            "strong": strong, "config4": config4,
            "native_library": os.path.basename(fm.lib_path()),
        }
        if host_cpus is not None:
            line["host_affinity_rank0"] = host_cpus
        print(json.dumps(line), flush=True)


def strong_record(fm, shard, args, rank, local_rank, world, stream, barrier):
    """The north-star operating point (SURVEY 8(d) config 5): 10,000 channels IN TOTAL dealt over
    the ranks (1250 per GPU at N = 8), 4 logical blocks per step; device-timed, end to end, and the
    slowest one-lane-per-channel stage (which is what sets the pace once a GPU holds few channels)."""
    import torch
    total, B = 10_000, 4
    mine = shard.split_total(total, world)[rank]
    steps = max(2, min(args.steps, 5))
    wl = Workload(fm, shard, args, rank, local_rank, world, len(mine), B, list(mine), 99 + rank)
    ms_rank, launches = wl.timed(stream, steps, args.warmup, args.sync_steps, barrier)
    ms = shard.max_over_ranks(ms_rank, wl.dev)
    n_total = total * wl.n_iq
    acc = wl.stage_times(stream, reps=2)
    lane = max((k for k in acc if k in LANE_STAGES), key=acc.get)
    rec = {"scaling": "strong", "total_channels": total, "channels_this_rank": len(mine),
           "blocks_per_step": B, "steps": steps, "ms_per_step": ms / steps,
           "value": n_total * steps / (ms * 1e-3) / 1e6, "unit": "MS/s",
           "realtime_factor": (B * BLOCK / 240000.0) / (ms / steps * 1e-3),
           "gpu_launches": int(launches),
           "slowest_lane_stage": {"kernel": lane, "ms_per_block": acc[lane] / B,
                                  "realtime_factor": (BLOCK / 240000.0) / (acc[lane] / B * 1e-3)},
           "stage_ms": {k: round(v, 4) for k, v in acc.items()}, "e2e": None}
    if not args.no_e2e:
        failed = 0.0
        try:
            iq_host, outs = wl.host_buffers()
        except RuntimeError:
            failed = 1.0
        if shard.max_over_ranks(failed, wl.dev) == 0:
            rec["e2e"] = wl.e2e(iq_host, outs, steps, args.warmup, args.sync_steps, barrier, shard, world)
    wl.close()
    return rec


def config4_record(fm, shard, args, rank, local_rank, world, stream, barrier):
    """BASELINE config 4: one 24 MS/s uint8 capture of the whole band (100 carriers, 200 kHz apart)
    resident in HBM on every rank; each rank channelizes ITS share of the carriers
    (fmgpu_channelizer_process(ch_first, ch_count)) to 240 kS/s complex float and runs the
    complex-float batch path (FMDemod::processSplitComplex ... RDS) on them. No collective."""
    import math

    import torch
    dev = torch.device("cuda", local_rank)
    n_ch, D, B = 100, 100, 2
    mine = shard.split_total(n_ch, world)[rank]
    steps = max(2, min(args.steps, 5))
    n_wide = B * BLOCK * D
    # synthetic band: every carrier FM-modulated (75 kHz) by a stereo multiplex of one tone + pilot
    t = torch.arange(n_wide, device=dev, dtype=torch.float64) / 24e6
    x = torch.zeros(n_wide, dtype=torch.complex64, device=dev)
    wp = 2 * math.pi * 19000.0
    for k in range(n_ch):
        fc = -9_900_000.0 + 200_000.0 * k
        a = 2 * math.pi * (400.0 + 37.0 * k)
        # integral of m(t) = 0.43 sin(at) + 0.43 sin(at) sin(2 wp t) + 0.1 sin(wp t)
        im = (-0.43 / a) * torch.cos(a * t) \
            + 0.215 * (torch.sin((2 * wp - a) * t) / (2 * wp - a) - torch.sin((2 * wp + a) * t) / (2 * wp + a)) \
            - (0.1 / wp) * torch.cos(wp * t)
        ph = 2 * math.pi * fc * t + 2 * math.pi * 75000.0 * im + 0.7 * k
        x += (0.03 * torch.exp(1j * ph)).to(torch.complex64)
    iq = torch.view_as_real(x).mul(127.5).add(127.5).round().clamp(0, 255).to(torch.uint8).contiguous()
    del x, t
    z = fm.Channelizer(device=local_rank)
    eng = fm.Engine(fm.make_config(iq_rate=240_000, decimation=1, max_blocks=B), len(mine), local_rank)
    n_dsp = B * BLOCK
    cf = torch.zeros((len(mine), n_dsp, 2), dtype=torch.float32, device=dev)
    acap, gcap = eng.audio_capacity(B), B + 8
    audio = torch.empty((len(mine), 2, acap), dtype=torch.float32, device=dev)
    n_audio = torch.zeros(len(mine), dtype=torch.int32, device=dev)
    status = torch.zeros((len(mine), B, 20), dtype=torch.uint8, device=dev)

    def step():
        z.process(iq.data_ptr(), n_wide, cf.data_ptr(), n_dsp, mine.start, len(mine), stream)
        eng.process_batch_cf32(cf.data_ptr(), n_dsp, B, audio.data_ptr(), acap, n_audio.data_ptr(),
                               None, gcap, None, status.data_ptr(), stream)

    zt0, zt1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        step()
    barrier()
    zt0.record()
    for _ in range(steps):
        z.process(iq.data_ptr(), n_wide, cf.data_ptr(), n_dsp, mine.start, len(mine), stream)
    zt1.record()
    barrier()
    z_ms = zt0.elapsed_time(zt1) / steps
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(steps):
        step()
    ev1.record()
    barrier()
    ms = shard.max_over_ranks(ev0.elapsed_time(ev1), dev)
    st = status.cpu().numpy().view(fm.STATUS_DTYPE).reshape(len(mine), B)
    taps = z.taps().size
    rec = {"workload": "24 MS/s uint8 capture, 100 carriers at 200 kHz spacing -> channelizer -> "
                       "240 kS/s complex float -> FMDemod::processSplitComplex ... audio + RDS",
           "channels_total": n_ch, "channels_this_rank": len(mine), "blocks_per_step": B,
           "steps": steps, "ms_per_step": ms / steps,
           "wideband_ms_per_s": n_wide * steps / (ms * 1e-3) / 1e6,
           "realtime_factor": (n_wide / 24e6) / (ms / steps * 1e-3),
           "channelizer": {"form": "polyphase: 120 commutator phases + one 120-point DFT row per channel",
                           "taps": int(taps), "ms_per_step": z_ms,
                           "algorithmic_bytes": 2.0 * n_wide + 8.0 * len(mine) * n_dsp,
                           "achieved_gbs": (2.0 * n_wide + 8.0 * len(mine) * n_dsp) / (z_ms * 1e-3) / 1e9,
                           # per output instant: 2 FMA per tap (complex x real) + 4 FMA per (phase, channel)
                           "fp32_tflops": 2.0 * (2.0 * taps + 4.0 * 120 * len(mine)) * n_dsp / (z_ms * 1e-3) / 1e12,
                           "bound": "fp32 (shared-memory operand reads); < 3 % of the config-4 step"},
           "pilot_tenths_mean": float(st["pilot_tenths"][:, -1].mean())}
    z.close()
    eng.close()
    return rec


TILE_STAGES = ("decimate", "chanfir", "chan_demod", "freqdem", "pilot_fir", "audio_lpf", "afpost", "rds_resample")
LANE_STAGES = ("dcblock", "agc", "stereo_pll", "rds", "rds_sync")

# DRAM bytes per DSP-rate sample (dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu
# --set full).
NCU_TRAFFIC_BYTES_PER_SAMPLE = {
    # fast flavour: profiles/r02_top_kernels_ncu.csv (the round-2 final capture, 81.92 M samples per launch)
    "decimate": 29.0, "chan_demod": 11.9, "pilot_fir": 8.0, "audio_lpf": 15.8, "stereo_pll": 15.7,
    "dcblock": 15.5, "rds": 3.0, "rds_resample": 6.5, "afpost": 10.7,
    # reference-order flavour: the round-1 captures of the same FP32 kernels
    "decimate_fp32": 27.8, "chanfir": 15.6, "pilot_fir_fp32": 7.6, "audio_lpf_fp32": 15.6, "agc": 10.7,
    "freqdem": 9.3,
}


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def stage_figures(stage: str, stage_ms: float, C: int, B: int, peak_hbm: float, fp32_peak: float,
                  decim_mode: str) -> dict:
    """Algorithmic bytes / flops of ONE LAUNCH of a stage (one logical block of all C channels,
    DESIGN.md section 4) over its average launch duration, against both roofs; `bound` names the one
    that binds the kernel's formulation."""
    n = C * BLOCK                # DSP-rate samples per launch
    launch_ms = stage_ms / B
    alg = {   # stage: (bytes, flops, bound)
        "decimate": (2.0 * n * DECIM + 8.0 * n, 2.0 * 2 * 280 * n, "hbm" if decim_mode == "tc" else "fp32"),
        "chanfir": (8.0 * n + 8.0 * n, 2.0 * 2 * 81 * n, "fp32"),
        # fused channel filter + discriminator (fir_tc.cu): complex samples in, MPX out
        "chan_demod": (8.0 * n + 4.0 * n, 2.0 * 2 * 81 * n + 30.0 * n, "hbm"),
        # tensor-core forms (fir_tc.cu): the FP32 pipe is out of the picture, HBM is the roof
        "pilot_fir": (4.0 * n + 4.0 * n, 2.0 * 305 * n, "hbm" if decim_mode == "tc" else "fp32"),
        "audio_lpf": (8.0 * n + 8.0 * n, 2.0 * 2 * 121 * n, "hbm" if decim_mode == "tc" else "fp32"),
        # bound by the shared-memory pipe (per-output branch rows + unaligned windows: one read per FMA)
        "rds_resample": (4.0 * n + 4.0 * n * 171.0 / 240.0, 2.0 * 26 * n * 171.0 / 240.0, "lsu"),
        "afpost": (8.0 * n + 8.0 * n * 32.0 / 240.0, 2.0 * 2 * 24 * n * 32.0 / 240.0, "hbm"),
        "freqdem": (8.0 * n + 4.0 * n, 30.0 * n, "hbm"),
        "stereo_pll": (8.0 * n + 8.0 * n, 75.0 * n, "latency"),
        "rds": (4.0 * n * 171.0 / 240.0, 2.0 * (22 + 20) * n * 171.0 / 240.0, "latency"),
        "rds_sync": (0.01 * n, 0.1 * n, "latency"),
        "dcblock": (8.0 * n + 8.0 * n, 6.0 * n, "latency"),
        "agc": (8.0 * n + 8.0 * n, 40.0 * n, "latency"),
    }.get(stage)
    if alg is None:
        return {"kernel": stage, "launch_ms": launch_ms}
    t = launch_ms * 1e-3
    gbs, tf = alg[0] / t / 1e9, alg[1] / t / 1e12
    key = stage
    if decim_mode != "tc" and stage in ("decimate", "pilot_fir", "audio_lpf"):
        key = stage + "_fp32"
    traffic = NCU_TRAFFIC_BYTES_PER_SAMPLE.get(key)
    out = {"kernel": stage, "bound": alg[2], "launch_ms": launch_ms, "launches_per_step": B,
           "algorithmic_bytes": alg[0], "hbm_gbs": gbs, "hbm_frac": gbs / peak_hbm,
           "fp32_tflops": tf, "fp32_frac": tf / fp32_peak,
           "traffic": traffic * n if traffic is not None else None}
    if alg[2] == "latency":
        out["lane_steps_per_s"] = n / t
    if alg[2] == "lsu":
        # algorithmic shared-memory wavefronts of the resampler: per warp of 32 outputs, 26 32-bit window
        # reads (one wavefront each when conflict-free) + 7 128-bit branch-row reads (four wavefronts
        # each); roof = one wavefront per SM and clock (148 SMs at the run's SM clock)
        outs = n * 171.0 / 240.0
        wf = outs / 32.0 * (26 + 7 * 4)
        peak = 148 * 1.965e9
        out["lsu_gwavefronts_s"] = wf / t / 1e9
        out["lsu_peak_gwavefronts_s"] = peak / 1e9
        out["lsu_frac"] = wf / t / peak
    return out


def roofline_record(acc: dict, C: int, B: int, fp32_peak: float, decim_mode: str, step_ms: float) -> dict:
    peak_hbm, hbm_how = hbm_peak()
    figs = {k: stage_figures(k, v, C, B, peak_hbm, fp32_peak, decim_mode) for k, v in acc.items()
            if k in TILE_STAGES or k in LANE_STAGES}
    serial = sum(acc.values())
    # dominant throughput-bound kernel: the largest stage time; stages within 3 % of it count as tied
    # and the one that moves more algorithmic bytes is named (in the fast flavour the tensor-core
    # decimator and the 171 kHz resampler sit at 1.23 / 1.24 ms per step)
    tiles = [k for k in acc if k in TILE_STAGES]
    top_ms = max(acc[k] for k in tiles)
    dom = max((k for k in tiles if acc[k] >= 0.97 * top_ms),
              key=lambda k: figs[k].get("algorithmic_bytes", 0.0))
    d = figs[dom]
    if d["bound"] == "hbm":
        top = {"bound": "hbm", "achieved": d["hbm_gbs"], "peak": peak_hbm, "unit": "GB/s",
               "frac": d["hbm_frac"], "peak_source": hbm_how}
    elif d["bound"] == "lsu":
        top = {"bound": "lsu", "achieved": d["lsu_gwavefronts_s"], "peak": d["lsu_peak_gwavefronts_s"],
               "unit": "G shared-memory wavefronts/s", "frac": d["lsu_frac"],
               "peak_source": "148 SMs x 1 wavefront per clock x 1.965 GHz (ncu of the same kernel: "
                              "l1tex LSU data pipe 95 % busy, profiles/r02_top_kernels_ncu.csv)"}
    else:
        top = {"bound": "fp32", "achieved": d["fp32_tflops"], "peak": fp32_peak, "unit": "TFLOP/s",
               "frac": d["fp32_frac"],
               "peak_source": "fmgpu_measure_fp32_tflops in this run (packed FFMA2 loop on every SM)"}
    lane = max((k for k in acc if k in LANE_STAGES), key=acc.get)
    n_iq_step = C * B * BLOCK * DECIM
    rec = {"kernel": dom, **top, "traffic": d["traffic"],
           "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum per DSP-rate sample of the "
                             "ncu --set full captures named at NCU_TRAFFIC_BYTES_PER_SAMPLE (profiles/) "
                             "x the samples of one launch; not re-measured by this run",
           "algorithmic_bytes": d["algorithmic_bytes"], "launch_ms": d["launch_ms"],
           "launches_per_step": B, "step_share": acc[dom] / serial,
           "hbm_peak_gbs": peak_hbm, "hbm_peak_source": hbm_how, "fp32_peak_tflops": fp32_peak,
           "scope": "dominant throughput-bound (tile) kernel; the one-lane-per-channel kernels are "
                    "latency-bound serial recursions and are reported as lane-steps/s (SURVEY 8(d))",
           "dominant_lane_kernel": {"kernel": lane, "launch_ms": acc[lane] / B, "lanes": C,
                                    "lane_steps_per_s": C * B * BLOCK / (acc[lane] * 1e-3),
                                    "realtime_factor": (B * BLOCK / 240000.0) / (acc[lane] * 1e-3)},
           "kernels": figs, "stage_sum_ms": serial, "overlap_factor": serial / step_ms,
           "overlap_note": "stage_ms are the stages run one after the other (fmgpu_set_stage_overlap(0)); "
                           "in the timed steps the block pipeline overlaps them: overlap_factor = "
                           "their sum / the measured step",
           "streaming_kernels": [], "whole_step": {
               "hbm_gbs": n_iq_step * BYTES_PER_IQ_SAMPLE_ALG / (step_ms * 1e-3) / 1e9,
               "hbm_frac": n_iq_step * BYTES_PER_IQ_SAMPLE_ALG / (step_ms * 1e-3) / 1e9 / peak_hbm,
               "fp32_tflops": n_iq_step * FLOP_PER_IQ_SAMPLE_ALG / (step_ms * 1e-3) / 1e12,
               "fp32_frac": n_iq_step * FLOP_PER_IQ_SAMPLE_ALG / (step_ms * 1e-3) / 1e12 / fp32_peak}}
    # the same record in the contract's own vocabulary (bound "hbm", GB/s against MEASURED_PEAKS.json)
    # for the largest HBM-bound tile kernel, whichever kernel is named above
    hbm_tiles = [k for k in tiles if figs[k]["bound"] == "hbm"]
    if hbm_tiles:
        h = max(hbm_tiles, key=acc.get)
        rec["largest_hbm_bound_kernel"] = {
            "kernel": h, "bound": "hbm", "achieved": figs[h]["hbm_gbs"], "peak": peak_hbm, "unit": "GB/s",
            "frac": figs[h]["hbm_frac"], "traffic": figs[h]["traffic"],
            "algorithmic_bytes": figs[h]["algorithmic_bytes"], "launch_ms": figs[h]["launch_ms"],
            "step_share": acc[h] / serial}
    if "freqdem" in figs:
        f = figs["freqdem"]
        rec["streaming_kernels"].append({"kernel": "freqdem", "bytes_per_launch": f["algorithmic_bytes"],
                                         "launch_ms": f["launch_ms"], "achieved": f["hbm_gbs"],
                                         "unit": "GB/s", "frac": f["hbm_frac"]})
    return rec


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_b200(args, rank, local_rank, world)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()

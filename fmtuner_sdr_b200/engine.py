"""ctypes view of the engine's C ABI (include/fmgpu.h).

Mirrors the reference's block-processing interface: the per-stage methods carry the
names of the reference classes' methods (FMDemod.processSplit, StereoDecoder.processAudio,
AFPostProcessor.process, RDSDecoder.process, ComplexDecimator.executeComplex) and the
batched `process_*` calls are the per-block body of src/main.cpp:1232-1308 for C channels.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

GROUP_DTYPE = np.dtype([("a", "<u2"), ("b", "<u2"), ("c", "<u2"), ("d", "<u2"), ("errors", "u1"),
                        ("pad", "u1", 3), ("block_index", "<u4")])
STATUS_DTYPE = np.dtype([("n_audio", "<i4"), ("stereo", "<i4"), ("pilot_tenths", "<i4"),
                         ("clip_ratio", "<f4"), ("n_groups", "<i4")])

RESET_DECIM, RESET_DEMOD, RESET_STEREO, RESET_AFPOST, RESET_RDS = 1, 2, 4, 8, 16
RESET_DSP, RESET_ALL = 15, 31


class EngineError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "iq_rate", "decimation", "output_rate", "block_samples", "max_blocks", "w0_bandwidth_hz",
        "bandwidth_hz", "dsp_agc", "stereo_blend", "deemphasis", "stereo", "force_mono",
        "decim_taps_per_phase", "decim_atten_db")]


def make_config(iq_rate=2_400_000, decimation=10, output_rate=32000, block_samples=8192,
                max_blocks=4, w0_bandwidth_hz=194000, bandwidth_hz=0, dsp_agc=0, stereo_blend=1,
                deemphasis=0, stereo=1, force_mono=0, decim_taps_per_phase=0,
                decim_atten_db=0) -> Config:
    return Config(iq_rate, decimation, output_rate, block_samples, max_blocks, w0_bandwidth_hz,
                  bandwidth_hz, dsp_agc, stereo_blend, deemphasis, stereo, force_mono,
                  decim_taps_per_phase, decim_atten_db)


class LevelSums(C.Structure):
    _fields_ = [("sum_i", C.c_uint64), ("sum_q", C.c_uint64), ("sum_ii", C.c_uint64),
                ("sum_qq", C.c_uint64), ("hard_clip", C.c_uint32), ("near_clip", C.c_uint32),
                ("n_samples", C.c_uint32), ("pad", C.c_uint32)]


class SignalLevel(C.Structure):
    _fields_ = [("level120", C.c_float), ("dbfs", C.c_double), ("compensated_dbfs", C.c_double),
                ("hard_clip_ratio", C.c_double), ("near_clip_ratio", C.c_double)]


class SynthParams(C.Structure):
    _fields_ = [("deviation_hz", C.c_float), ("tone_l_hz", C.c_float), ("tone_l_amp", C.c_float),
                ("tone_r_hz", C.c_float), ("tone_r_amp", C.c_float), ("pilot_amp", C.c_float),
                ("rds_amp", C.c_float), ("iq_amp", C.c_float), ("snr_db", C.c_float),
                ("seed", C.c_uint32), ("pi", C.c_uint16), ("pad", C.c_uint16)]


_lib = None


def lib_path() -> str:
    return _build.LIB


def load_library(build: bool = True):
    """Load libfmgpu.so (building it in-tree if missing). Fails loudly if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if build and not os.path.exists(_build.LIB):
        _build.build_lib()
    if not os.path.exists(_build.LIB):
        raise EngineError(f"{_build.LIB} is missing: run __graft_entry__.build() (no CPU fallback)")
    # FMGPU_LIB: an alternative build of the same library (A/B timing of compile-time variants)
    L = C.CDLL(os.environ.get("FMGPU_LIB") or _build.LIB)
    vp, i32, sz, u8p, f32p = C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_void_p
    L.fmgpu_engine_create.argtypes = [C.POINTER(Config), i32, i32, C.POINTER(vp)]
    L.fmgpu_engine_destroy.argtypes = [vp]
    L.fmgpu_last_error.restype = C.c_char_p
    L.fmgpu_last_error.argtypes = [vp]
    L.fmgpu_n_channels.argtypes = [vp]
    L.fmgpu_dsp_rate.argtypes = [vp]
    for name in ("set_bandwidth_hz", "set_bandwidth_mode", "set_w0_bandwidth_hz", "set_agc_mode",
                 "set_deemphasis_us", "set_blend_mode", "set_force_mono", "set_force_stereo"):
        getattr(L, f"fmgpu_{name}").argtypes = [vp, i32, i32]
    L.fmgpu_reset.argtypes = [vp, i32, C.c_uint]
    L.fmgpu_measure_fp32_tflops.argtypes = [i32, C.POINTER(C.c_double)]
    L.fmgpu_set_decimator_mode.argtypes = [vp, i32]
    L.fmgpu_get_decimator_mode.argtypes = [vp]
    L.fmgpu_set_scan_mode.argtypes = [vp, i32]
    L.fmgpu_get_scan_mode.argtypes = [vp]
    L.fmgpu_set_fir_mode.argtypes = [vp, i32]
    L.fmgpu_get_fir_mode.argtypes = [vp]
    L.fmgpu_set_demod_mode.argtypes = [vp, i32]
    L.fmgpu_get_demod_mode.argtypes = [vp]
    L.fmgpu_set_pipeline_groups.argtypes = [vp, i32]
    L.fmgpu_set_stage_overlap.argtypes = [vp, i32]
    L.fmgpu_is_stereo.argtypes = [vp, i32]
    L.fmgpu_pilot_tenths.argtypes = [vp, i32]
    L.fmgpu_clip_ratio.argtypes = [vp, i32]
    L.fmgpu_clip_ratio.restype = C.c_float
    L.fmgpu_is_clipping.argtypes = [vp, i32]
    L.fmgpu_process_batch.argtypes = [vp, u8p, sz, i32, f32p, sz, vp, vp, sz, vp, vp, vp]
    L.fmgpu_process_host.argtypes = [vp, u8p, sz, i32, f32p, sz, vp, vp, sz, vp, vp]
    L.fmgpu_process_batch_async.argtypes = [vp, u8p, sz, i32, f32p, sz, vp, vp, sz, vp, vp, vp]
    L.fmgpu_join.argtypes = [vp, vp]
    L.fmgpu_process_batch_cf32.argtypes = [vp, f32p, sz, i32, f32p, sz, vp, vp, sz, vp, vp, vp]
    L.fmgpu_channelizer_create.argtypes = [i32, i32, i32, i32, C.c_double, C.c_double, i32,
                                           C.c_double, C.c_float, C.POINTER(vp)]
    L.fmgpu_channelizer_destroy.argtypes = [vp]
    L.fmgpu_channelizer_destroy.restype = None
    L.fmgpu_channelizer_output_rate.argtypes = [vp]
    L.fmgpu_channelizer_taps.argtypes = [vp, f32p, sz]
    L.fmgpu_channelizer_taps.restype = sz
    L.fmgpu_channelizer_process.argtypes = [vp, u8p, sz, i32, i32, f32p, sz, vp]
    L.fmgpu_channelizer_create_multi.argtypes = [i32, i32, i32, i32, i32, C.POINTER(C.c_double),
                                                 C.c_double, i32, C.c_double, C.c_float, C.POINTER(vp)]
    L.fmgpu_channelizer_n_captures.argtypes = [vp]
    L.fmgpu_channelizer_process_multi.argtypes = [vp, u8p, sz, sz, i32, i32, f32p, sz, vp]
    L.fmgpu_channelizer_create_format.argtypes = [i32, i32, i32, i32, i32, i32, C.POINTER(C.c_double),
                                                  C.c_double, i32, C.c_double, C.c_float, C.POINTER(vp)]
    L.fmgpu_channelizer_sample_format.argtypes = [vp]
    L.fmgpu_channelizer_process_iq.argtypes = [vp, vp, sz, sz, i32, i32, f32p, sz, vp]
    L.fmgpu_channelizer_create_rate.argtypes = [i32, i32, i32, i32, i32, i32, C.POINTER(C.c_double),
                                                C.c_double, i32, C.c_double, C.c_float, C.POINTER(vp)]
    L.fmgpu_channelizer_interpolation.argtypes = [vp]
    L.fmgpu_channelizer_decimation.argtypes = [vp]
    L.fmgpu_channelizer_outputs.argtypes = [vp, sz]
    L.fmgpu_channelizer_outputs.restype = sz
    L.fmgpu_channelizer_process_stream.argtypes = [vp, vp, sz, sz, i32, i32, f32p, sz, C.POINTER(sz), vp]
    L.fmgpu_submit_host.argtypes = [vp, u8p, sz, i32, f32p, sz, vp, vp, sz, vp, vp]
    L.fmgpu_wait_host.argtypes = [vp, i32]
    L.fmgpu_decimate.restype = sz
    L.fmgpu_decimate.argtypes = [vp, i32, u8p, sz, f32p, sz]
    L.fmgpu_demod_u8.restype = sz
    L.fmgpu_demod_u8.argtypes = [vp, i32, u8p, f32p, f32p, sz]
    L.fmgpu_demod_cf32.restype = sz
    L.fmgpu_demod_cf32.argtypes = [vp, i32, f32p, f32p, f32p, sz]
    L.fmgpu_downsample_mono.restype = sz
    L.fmgpu_downsample_mono.argtypes = [vp, i32, f32p, f32p, sz]
    L.fmgpu_set_deviation_hz.argtypes = [vp, C.c_double]
    L.fmgpu_stereo.restype = sz
    L.fmgpu_stereo.argtypes = [vp, i32, f32p, f32p, f32p, sz]
    L.fmgpu_afpost.restype = sz
    L.fmgpu_afpost.argtypes = [vp, i32, f32p, f32p, sz, f32p, f32p, sz]
    L.fmgpu_rds.restype = sz
    L.fmgpu_rds.argtypes = [vp, i32, f32p, sz, vp, sz]
    L.fmgpu_get_design.restype = sz
    L.fmgpu_get_design.argtypes = [vp, i32, i32, f32p, sz, C.POINTER(C.c_float)]
    L.fmgpu_debug_read.restype = sz
    L.fmgpu_debug_read.argtypes = [vp, i32, i32, f32p, sz]
    L.fmgpu_debug_rds_bits.restype = sz
    L.fmgpu_debug_rds_bits.argtypes = [vp, i32, u8p, sz]
    L.fmgpu_launch_count.restype = C.c_uint64
    L.fmgpu_launch_count.argtypes = [vp]
    L.fmgpu_enable_stage_timing.argtypes = [vp, i32]
    L.fmgpu_debug_timeline.argtypes = [vp, C.POINTER(C.c_char_p), C.POINTER(i32), C.POINTER(C.c_float),
                                       C.POINTER(C.c_float), i32]
    L.fmgpu_get_stage_times.argtypes = [vp, C.POINTER(C.c_char_p), C.POINTER(C.c_float), i32]
    L.fmgpu_signal_level_batch.argtypes = [vp, u8p, sz, i32, vp, vp]
    L.fmgpu_signal_level_finish.restype = None
    L.fmgpu_signal_level_finish.argtypes = [C.POINTER(LevelSums), i32, C.c_double, C.c_double,
                                            C.c_double, C.c_double, C.POINTER(SignalLevel)]
    L.fmgpu_pack_pcm16.argtypes = [vp, f32p, sz, vp, C.c_float, vp, vp]
    L.fmgpu_synth_iq.argtypes = [i32, C.POINTER(SynthParams), i32, C.c_double, sz, u8p, sz, vp]
    _lib = L
    return L


def _ptr(a):
    return a.ctypes.data if a is not None else None


def measure_fp32_tflops(device: int = 0) -> float:
    """The FP32 FMA roof of `device`, measured (fmgpu_measure_fp32_tflops)."""
    out = C.c_double(0.0)
    rc = load_library().fmgpu_measure_fp32_tflops(device, C.byref(out))
    if rc != 0:
        raise EngineError(f"fmgpu_measure_fp32_tflops failed ({rc})")
    return out.value


def synth_iq(device: int, params, fs_iq: float, n_samples: int, iq_dev_ptr: int,
             stride_bytes: int, stream: int | None = None) -> None:
    """Fill a device buffer [C][stride] with synthetic uint8 IQ (bench input)."""
    L = load_library()
    arr = (SynthParams * len(params))(*params)
    rc = L.fmgpu_synth_iq(device, arr, len(params), float(fs_iq), n_samples, iq_dev_ptr,
                          stride_bytes, stream)
    if rc != 0:
        raise EngineError(f"fmgpu_synth_iq failed: {rc}")


class Engine:
    """n_channels independent FM stereo + RDS receivers on one GPU."""

    def __init__(self, cfg: Config, n_channels: int = 1, device: int = 0):
        self.L = load_library()
        self.cfg = cfg
        self.n_channels = n_channels
        self.device = device
        h = C.c_void_p()
        rc = self.L.fmgpu_engine_create(C.byref(cfg), n_channels, device, C.byref(h))
        if rc != 0:
            raise EngineError(f"fmgpu_engine_create failed ({rc}): "
                              f"{self.L.fmgpu_last_error(None).decode()}")
        self.h = h
        self.fs = self.L.fmgpu_dsp_rate(h)
        self.block = cfg.block_samples
        self.decim = cfg.decimation
        self.iq_bytes_per_block = self.block * self.decim * 2

    def close(self):
        if getattr(self, "h", None):
            self.L.fmgpu_engine_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise EngineError(f"{what} failed ({rc}): {self.L.fmgpu_last_error(self.h).decode()}")

    def error(self) -> str:
        return self.L.fmgpu_last_error(self.h).decode()

    # ---- settings (reference setters) -------------------------------------
    def set_bandwidth_hz(self, bw, channel=-1):
        self._check(self.L.fmgpu_set_bandwidth_hz(self.h, channel, bw), "set_bandwidth_hz")

    def set_bandwidth_mode(self, mode, channel=-1):
        self._check(self.L.fmgpu_set_bandwidth_mode(self.h, channel, mode), "set_bandwidth_mode")

    def set_w0_bandwidth_hz(self, bw, channel=-1):
        self._check(self.L.fmgpu_set_w0_bandwidth_hz(self.h, channel, bw), "set_w0_bandwidth_hz")

    def set_agc_mode(self, mode, channel=-1):
        self._check(self.L.fmgpu_set_agc_mode(self.h, channel, mode), "set_agc_mode")

    def set_deemphasis_us(self, us, channel=-1):
        self._check(self.L.fmgpu_set_deemphasis_us(self.h, channel, us), "set_deemphasis_us")

    def set_blend_mode(self, mode, channel=-1):
        self._check(self.L.fmgpu_set_blend_mode(self.h, channel, mode), "set_blend_mode")

    def set_force_mono(self, on, channel=-1):
        self._check(self.L.fmgpu_set_force_mono(self.h, channel, int(on)), "set_force_mono")

    def set_force_stereo(self, on, channel=-1):
        self._check(self.L.fmgpu_set_force_stereo(self.h, channel, int(on)), "set_force_stereo")

    def set_decimator_mode(self, mode: int):
        """0 = FP32 chain (bit-identical to the oracle), 1 = tensor-core integer contraction."""
        self._check(self.L.fmgpu_set_decimator_mode(self.h, mode), "set_decimator_mode")

    def decimator_mode(self) -> int:
        return self.L.fmgpu_get_decimator_mode(self.h)

    def set_scan_mode(self, mode: int):
        """0 = serial lane recursion (bit-identical to the oracle), 1 = warp-shuffle parallel scan."""
        self._check(self.L.fmgpu_set_scan_mode(self.h, mode), "set_scan_mode")

    def scan_mode(self) -> int:
        return self.L.fmgpu_get_scan_mode(self.h)

    def set_fir_mode(self, mode: int):
        """0 = FP32 pilot band-pass / L-R low-pass (bit-exact flavour), 1 = tensor-core integer form."""
        self._check(self.L.fmgpu_set_fir_mode(self.h, mode), "set_fir_mode")

    def fir_mode(self) -> int:
        return self.L.fmgpu_get_fir_mode(self.h)

    def set_demod_mode(self, mode: int):
        """0 = channel filter, AGC, discriminator as three kernels (bit-exact flavour); 1 = one
        tensor-core kernel (integer channel filter + discriminator, AGC elided)."""
        self._check(self.L.fmgpu_set_demod_mode(self.h, mode), "set_demod_mode")

    def demod_mode(self) -> int:
        return self.L.fmgpu_get_demod_mode(self.h)

    def set_pipeline_groups(self, groups: int):
        self._check(self.L.fmgpu_set_pipeline_groups(self.h, groups), "set_pipeline_groups")

    def set_stage_overlap(self, on: bool):
        self._check(self.L.fmgpu_set_stage_overlap(self.h, int(on)), "set_stage_overlap")

    def reset(self, what=RESET_ALL, channel=-1):
        self._check(self.L.fmgpu_reset(self.h, channel, what), "reset")

    # ---- observables -------------------------------------------------------
    def is_stereo(self, channel=0):
        return bool(self.L.fmgpu_is_stereo(self.h, channel))

    def pilot_tenths(self, channel=0):
        return self.L.fmgpu_pilot_tenths(self.h, channel)

    def clip_ratio(self, channel=0):
        return self.L.fmgpu_clip_ratio(self.h, channel)

    def is_clipping(self, channel=0):
        return bool(self.L.fmgpu_is_clipping(self.h, channel))

    # ---- batched paths -----------------------------------------------------
    def audio_capacity(self, n_blocks: int) -> int:
        return int(n_blocks * self.block * 32000 / self.fs * (1.0 + 1e-6)) + 16

    def process_host(self, iq: np.ndarray, n_blocks: int | None = None, group_cap: int | None = None):
        """iq: uint8 [C, >= n_blocks*block*decim*2]. Returns (audio[C,2,cap], n_audio[C],
        groups[C,gcap], n_groups[C], status[C,n_blocks])."""
        iq = np.ascontiguousarray(iq, np.uint8)
        if iq.ndim == 1:
            iq = iq.reshape(1, -1)
        Cn = self.n_channels
        if iq.shape[0] != Cn:
            raise ValueError("iq must have one row per channel")
        if n_blocks is None:
            n_blocks = iq.shape[1] // self.iq_bytes_per_block
        acap = self.audio_capacity(n_blocks)
        gcap = group_cap or (n_blocks + 8)
        audio = np.zeros((Cn, 2, acap), np.float32)
        n_audio = np.zeros(Cn, np.uint32)
        groups = np.zeros((Cn, gcap), GROUP_DTYPE)
        n_groups = np.zeros(Cn, np.uint32)
        status = np.zeros((Cn, n_blocks), STATUS_DTYPE)
        rc = self.L.fmgpu_process_host(self.h, _ptr(iq), iq.strides[0], n_blocks, _ptr(audio), acap,
                                       _ptr(n_audio), _ptr(groups), gcap, _ptr(n_groups),
                                       _ptr(status))
        self._check(rc, "process_host")
        return audio, n_audio, groups, n_groups, status

    def process_host_raw(self, iq_ptr, stride, n_blocks, audio_ptr, acap, n_audio_ptr, groups_ptr,
                         gcap, n_groups_ptr, status_ptr):
        self._check(self.L.fmgpu_process_host(self.h, iq_ptr, stride, n_blocks, audio_ptr, acap,
                                              n_audio_ptr, groups_ptr, gcap, n_groups_ptr,
                                              status_ptr), "process_host")

    def process_batch(self, iq_dev_ptr, stride, n_blocks, audio_ptr=None, acap=0, n_audio_ptr=None,
                      groups_ptr=None, gcap=0, n_groups_ptr=None, status_ptr=None, stream=None):
        """Device pointers (ints), asynchronous on `stream` (cudaStream_t as int)."""
        self._check(self.L.fmgpu_process_batch(self.h, iq_dev_ptr, stride, n_blocks, audio_ptr, acap,
                                               n_audio_ptr, groups_ptr, gcap, n_groups_ptr,
                                               status_ptr, stream), "process_batch")

    def process_batch_async(self, iq_dev_ptr, stride, n_blocks, audio_ptr=None, acap=0,
                            n_audio_ptr=None, groups_ptr=None, gcap=0, n_groups_ptr=None,
                            status_ptr=None, stream=None):
        """Streaming form: `stream` does not wait for the batch; call join(stream) for that."""
        self._check(self.L.fmgpu_process_batch_async(self.h, iq_dev_ptr, stride, n_blocks, audio_ptr,
                                                     acap, n_audio_ptr, groups_ptr, gcap,
                                                     n_groups_ptr, status_ptr, stream),
                    "process_batch_async")

    def process_batch_cf32(self, x_dev_ptr, stride_samples, n_blocks, audio_ptr=None, acap=0,
                           n_audio_ptr=None, groups_ptr=None, gcap=0, n_groups_ptr=None,
                           status_ptr=None, stream=None):
        """Complex-float input at the DSP rate (engine created with decimation=1)."""
        self._check(self.L.fmgpu_process_batch_cf32(self.h, x_dev_ptr, stride_samples, n_blocks,
                                                    audio_ptr, acap, n_audio_ptr, groups_ptr, gcap,
                                                    n_groups_ptr, status_ptr, stream),
                    "process_batch_cf32")

    def join(self, stream=None):
        self._check(self.L.fmgpu_join(self.h, stream), "join")

    def submit_host_raw(self, iq_ptr, stride, n_blocks, audio_ptr, acap, n_audio_ptr, groups_ptr,
                        gcap, n_groups_ptr, status_ptr) -> int:
        """Queue one host-buffer batch without waiting; returns the ticket for wait_host()."""
        t = self.L.fmgpu_submit_host(self.h, iq_ptr, stride, n_blocks, audio_ptr, acap, n_audio_ptr,
                                     groups_ptr, gcap, n_groups_ptr, status_ptr)
        if t < 0:
            self._check(t, "submit_host")
        return t

    def wait_host(self, ticket: int):
        self._check(self.L.fmgpu_wait_host(self.h, ticket), "wait_host")

    def debug_timeline(self, cap: int = 8192):
        """[(stage, group, t0_ms, t1_ms)] of the spans recorded since the last call."""
        names = (C.c_char_p * cap)()
        groups = (C.c_int32 * cap)()
        t0 = (C.c_float * cap)()
        t1 = (C.c_float * cap)()
        n = min(cap, self.L.fmgpu_debug_timeline(self.h, names, groups, t0, t1, cap))
        return [(names[i].decode(), groups[i], t0[i], t1[i]) for i in range(n)]

    def pack_pcm16(self, audio_ptr, acap, n_audio_ptr, volume_scale, pcm_ptr, stream=None):
        self._check(self.L.fmgpu_pack_pcm16(self.h, audio_ptr, acap, n_audio_ptr, volume_scale,
                                            pcm_ptr, stream), "pack_pcm16")

    def signal_level_batch(self, iq_dev_ptr, stride, n_blocks, sums_dev_ptr, stream=None):
        self._check(self.L.fmgpu_signal_level_batch(self.h, iq_dev_ptr, stride, n_blocks,
                                                    sums_dev_ptr, stream), "signal_level_batch")

    def signal_level_finish(self, sums: "LevelSums", gain_db=0, comp=0.0, bias=0.0, floor=-70.0,
                            ceil=-5.0) -> "SignalLevel":
        out = SignalLevel()
        self.L.fmgpu_signal_level_finish(C.byref(sums), gain_db, comp, bias, floor, ceil,
                                         C.byref(out))
        return out

    # ---- stage-level (reference method names) --------------------------------
    def executeComplex(self, iq: np.ndarray, out_capacity: int, channel=0) -> np.ndarray:
        iq = np.ascontiguousarray(iq, np.uint8).reshape(-1)
        out = np.zeros(2 * out_capacity, np.float32)
        n = self.L.fmgpu_decimate(self.h, channel, _ptr(iq), iq.size // 2, _ptr(out), out_capacity)
        return out[:2 * n].view(np.complex64)

    def processSplit(self, iq: np.ndarray, want_mono=False, channel=0):
        iq = np.ascontiguousarray(iq, np.uint8).reshape(-1)
        n = iq.size // 2
        mpx = np.zeros(n, np.float32)
        mono = np.zeros(n, np.float32) if want_mono else None
        k = self.L.fmgpu_demod_u8(self.h, channel, _ptr(iq), _ptr(mpx), _ptr(mono), n)
        return mpx, (mono[:k] if want_mono else None)

    def processSplitComplex(self, iq: np.ndarray, want_mono=False, channel=0):
        iq = np.ascontiguousarray(iq, np.complex64).reshape(-1)
        n = iq.size
        mpx = np.zeros(n, np.float32)
        mono = np.zeros(n, np.float32) if want_mono else None
        k = self.L.fmgpu_demod_cf32(self.h, channel, _ptr(iq), _ptr(mpx), _ptr(mono), n)
        return mpx, (mono[:k] if want_mono else None)

    def downsampleAudio(self, mpx: np.ndarray, channel=0) -> np.ndarray:
        mpx = np.ascontiguousarray(mpx, np.float32).reshape(-1)
        out = np.zeros(mpx.size, np.float32)
        n = self.L.fmgpu_downsample_mono(self.h, channel, _ptr(mpx), _ptr(out), mpx.size)
        return out[:n]

    def set_deviation_hz(self, hz: float):
        self._check(self.L.fmgpu_set_deviation_hz(self.h, float(hz)), "set_deviation_hz")

    def processAudio(self, mpx: np.ndarray, channel=0):
        mpx = np.ascontiguousarray(mpx, np.float32).reshape(-1)
        l = np.zeros(mpx.size, np.float32)
        r = np.zeros(mpx.size, np.float32)
        n = self.L.fmgpu_stereo(self.h, channel, _ptr(mpx), _ptr(l), _ptr(r), mpx.size)
        return l[:n], r[:n]

    def afpost(self, left: np.ndarray, right: np.ndarray, out_capacity: int, channel=0):
        left = np.ascontiguousarray(left, np.float32).reshape(-1)
        right = np.ascontiguousarray(right, np.float32).reshape(-1)
        ol = np.zeros(out_capacity, np.float32)
        orr = np.zeros(out_capacity, np.float32)
        n = self.L.fmgpu_afpost(self.h, channel, _ptr(left), _ptr(right), left.size, _ptr(ol),
                                _ptr(orr), out_capacity)
        return ol[:n], orr[:n]

    def rds(self, mpx: np.ndarray, channel=0, cap=64) -> np.ndarray:
        mpx = np.ascontiguousarray(mpx, np.float32).reshape(-1)
        out = np.zeros(cap, GROUP_DTYPE)
        n = self.L.fmgpu_rds(self.h, channel, _ptr(mpx), mpx.size, _ptr(out), cap)
        return out[:min(n, cap)]

    # ---- introspection ---------------------------------------------------------
    def design(self, which: int, channel: int = 0):
        buf = np.zeros(65536, np.float32)
        sc = C.c_float(0)
        n = self.L.fmgpu_get_design(self.h, which, channel, _ptr(buf), buf.size, C.byref(sc))
        return buf[:n].copy(), sc.value

    def debug_read(self, which: int, channel: int = 0) -> np.ndarray:
        buf = np.zeros(2 * self.cfg.block_samples * self.cfg.max_blocks + 16, np.float32)
        n = self.L.fmgpu_debug_read(self.h, which, channel, _ptr(buf), buf.size)
        out = buf[:n].copy()
        return out.view(np.complex64) if which == 0 else out

    def debug_rds_bits(self, channel: int = 0) -> np.ndarray:
        buf = np.zeros(1 << 16, np.uint8)
        n = self.L.fmgpu_debug_rds_bits(self.h, channel, _ptr(buf), buf.size)
        return buf[:n].copy()

    def launch_count(self) -> int:
        return int(self.L.fmgpu_launch_count(self.h))

    def enable_stage_timing(self, on=True):
        self.L.fmgpu_enable_stage_timing(self.h, int(on))

    def stage_times(self) -> dict:
        names = (C.c_char_p * 32)()
        ms = (C.c_float * 32)()
        n = self.L.fmgpu_get_stage_times(self.h, names, ms, 32)
        return {names[i].decode(): float(ms[i]) for i in range(min(n, 32))}


class XdrRdsState(C.Structure):
    _fields_ = [("pi_buffer", C.c_uint16 * 64), ("pi_error", C.c_uint8 * 8), ("pi_fill", C.c_uint8),
                ("pi_pos", C.c_uint8), ("pi_last_state", C.c_uint8), ("pad", C.c_uint8),
                ("pi_last_value", C.c_uint16)]


class XdrRdsFormatter:
    """Per-channel XDR / FM-DX view of an RDS stream (fmgpu_xdr_rds_*: XDRServer::updateRDS)."""

    def __init__(self):
        self.L = load_library()
        self.L.fmgpu_xdr_rds_init.argtypes = [C.POINTER(XdrRdsState)]
        self.L.fmgpu_xdr_rds_init.restype = None
        self.L.fmgpu_xdr_rds_lines.argtypes = [C.POINTER(XdrRdsState), C.c_void_p, C.c_char_p]
        self.state = XdrRdsState()
        self.reset()

    def reset(self):
        self.L.fmgpu_xdr_rds_init(C.byref(self.state))

    def lines(self, group) -> list:
        """group: one element of a GROUP_DTYPE array -> the text lines it produces."""
        one = np.array([group], GROUP_DTYPE)
        buf = C.create_string_buffer(64)
        n = self.L.fmgpu_xdr_rds_lines(C.byref(self.state), one.ctypes.data, buf)
        return [buf.raw[32 * i:32 * i + 32].split(b"\0")[0].decode() for i in range(n)]


SAMPLE_FORMATS = {"cu8": 0, "cs8": 1, "cs16": 2}     # include/fmgpu.h FMGPU_IQ_*
PAIR_BYTES = {"cu8": 2, "cs8": 2, "cs16": 4}


class Channelizer:
    """Wideband front end for BASELINE config 4 (include/fmgpu.h: fmgpu_channelizer_*): one IQ
    capture -> n_channels complex-float streams at wide_rate / decimation.

    sample_format is the captures' I,Q pair format: "cu8" (uint8 offset binary, RTL-SDR), "cs8"
    (int8, HackRF) or "cs16" (int16, USRP / bladeRF / LimeSDR / SDRplay, SoapySDR CS16).

    first_center_hz may be a sequence: one capture per entry, all advancing together, capture w's
    carrier k at first_center_hz[w] + k * spacing_hz from its own centre; its outputs are
    n_captures * ch_count rows, capture-major.

    output_rate, when given, replaces decimation: the object resamples by the reduced ratio
    U / D = output_rate / wide_rate (fmgpu_channelizer_create_rate, U <= 64), and a call writes a
    varying number of outputs (outputs(), process_stream())."""

    def __init__(self, wide_rate=24_000_000, decimation=100, n_channels=100,
                 first_center_hz=-9_900_000.0, spacing_hz=200_000.0, taps_per_phase=16,
                 cutoff_hz=100_000.0, atten_db=60.0, device=0, sample_format="cu8", output_rate=None):
        if sample_format not in SAMPLE_FORMATS:
            raise ValueError(f"sample_format must be one of {sorted(SAMPLE_FORMATS)}, not {sample_format!r}")
        self.L = load_library()
        self.h = None
        h = C.c_void_p()
        firsts = [float(first_center_hz)] if np.ndim(first_center_hz) == 0 else \
            [float(f) for f in first_center_hz]
        arr = (C.c_double * len(firsts))(*firsts)
        if output_rate is None:
            create, rate = self.L.fmgpu_channelizer_create_format, decimation
        else:
            create, rate = self.L.fmgpu_channelizer_create_rate, output_rate
        rc = create(device, SAMPLE_FORMATS[sample_format], len(firsts), wide_rate, rate, n_channels, arr,
                    spacing_hz, taps_per_phase, cutoff_hz, atten_db, C.byref(h))
        if rc != 0:
            raise EngineError(f"{create.__name__} failed ({rc}); no CPU fallback")
        if np.ndim(first_center_hz) != 0:
            first_center_hz = firsts
        self.h = h
        self._format = sample_format
        self.wide_rate, self.n_channels = wide_rate, n_channels
        self.decimation = self.L.fmgpu_channelizer_decimation(h)
        self.first_center_hz, self.spacing_hz = first_center_hz, spacing_hz

    @property
    def output_rate(self) -> int:
        return self.L.fmgpu_channelizer_output_rate(self.h)

    @property
    def interpolation(self) -> int:
        """U of the rate ratio U / D (1 unless output_rate was given)."""
        return self.L.fmgpu_channelizer_interpolation(self.h)

    @property
    def n_captures(self) -> int:
        return self.L.fmgpu_channelizer_n_captures(self.h)

    @property
    def sample_format(self) -> str:
        return self._format

    @property
    def pair_bytes(self) -> int:
        """Bytes of one I,Q pair of the input."""
        return PAIR_BYTES[self._format]

    def taps(self) -> np.ndarray:
        n = self.L.fmgpu_channelizer_taps(self.h, None, 0)
        out = np.zeros(n, np.float32)
        self.L.fmgpu_channelizer_taps(self.h, _ptr(out), n)
        return out

    def process(self, iq_dev_ptr, n_in, out_dev_ptr, out_stride_samples, ch_first=0, ch_count=None,
                stream=None, iq_stride_bytes=None):
        """iq [n_captures][iq_stride_bytes] (default pair_bytes * n_in): n_in pairs per capture;
        out [n_captures][ch_count][out_stride_samples] (fmgpu_channelizer_process_iq)."""
        ch_count = self.n_channels - ch_first if ch_count is None else ch_count
        stride = self.pair_bytes * n_in if iq_stride_bytes is None else iq_stride_bytes
        rc = self.L.fmgpu_channelizer_process_iq(self.h, iq_dev_ptr, stride, n_in, ch_first, ch_count,
                                                 out_dev_ptr, out_stride_samples, stream)
        if rc != 0:
            raise EngineError(f"fmgpu_channelizer_process_iq failed ({rc})")

    def outputs(self, n_in) -> int:
        """Outputs per row the next call with n_in pairs per capture writes."""
        return self.L.fmgpu_channelizer_outputs(self.h, n_in)

    def process_stream(self, iq_dev_ptr, n_in, out_dev_ptr, out_stride_samples, ch_first=0, ch_count=None,
                       stream=None, iq_stride_bytes=None) -> int:
        """As process, for any object and any n_in >= 1 (fmgpu_channelizer_process_stream): writes
        outputs [0, n_out) of every row and returns n_out."""
        ch_count = self.n_channels - ch_first if ch_count is None else ch_count
        stride = self.pair_bytes * n_in if iq_stride_bytes is None else iq_stride_bytes
        n_out = C.c_size_t()
        rc = self.L.fmgpu_channelizer_process_stream(self.h, iq_dev_ptr, stride, n_in, ch_first, ch_count,
                                                     out_dev_ptr, out_stride_samples, C.byref(n_out), stream)
        if rc != 0:
            raise EngineError(f"fmgpu_channelizer_process_stream failed ({rc})")
        return n_out.value

    def close(self):
        if self.h:
            self.L.fmgpu_channelizer_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

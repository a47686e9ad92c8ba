"""oracle/orc.py — TEST INFRASTRUCTURE, NOT PRODUCT CODE.

ctypes binding over the CPU oracle (oracle_capi.cpp), the synthetic signal generator
(siggen.cpp) and, when built, the reference's own integer RDS back end
(oracle/_ref/libredsea_ref.so). Only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs may import this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass, field

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def build(force: bool = False) -> None:
    """Compile the oracle (and oracle/_ref when /root/reference is present) if stale."""
    def mtime(f):
        return os.path.getmtime(os.path.join(HERE, f))

    def stale(target, deps):
        return (not os.path.exists(os.path.join(HERE, target))) or mtime(target) < max(map(mtime, deps))

    oracle_deps = ("oracle_capi.cpp", "pipeline.hpp", "liquid_restated.hpp", "Makefile",
                   os.path.join("..", "fmtuner_sdr_b200", "csrc", "fm_math.h"))
    ref_deps = ("oracle_capi.cpp", "liquid_restated.hpp", "Makefile",
                os.path.join("liquid_shim", "liquid_shim.cpp"),
                os.path.join("liquid_shim", "liquid", "liquid.h"))
    need = force or any(stale(f"liboracle_{m}.so", oracle_deps) for m in ("libm", "libm_contract", "fm")) \
        or stale("libsiggen.so", ("siggen.cpp", "Makefile"))
    have_ref_src = os.path.isdir("/root/reference/src/redsea_port")
    ref_missing = have_ref_src and not all(
        os.path.exists(os.path.join(HERE, "_ref", f))
        for f in ("libredsea_ref.so", "libsiglevel_ref.so", "libxdr_ref.so", "libfmref.so",
                  "libfmref_contract.so"))
    if have_ref_src and not ref_missing:
        ref_missing = stale(os.path.join("_ref", "libfmref.so"), ref_deps)
    if need or ref_missing:
        subprocess.run(["make", "-C", HERE, "--no-print-directory"], check=True,
                       stdout=subprocess.DEVNULL)


class Config(C.Structure):
    _fields_ = [
        ("iq_rate", C.c_int32),
        ("decimation", C.c_int32),
        ("block_samples", C.c_int32),
        ("w0_bandwidth_hz", C.c_int32),
        ("bandwidth_hz", C.c_int32),
        ("dsp_agc", C.c_int32),
        ("stereo_blend", C.c_int32),
        ("deemphasis", C.c_int32),
        ("stereo", C.c_int32),
        ("force_mono", C.c_int32),
    ]


def make_config(iq_rate=2_400_000, decimation=10, block_samples=8192, w0_bandwidth_hz=194000,
                bandwidth_hz=0, dsp_agc=0, stereo_blend=1, deemphasis=0, stereo=1,
                force_mono=0) -> Config:
    return Config(iq_rate, decimation, block_samples, w0_bandwidth_hz, bandwidth_hz, dsp_agc,
                  stereo_blend, deemphasis, stereo, force_mono)


class BlockStatus(C.Structure):
    _fields_ = [
        ("n_audio", C.c_int32),
        ("stereo", C.c_int32),
        ("pilot_tenths", C.c_int32),
        ("clip_ratio", C.c_float),
        ("n_groups", C.c_int32),
    ]


class Group(C.Structure):
    _fields_ = [
        ("a", C.c_uint16),
        ("b", C.c_uint16),
        ("c", C.c_uint16),
        ("d", C.c_uint16),
        ("errors", C.c_uint8),
        ("pad", C.c_uint8 * 3),
        ("block_index", C.c_uint32),
    ]


GROUP_DTYPE = np.dtype([("a", "<u2"), ("b", "<u2"), ("c", "<u2"), ("d", "<u2"), ("errors", "u1"),
                        ("pad", "u1", 3), ("block_index", "<u4")])
STATUS_DTYPE = np.dtype([("n_audio", "<i4"), ("stereo", "<i4"), ("pilot_tenths", "<i4"),
                         ("clip_ratio", "<f4"), ("n_groups", "<i4")])


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


class OracleLib:
    """One flavour of the oracle: math='libm' (faithful) or 'fm' (engine-shared kernels) are the
    restated pipeline, 'libm_contract' the faithful one with gcc's default FMA contraction; 'ref'
    is the REFERENCE's own sources compiled unmodified over
    liquid_shim/ (oracle/_ref/libfmref.so, -ffp-contract=off) and 'ref_contract' the same with
    gcc's default FMA contraction. The reference flavours have the channel- and class-level
    entry points only (no design getters, no block-sync / math hooks)."""

    REF_LIBS = {"ref": "libfmref.so", "ref_contract": "libfmref_contract.so"}

    @classmethod
    def ref_path(cls, math: str = "ref") -> str:
        return os.path.join(HERE, "_ref", cls.REF_LIBS[math])

    @classmethod
    def have_ref(cls, math: str = "ref") -> bool:
        build()
        return os.path.exists(cls.ref_path(math))

    def __init__(self, math: str = "fm"):
        build()
        self.math = math
        self.is_ref = math in self.REF_LIBS
        path = self.ref_path(math) if self.is_ref else os.path.join(HERE, f"liboracle_{math}.so")
        self.lib = C.CDLL(path)
        L = self.lib
        L.orc_math_name.restype = C.c_char_p
        L.orc_channel_create.restype = C.c_void_p
        L.orc_channel_create.argtypes = [C.POINTER(Config)]
        L.orc_channel_destroy.argtypes = [C.c_void_p]
        L.orc_channel_reset.argtypes = [C.c_void_p, C.c_int, C.c_int]
        for n in ("set_bandwidth_hz", "set_force_mono", "set_force_stereo", "set_deemphasis"):
            getattr(L, f"orc_channel_{n}").argtypes = [C.c_void_p, C.c_int]
        L.orc_channel_process.restype = C.c_long
        L.orc_channel_process.argtypes = [
            C.c_void_p, C.POINTER(C.c_uint8), C.c_size_t, C.POINTER(C.c_float),
            C.POINTER(C.c_float), C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t,
            C.POINTER(C.c_size_t), C.POINTER(C.c_float), C.POINTER(C.c_float),
            C.POINTER(C.c_float), C.POINTER(C.c_float)]
        L.orc_channel_rds_bits.restype = C.c_size_t
        L.orc_channel_rds_bits.argtypes = [C.c_void_p, C.POINTER(C.c_uint8), C.c_size_t]
        L.orc_channel_enable_bits_tap.argtypes = [C.c_void_p]
        # class-level
        L.orc_decim_create.restype = C.c_void_p
        L.orc_decim_create.argtypes = [C.c_uint32, C.c_uint32, C.c_float]
        L.orc_decim_destroy.argtypes = [C.c_void_p]
        L.orc_decim_reset.argtypes = [C.c_void_p]
        L.orc_decim_execute_complex.restype = C.c_size_t
        L.orc_decim_execute_complex.argtypes = [C.c_void_p, C.POINTER(C.c_uint8), C.c_size_t,
                                                C.POINTER(C.c_float), C.c_size_t]
        L.orc_decim_execute_u8.restype = C.c_size_t
        L.orc_decim_execute_u8.argtypes = [C.c_void_p, C.POINTER(C.c_uint8), C.c_size_t,
                                           C.POINTER(C.c_uint8), C.c_size_t]
        L.orc_demod_create.restype = C.c_void_p
        L.orc_demod_create.argtypes = [C.c_int, C.c_int]
        L.orc_demod_destroy.argtypes = [C.c_void_p]
        L.orc_demod_reset.argtypes = [C.c_void_p]
        for n in ("set_w0", "set_bandwidth_hz", "set_bandwidth_mode", "set_agc", "set_deemphasis"):
            getattr(L, f"orc_demod_{n}").argtypes = [C.c_void_p, C.c_int]
        L.orc_demod_process_split.restype = C.c_size_t
        L.orc_demod_process_split.argtypes = [C.c_void_p, C.POINTER(C.c_uint8),
                                              C.POINTER(C.c_float), C.POINTER(C.c_float),
                                              C.c_size_t]
        L.orc_demod_process_split_complex.restype = C.c_size_t
        L.orc_demod_process_split_complex.argtypes = [C.c_void_p, C.POINTER(C.c_float),
                                                      C.POINTER(C.c_float), C.POINTER(C.c_float),
                                                      C.c_size_t]
        L.orc_demod_set_deviation.argtypes = [C.c_void_p, C.c_double]
        L.orc_demod_downsample.restype = C.c_size_t
        L.orc_demod_downsample.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                           C.c_size_t]
        L.orc_demod_clip_ratio.restype = C.c_float
        L.orc_demod_clip_ratio.argtypes = [C.c_void_p]
        L.orc_demod_is_clipping.argtypes = [C.c_void_p]
        L.orc_stereo_create.restype = C.c_void_p
        L.orc_stereo_create.argtypes = [C.c_int]
        L.orc_stereo_destroy.argtypes = [C.c_void_p]
        L.orc_stereo_reset.argtypes = [C.c_void_p]
        for n in ("set_blend", "set_force_mono", "set_force_stereo"):
            getattr(L, f"orc_stereo_{n}").argtypes = [C.c_void_p, C.c_int]
        L.orc_stereo_process.restype = C.c_size_t
        L.orc_stereo_process.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                         C.POINTER(C.c_float), C.c_size_t]
        L.orc_stereo_is_stereo.argtypes = [C.c_void_p]
        L.orc_stereo_pilot_tenths.argtypes = [C.c_void_p]
        L.orc_afpost_create.restype = C.c_void_p
        L.orc_afpost_create.argtypes = [C.c_int, C.c_int]
        L.orc_afpost_destroy.argtypes = [C.c_void_p]
        L.orc_afpost_reset.argtypes = [C.c_void_p]
        L.orc_afpost_set_deemphasis.argtypes = [C.c_void_p, C.c_int]
        L.orc_afpost_process.restype = C.c_size_t
        L.orc_afpost_process.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                         C.c_size_t, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                         C.c_size_t]
        L.orc_rds_create.restype = C.c_void_p
        L.orc_rds_create.argtypes = [C.c_int]
        L.orc_rds_destroy.argtypes = [C.c_void_p]
        L.orc_rds_reset.argtypes = [C.c_void_p]
        L.orc_rds_process.restype = C.c_size_t
        L.orc_rds_process.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.c_size_t, C.c_void_p,
                                      C.c_size_t]
        if self.is_ref:
            return
        L.orc_rds_bits.restype = C.c_size_t
        L.orc_rds_bits.argtypes = [C.c_void_p, C.POINTER(C.c_uint8), C.c_size_t]
        L.orc_blockstream_run.restype = C.c_size_t
        L.orc_blockstream_run.argtypes = [C.POINTER(C.c_uint8), C.c_size_t, C.c_void_p, C.c_size_t]
        L.orc_rds_syndrome.restype = C.c_uint32
        L.orc_rds_syndrome.argtypes = [C.c_uint32]
        L.orc_design.restype = C.c_size_t
        L.orc_design.argtypes = [C.c_int, C.c_int, C.c_int, C.c_float, C.POINTER(C.c_float),
                                 C.c_size_t, C.POINTER(C.c_float)]
        for n in ("exp", "log"):
            getattr(L, f"orc_math_{n}").argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float),
                                                    C.c_size_t]
        L.orc_math_sincos.argtypes = [C.POINTER(C.c_float)] * 3 + [C.c_size_t]
        L.orc_math_atan2.argtypes = [C.POINTER(C.c_float)] * 3 + [C.c_size_t]
        L.orc_nco_constrain.restype = C.c_uint32
        L.orc_nco_constrain.argtypes = [C.c_float]

    # -- helpers -------------------------------------------------------------
    def design(self, which: int, a: int = 0, b: int = 0, fa: float = 0.0):
        buf = np.zeros(65536, np.float32)
        sc = C.c_float(0)
        n = self.lib.orc_design(which, a, b, fa, _p(buf, C.c_float), buf.size, C.byref(sc))
        return buf[:n].copy(), sc.value

    def blockstream(self, bits: np.ndarray) -> np.ndarray:
        bits = np.ascontiguousarray(bits, np.uint8)
        out = np.zeros(max(4, bits.size // 26 + 4), GROUP_DTYPE)
        n = self.lib.orc_blockstream_run(_p(bits, C.c_uint8), bits.size, out.ctypes.data, out.size)
        return out[:n]


@dataclass
class ChannelResult:
    left: np.ndarray
    right: np.ndarray
    status: np.ndarray   # STATUS_DTYPE per block
    groups: np.ndarray   # GROUP_DTYPE
    dec: np.ndarray | None = None
    mpx: np.ndarray | None = None
    sl: np.ndarray | None = None
    sr: np.ndarray | None = None


class Channel:
    """The reference's per-block pipeline for one channel (src/main.cpp:1232-1308)."""

    def __init__(self, lib: OracleLib, cfg: Config):
        self.L = lib
        self.cfg = cfg
        self.h = lib.lib.orc_channel_create(C.byref(cfg))
        if not self.h:
            raise RuntimeError("oracle channel creation failed")

    def __del__(self):
        if getattr(self, "h", None):
            self.L.lib.orc_channel_destroy(self.h)
            self.h = None

    def reset(self, dsp=True, rds=True):
        self.L.lib.orc_channel_reset(self.h, int(dsp), int(rds))

    def set_bandwidth_hz(self, bw):
        self.L.lib.orc_channel_set_bandwidth_hz(self.h, bw)

    def set_force_mono(self, f):
        self.L.lib.orc_channel_set_force_mono(self.h, int(f))

    def set_force_stereo(self, f):
        self.L.lib.orc_channel_set_force_stereo(self.h, int(f))

    def set_deemphasis(self, mode):
        self.L.lib.orc_channel_set_deemphasis(self.h, mode)

    def process(self, iq: np.ndarray, debug: bool = False) -> ChannelResult:
        iq = np.ascontiguousarray(iq, np.uint8).reshape(-1)
        n = self.cfg.block_samples
        per_block = n * self.cfg.decimation * 2
        nblk = iq.size // per_block
        cap = nblk * n
        outL = np.zeros(cap, np.float32)
        outR = np.zeros(cap, np.float32)
        status = np.zeros(nblk, STATUS_DTYPE)
        groups = np.zeros(nblk * 2 + 8, GROUP_DTYPE)
        ng = C.c_size_t(0)
        dec = np.zeros(2 * cap, np.float32) if debug and self.cfg.decimation > 1 else None
        mpx = np.zeros(cap, np.float32) if debug else None
        sl = np.zeros(cap, np.float32) if debug else None
        sr = np.zeros(cap, np.float32) if debug else None
        tot = self.L.lib.orc_channel_process(
            self.h, _p(iq, C.c_uint8), nblk, _p(outL, C.c_float), _p(outR, C.c_float), cap,
            status.ctypes.data, groups.ctypes.data, groups.size, C.byref(ng),
            _p(dec, C.c_float), _p(mpx, C.c_float), _p(sl, C.c_float), _p(sr, C.c_float))
        if tot < 0:
            raise RuntimeError("oracle capacity exceeded")
        return ChannelResult(outL[:tot], outR[:tot], status, groups[:ng.value].copy(),
                             dec.view(np.complex64) if dec is not None else None, mpx, sl, sr)

    def enable_bits_tap(self):
        """Reference flavours: collect demodulated bits from now on (rds_bits())."""
        self.L.lib.orc_channel_enable_bits_tap(self.h)

    def rds_bits(self) -> np.ndarray:
        n = self.L.lib.orc_channel_rds_bits(self.h, None, 0)
        out = np.zeros(n, np.uint8)
        self.L.lib.orc_channel_rds_bits(self.h, _p(out, C.c_uint8), n)
        return out


# ---------------------------------------------------------------------------
# signal generator
# ---------------------------------------------------------------------------
class SigParams(C.Structure):
    _fields_ = [
        ("fs_iq", C.c_double), ("deviation", C.c_double),
        ("tone_l_hz", C.c_double), ("tone_l_amp", C.c_double),
        ("tone_r_hz", C.c_double), ("tone_r_amp", C.c_double),
        ("audio_gain", C.c_double), ("pilot_amp", C.c_double), ("rds_amp", C.c_double),
        ("iq_amp", C.c_double), ("snr_db", C.c_double), ("freq_offset_hz", C.c_double),
        ("dc_i", C.c_double), ("dc_q", C.c_double),
        ("seed", C.c_uint64), ("start_sample", C.c_uint64),
    ]


_sig = None


def _siglib():
    global _sig
    if _sig is None:
        build()
        _sig = C.CDLL(os.path.join(HERE, "libsiggen.so"))
        _sig.sig_generate.argtypes = [C.POINTER(SigParams), C.POINTER(C.c_uint8), C.c_size_t,
                                      C.POINTER(C.c_uint8), C.c_size_t]
        _sig.sig_rds_encode_block.restype = C.c_uint32
        _sig.sig_rds_encode_block.argtypes = [C.c_uint16, C.c_int]
    return _sig


def rds_encode_groups(groups) -> np.ndarray:
    """groups: iterable of (A, B, C, D[, version_b]) -> bit array (MSB first)."""
    lib = _siglib()
    bits = []
    for g in groups:
        a, b, c, d = g[:4]
        vb = bool(g[4]) if len(g) > 4 else bool((b >> 11) & 1)
        for word, off in ((a, 0), (b, 1), (c, 3 if vb else 2), (d, 4)):
            blk = lib.sig_rds_encode_block(word, off)
            bits.extend((blk >> (25 - i)) & 1 for i in range(26))
    return np.array(bits, np.uint8)


def rds_groups_ps_rt(pi: int, ps: str, rt: str = "", pty: int = 10):
    """Group sequence: four 0A groups carrying PS, then 2A groups carrying RT."""
    ps = (ps + " " * 8)[:8]
    out = []
    for seg in range(4):
        b = (0 << 12) | (0 << 11) | (pty << 5) | (1 << 3) | seg
        out.append((pi, b, 0xE0CD, (ord(ps[2 * seg]) << 8) | ord(ps[2 * seg + 1])))
    if rt:
        rt = rt + "\r"
        rt = rt + " " * ((-len(rt)) % 4)
        for seg in range(min(16, len(rt) // 4)):
            b = (2 << 12) | (0 << 11) | (pty << 5) | seg
            ch = [ord(x) for x in rt[4 * seg:4 * seg + 4]]
            out.append((pi, b, (ch[0] << 8) | ch[1], (ch[2] << 8) | ch[3]))
    return out


def decode_ps_rt(groups: np.ndarray):
    """Test-side decoder of 0A/2A groups -> (pi, ps, rt) using only error-free blocks."""
    ps = [" "] * 8
    rt = [" "] * 64
    pi = None
    for g in groups:
        e = int(g["errors"])
        ea, eb, ec, ed = (e >> 6) & 3, (e >> 4) & 3, (e >> 2) & 3, e & 3
        if ea == 0:
            pi = int(g["a"])
        if eb != 0:
            continue
        gt = int(g["b"]) >> 11
        if gt == 0 and ed == 0:
            seg = int(g["b"]) & 3
            ps[2 * seg] = chr(int(g["d"]) >> 8)
            ps[2 * seg + 1] = chr(int(g["d"]) & 0xFF)
        elif gt == 4 and ec == 0 and ed == 0:
            seg = int(g["b"]) & 15
            for k, v in enumerate((int(g["c"]) >> 8, int(g["c"]) & 0xFF, int(g["d"]) >> 8,
                                   int(g["d"]) & 0xFF)):
                rt[4 * seg + k] = chr(v)
    return pi, "".join(ps), "".join(rt).split("\r")[0].rstrip()


@dataclass
class Signal:
    fs_iq: float = 2_400_000.0
    deviation: float = 75_000.0
    tone_l_hz: float = 1000.0
    tone_l_amp: float = 1.0
    tone_r_hz: float = 0.0
    tone_r_amp: float = 0.0
    audio_gain: float = 0.43
    pilot_amp: float = 0.10
    rds_amp: float = 0.04
    iq_amp: float = 0.5
    snr_db: float = 300.0
    freq_offset_hz: float = 0.0
    dc_i: float = 0.0
    dc_q: float = 0.0
    seed: int = 0
    rds_bits: np.ndarray = field(default_factory=lambda: np.zeros(0, np.uint8))

    def generate(self, n_samples: int, start_sample: int = 0) -> np.ndarray:
        lib = _siglib()
        p = SigParams(self.fs_iq, self.deviation, self.tone_l_hz, self.tone_l_amp, self.tone_r_hz,
                      self.tone_r_amp, self.audio_gain, self.pilot_amp, self.rds_amp, self.iq_amp,
                      self.snr_db, self.freq_offset_hz, self.dc_i, self.dc_q, self.seed,
                      start_sample)
        bits = np.ascontiguousarray(self.rds_bits, np.uint8)
        out = np.zeros(2 * n_samples, np.uint8)
        rc = lib.sig_generate(C.byref(p), _p(bits, C.c_uint8) if bits.size else None, bits.size,
                              _p(out, C.c_uint8), n_samples)
        if rc != 0:
            raise RuntimeError("sig_generate failed")
        return out


def config1_signal(fs_iq=2_400_000.0, seed=0) -> Signal:
    """BASELINE config 1: 1 kHz L-only tone, pilot, RDS PI 0x1234 PS 'B200TEST' + RT."""
    groups = rds_groups_ps_rt(0x1234, "B200TEST", "FM ON B200")
    return Signal(fs_iq=fs_iq, seed=seed, rds_bits=rds_encode_groups(groups))


def config3_signal(c: int, fs_iq=2_400_000.0) -> Signal:
    """BASELINE config 3 channel c (SURVEY §8(d))."""
    rng = np.random.default_rng(1000 + c)
    dev = float(rng.choice([22_500.0, 37_500.0, 50_000.0, 60_000.0, 75_000.0]))
    snr = float(rng.uniform(20.0, 60.0))
    groups = rds_groups_ps_rt(0x1000 + c, f"CH{c:04d}  ", f"CHANNEL {c}")
    return Signal(fs_iq=fs_iq, deviation=dev, tone_l_hz=400.0 + 37.0 * c, tone_l_amp=0.8,
                  tone_r_hz=700.0 + 53.0 * c, tone_r_amp=0.8, snr_db=snr, seed=c,
                  rds_bits=rds_encode_groups(groups))


def ref_blockstream(bits: np.ndarray):
    """The REFERENCE's own BlockStream (oracle/_ref); None when it was not built."""
    path = os.path.join(HERE, "_ref", "libredsea_ref.so")
    if not os.path.exists(path):
        return None
    lib = C.CDLL(path)
    lib.ref_blockstream_run.restype = C.c_size_t
    lib.ref_blockstream_run.argtypes = [C.POINTER(C.c_uint8), C.c_size_t, C.c_void_p, C.c_size_t]
    bits = np.ascontiguousarray(bits, np.uint8)
    out = np.zeros(max(4, bits.size // 26 + 4), GROUP_DTYPE)
    n = lib.ref_blockstream_run(_p(bits, C.c_uint8), bits.size, out.ctypes.data, out.size)
    return out[:n]


def signal_level(iq: np.ndarray, gain_db=0, comp=0.0, bias=0.0, floor=-70.0, ceil=-5.0):
    """RF level of one block of IQ bytes: the REFERENCE's computeSignalLevel when oracle/_ref was
    built, else a numpy restatement of src/signal_level.cpp:145-203 (sequential double sums).
    Returns (level120, dbfs, compensated_dbfs, hard_clip_ratio, near_clip_ratio, source)."""
    iq = np.ascontiguousarray(iq, np.uint8).reshape(-1)
    n = iq.size // 2
    path = os.path.join(HERE, "_ref", "libsiglevel_ref.so")
    if os.path.exists(path):
        lib = C.CDLL(path)
        lib.ref_compute_signal_level.argtypes = [C.POINTER(C.c_uint8), C.c_size_t, C.c_int, C.c_double,
                                                 C.c_double, C.c_double, C.c_double,
                                                 C.POINTER(C.c_double)]
        out = (C.c_double * 5)()
        lib.ref_compute_signal_level(_p(iq, C.c_uint8), n, gain_db, comp, bias, floor, ceil, out)
        return (float(np.float32(out[0])), out[1], out[2], out[3], out[4], "reference")
    i = (iq[0::2].astype(np.float64) - 127.5) * (1.0 / 127.5)
    q = (iq[1::2].astype(np.float64) - 127.5) * (1.0 / 127.5)
    s_i, s_q = np.cumsum(i)[-1], np.cumsum(q)[-1]
    s_ii, s_qq = np.cumsum(i * i)[-1], np.cumsum(q * q)[-1]
    ib, qb = iq[0::2], iq[1::2]
    hard = 2 * int(((ib <= 1) | (ib >= 254) | (qb <= 1) | (qb >= 254)).sum())
    near = 2 * int(((ib <= 8) | (ib >= 247) | (qb <= 8) | (qb >= 247)).sum())
    mi, mq = s_i / n, s_q / n
    var_i = max(0.0, s_ii / n - mi * mi)
    var_q = max(0.0, s_qq / n - mq * mq)
    rms = np.sqrt(max(1e-15, 0.5 * (var_i + var_q)))
    dbfs = 20.0 * np.log10(rms + 1e-12)
    cdb = dbfs - gain_db * comp + bias
    norm = (cdb - floor) / (max(ceil, floor + 1.0) - floor)
    lvl = float(np.clip(np.float32(norm * 120.0), np.float32(0), np.float32(120)))
    return (lvl, dbfs, cdb, hard / (2.0 * n), near / (2.0 * n), "restated")

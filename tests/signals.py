"""Test signals beyond uint8: the oracle's FM-stereo + RDS generator before its quantisation.

generate_cf64(sig, n) returns the complex128 samples x (full scale 1) of which oracle.orc.Signal's
generate(n) is the uint8 quantisation clip(round(127.5 + 127.5 x), 0, 255) (tests/siggen_cf64.cpp).
The library is compiled on first use into a per-user directory under the system's temporary
directory, keyed by the sources, so a read-only checkout works."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import orc

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "siggen_cf64.cpp")
DEPS = (SRC, os.path.join(HERE, "..", "oracle", "siggen.cpp"))
# oracle/Makefile's flags for libsiggen.so: the restated loop rounds exactly as sig_generate does
FLAGS = ["-std=c++17", "-O2", "-fPIC", "-shared"]
_lib = None


def _library():
    global _lib
    if _lib is not None:
        return _lib
    h = hashlib.sha256(" ".join(FLAGS).encode())
    for d in DEPS:
        with open(d, "rb") as f:
            h.update(f.read())
    out_dir = os.path.join(tempfile.gettempdir(), f"fmgpu_siggen_cf64_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"libsiggen_cf64_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run([os.environ.get("CXX", "g++")] + FLAGS + ["-o", tmp, SRC], check=True)
        os.replace(tmp, so)
    lib = C.CDLL(so)
    lib.sig_generate_cf64.argtypes = [C.POINTER(orc.SigParams), C.POINTER(C.c_uint8), C.c_size_t,
                                      C.POINTER(C.c_double), C.c_size_t]
    _lib = lib
    return lib


def generate_cf64(sig: "orc.Signal", n_samples: int, start_sample: int = 0) -> np.ndarray:
    """sig.generate(n_samples, start_sample) before quantisation, complex128."""
    lib = _library()
    p = orc.SigParams(sig.fs_iq, sig.deviation, sig.tone_l_hz, sig.tone_l_amp, sig.tone_r_hz,
                      sig.tone_r_amp, sig.audio_gain, sig.pilot_amp, sig.rds_amp, sig.iq_amp,
                      sig.snr_db, sig.freq_offset_hz, sig.dc_i, sig.dc_q, sig.seed, start_sample)
    bits = np.ascontiguousarray(sig.rds_bits, np.uint8)
    out = np.zeros(2 * n_samples, np.float64)
    rc = lib.sig_generate_cf64(C.byref(p), bits.ctypes.data_as(C.POINTER(C.c_uint8)) if bits.size else None,
                               bits.size, out.ctypes.data_as(C.POINTER(C.c_double)), n_samples)
    if rc != 0:
        raise RuntimeError("sig_generate_cf64 failed")
    return out.view(np.complex128)

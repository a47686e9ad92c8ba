"""tests/signals.generate_cf64 (sig_generate_cf64) is the oracle generator's sample loop before
quantisation: the generator's own rule, clip(round(127.5 + 127.5 x), 0, 255), turns it into
oracle.orc.Signal.generate's bytes exactly."""
import numpy as np
import pytest

from oracle import orc
from tests.signals import generate_cf64


def _u8(x: np.ndarray) -> np.ndarray:
    out = np.empty(2 * x.size, np.uint8)
    out[0::2] = np.clip(np.round(127.5 + 127.5 * x.real), 0, 255)
    out[1::2] = np.clip(np.round(127.5 + 127.5 * x.imag), 0, 255)
    return out


@pytest.mark.parametrize("kw, start", [
    (dict(), 0),                                                         # config-1-like, no noise
    (dict(snr_db=18.0, dc_i=0.03, dc_q=-0.02, freq_offset_hz=123_456.0, seed=9), 0),
    (dict(snr_db=25.0, iq_amp=1.3, seed=4), 0),                          # clips at both rails
    (dict(snr_db=30.0, seed=5), 77_777),                                 # a later piece of the stream
])
def test_cf64_quantises_to_generate(kw, start):
    sig = orc.Signal(rds_bits=orc.rds_encode_groups(orc.rds_groups_ps_rt(0x1234, "B200TEST")), **kw)
    n = 60_000
    x = generate_cf64(sig, n, start)
    assert x.dtype == np.complex128 and x.shape == (n,)
    assert np.array_equal(_u8(x), sig.generate(n, start))

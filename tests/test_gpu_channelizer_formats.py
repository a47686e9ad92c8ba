"""Sample formats of the channelizer (fmgpu_channelizer_create_format / _process_iq): signed 8-bit
(cs8, HackRF) and signed 16-bit (cs16, USRP / bladeRF / LimeSDR / SDRplay) captures beside RTL's
unsigned bytes (cu8).

Each format must give the header's definition with its own conversion of x, in both forms and across
calls; cs8 and cs16 carrying the same values must give the same bits; and a station 70 dB below a
strong one, which uint8 samples cannot carry, must decode from cs16 through the engine exactly as the
oracle's reference classes decode the same channelizer output."""
import ctypes as C
import os

import numpy as np
import pytest

import fmtuner_sdr_b200 as fm
from oracle import orc
from tests.common import groups_equal
from tests.signals import generate_cf64
from tests.test_gpu_channelizer import _oracle_chain

pytestmark = pytest.mark.gpu
EINVAL = -1
CU8, CS8, CS16 = 0, 1, 2
SCALE = {"cs8": 128.0, "cs16": 32768.0}
DTYPE = {"cs8": np.int8, "cs16": np.int16}


def _model(z, first_center_hz: float, x: np.ndarray, ks, n_out: int) -> np.ndarray:
    """float64 evaluation of y_k[m] = sum_n h[n] x[mD-n] exp(-j 2 pi f_k (mD-n) / Fs), x complex."""
    h = z.taps().astype(np.float64)
    L, D = h.size, z.decimation
    xp = np.concatenate([np.zeros(L - 1, np.complex128), x])   # input before the first call = 0
    out = np.zeros((len(ks), n_out), np.complex128)
    n = np.arange(L)
    for i, k in enumerate(ks):
        nu = (first_center_hz + z.spacing_hz * k) / z.wide_rate
        for m in range(n_out):
            s = m * D - n
            out[i, m] = np.sum(h * xp[(L - 1) + s] * np.exp(-2j * np.pi * nu * s))
    return out


def _channelizer(form, **kw):
    if form == "direct":
        os.environ["FMGPU_CHANNELIZER_DIRECT"] = "1"
    try:
        return fm.Channelizer(**kw)
    finally:
        os.environ.pop("FMGPU_CHANNELIZER_DIRECT", None)


def _run_calls(z, iq_dev, calls, n_out, row_bytes, ch_first=0, ch_count=None):
    """Ragged calls over [W][n_tot] pairs; returns the [W][ch_count][n_out] complex output."""
    import torch
    ch_count = z.n_channels - ch_first if ch_count is None else ch_count
    out = torch.zeros((z.n_captures, ch_count, n_out, 2), dtype=torch.float32, device=iq_dev.device)
    s0 = 0
    for n in calls:
        z.process(iq_dev.data_ptr() + z.pair_bytes * s0, n, out.data_ptr() + 8 * (s0 // z.decimation), n_out,
                  ch_first, ch_count, iq_stride_bytes=row_bytes)
        s0 += n
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("form", ["polyphase", "direct"])
@pytest.mark.parametrize("fmt", ["cs8", "cs16"])
def test_format_matches_definition_across_calls(fmt, form):
    import torch
    dev = torch.device("cuda", 0)
    offsets = [-9.9e6, -9.8e6, -9.85e6]                        # c0 = -49.5, -49, -49.25
    W, D, calls = len(offsets), 100, [1500, 100, 7300, 3200]   # ragged, two calls shorter than L - 1
    n_tot = sum(calls)
    n_out = n_tot // D
    z = _channelizer(form, first_center_hz=offsets, sample_format=fmt)
    assert z.sample_format == fmt and z.pair_bytes == (4 if fmt == "cs16" else 2)
    assert fm.load_library().fmgpu_channelizer_sample_format(z.h) == (CS16 if fmt == "cs16" else CS8)
    info = np.iinfo(DTYPE[fmt])
    rng = np.random.default_rng(40 + len(fmt))
    raw = rng.integers(info.min, info.max + 1, (W, n_tot, 2)).astype(DTYPE[fmt])
    out = _run_calls(z, torch.from_numpy(raw).to(dev), calls, n_out, raw[0].nbytes)
    got = out.cpu().numpy()
    got = got[..., 0] + 1j * got[..., 1]
    x = raw.astype(np.float64) / SCALE[fmt]
    x = x[..., 0] + 1j * x[..., 1]
    for w, ks in ((0, [0, 99]), (1, [37, 50]), (2, [13, 64])):
        err = np.abs(got[w, ks] - _model(z, offsets[w], x[w], ks, n_out)).max()
        assert err < 2e-5, (w, err)
    z.close()


@pytest.mark.parametrize("form", ["polyphase", "direct"])
def test_cs16_low_amplitude_keeps_its_low_bits(form):
    """|v| <= 64: the error relative to the input's scale, so a loader that drops low bits fails."""
    import torch
    dev = torch.device("cuda", 0)
    offsets = [-9.9e6, -9.85e6]
    W, D, calls = len(offsets), 100, [4800, 3200]
    n_tot = sum(calls)
    n_out = n_tot // D
    z = _channelizer(form, first_center_hz=offsets, sample_format="cs16")
    raw = np.random.default_rng(77).integers(-64, 65, (W, n_tot, 2)).astype(np.int16)
    out = _run_calls(z, torch.from_numpy(raw).to(dev), calls, n_out, raw[0].nbytes)
    got = out.cpu().numpy()
    got = got[..., 0] + 1j * got[..., 1]
    x = raw.astype(np.float64) / 32768.0
    x = x[..., 0] + 1j * x[..., 1]
    scale = np.abs(x).max()
    for w in range(W):
        ks = [5, 50, 94]
        ref = _model(z, offsets[w], x[w], ks, n_out)
        assert np.abs(ref).max() > 0.05 * scale
        err = np.abs(got[w, ks] - ref).max()
        assert err / scale < 2e-5, (w, err / scale)
    z.close()


@pytest.mark.parametrize("form", ["polyphase", "direct"])
def test_cs16_of_256s_is_cs8_of_s_bit_for_bit(form):
    """v = 256 s converts exactly to s / 128, so the two formats must give the same bits."""
    import torch
    dev = torch.device("cuda", 0)
    offsets = [-9.9e6, -9.85e6]
    calls = [1500, 3200, 7300, 100]
    n_tot = sum(calls)
    n_out = n_tot // 100
    s = np.random.default_rng(8).integers(-128, 128, (len(offsets), n_tot, 2)).astype(np.int8)
    s.reshape(-1)[:256] = np.arange(-128, 128)                 # every value at least once
    v = s.astype(np.int16) * 256
    z8 = _channelizer(form, first_center_hz=offsets, sample_format="cs8")
    z16 = _channelizer(form, first_center_hz=offsets, sample_format="cs16")
    y8 = _run_calls(z8, torch.from_numpy(s).to(dev), calls, n_out, s[0].nbytes)
    y16 = _run_calls(z16, torch.from_numpy(v).to(dev), calls, n_out, v[0].nbytes)
    assert torch.equal(y8, y16)
    assert y8.abs().max().item() > 0.1
    z8.close()
    z16.close()


def _band_to_engine(z, iq_dev, nblk, chunk, N=8192):
    """Channelizer -> fmgpu_process_batch_cf32 chunk by chunk, as tests/test_gpu_channelizer.py does."""
    import torch
    dev = iq_dev.device
    Cn = z.n_channels
    stride = nblk * N
    D = z.decimation
    x_dev = torch.zeros((Cn, stride, 2), dtype=torch.float32, device=dev)
    eng = fm.Engine(fm.make_config(iq_rate=240_000, decimation=1, max_blocks=chunk), Cn, 0)
    acap, gcap = eng.audio_capacity(chunk), chunk + 8
    audio = [[] for _ in range(Cn)]
    groups = [[] for _ in range(Cn)]
    stereo_last = None
    st_ = torch.cuda.current_stream().cuda_stream
    for b0 in range(0, nblk, chunk):
        z.process(iq_dev.data_ptr() + z.pair_bytes * b0 * N * D, chunk * N * D, x_dev.data_ptr() + 8 * b0 * N,
                  stride, stream=st_)
        a = torch.zeros((Cn, 2, acap), dtype=torch.float32, device=dev)
        na = torch.zeros(Cn, dtype=torch.int32, device=dev)
        g = torch.zeros((Cn, gcap, 16), dtype=torch.uint8, device=dev)
        ng = torch.zeros(Cn, dtype=torch.int32, device=dev)
        stt = torch.zeros((Cn, chunk, 20), dtype=torch.uint8, device=dev)
        eng.process_batch_cf32(x_dev.data_ptr() + 8 * b0 * N, stride, chunk, a.data_ptr(), acap,
                               na.data_ptr(), g.data_ptr(), gcap, ng.data_ptr(), stt.data_ptr(), st_)
        torch.cuda.synchronize()
        a, na, ng = a.cpu().numpy(), na.cpu().numpy(), ng.cpu().numpy()
        gv = g.cpu().numpy().view(fm.GROUP_DTYPE).reshape(Cn, gcap)
        stereo_last = stt.cpu().numpy().view(fm.STATUS_DTYPE).reshape(Cn, chunk)["stereo"][:, -1]
        for c in range(Cn):
            audio[c].append(a[c, :, :na[c]])
            gg = gv[c, :ng[c]].copy()
            gg["block_index"] += b0
            groups[c].append(gg)
    x_host = x_dev.cpu().numpy().view(np.complex64).reshape(Cn, stride)
    eng.close()
    audio = [np.concatenate(a, axis=1) for a in audio]
    groups = [np.concatenate(g) for g in groups]
    return audio, groups, stereo_last, x_host


def _clean_pis(g):
    return [int(x["a"]) for x in g if ((int(x["errors"]) >> 6) & 3) == 0]   # block A received clean


def test_weak_station_beside_strong_one_needs_cs16(orc_fm):
    """9.6 MS/s band, 40 carriers at 200 kHz (D = 40, P = 48): one FM-stereo+RDS station at -6 dBFS,
    a second 70 dB below it four slots away, 1 LSB of cs16 noise as dither. From cs16 both decode,
    equal to the oracle bit for bit; from the same band in uint8 the weak one is below the bytes'
    quantisation floor and yields no clean group."""
    import torch
    dev = torch.device("cuda", 0)
    wide, D, N, nblk, chunk, Cn, sp, c0 = 9_600_000, 40, 8192, 24, 4, 40, 200_000.0, -19.5
    n_wide = nblk * N * D
    strong, weak = 12, 16
    stations = {strong: (0x5112, "STRONG  ", 1000.0, 0.0, 0.5),
                weak: (0x3716, "WEAK -70", 600.0, 1500.0, 0.5 * 10 ** (-70 / 20))}
    x = np.zeros(n_wide, np.complex128)
    for k, (pi, ps, fl, fr, amp) in stations.items():
        s = orc.Signal(fs_iq=float(wide), deviation=60_000.0, tone_l_hz=fl, tone_l_amp=0.8,
                       tone_r_hz=fr, tone_r_amp=0.8 if fr else 0.0, iq_amp=amp,
                       freq_offset_hz=(c0 + k) * sp, seed=k,
                       rds_bits=orc.rds_encode_groups(orc.rds_groups_ps_rt(pi, ps)))
        x += generate_cf64(s, n_wide)
    rng = np.random.default_rng(7)
    x += (rng.standard_normal(n_wide) + 1j * rng.standard_normal(n_wide)) / 32768.0
    iq16 = np.empty((n_wide, 2), np.int16)
    iq16[:, 0] = np.clip(np.round(32768.0 * x.real), -32768, 32767)
    iq16[:, 1] = np.clip(np.round(32768.0 * x.imag), -32768, 32767)
    iq8 = np.empty((n_wide, 2), np.uint8)                      # the generator's uint8 rule
    iq8[:, 0] = np.clip(np.round(127.5 + 127.5 * x.real), 0, 255)
    iq8[:, 1] = np.clip(np.round(127.5 + 127.5 * x.imag), 0, 255)
    del x
    # 100 dB and 32 taps per phase: with 60 dB and 16 (the float64 model of this band) the strong
    # station leaks into the weak one's channel only about 17 dB below it
    zkw = dict(wide_rate=wide, decimation=D, n_channels=Cn, first_center_hz=c0 * sp, spacing_hz=sp,
               taps_per_phase=32, cutoff_hz=100_000.0, atten_db=100.0)

    z = fm.Channelizer(sample_format="cs16", **zkw)
    assert z.output_rate == 240_000
    audio, groups, stereo_last, x_host = _band_to_engine(z, torch.from_numpy(iq16).to(dev), nblk, chunk)
    z.close()
    for k, (pi, ps, fl, fr, amp) in stations.items():
        assert stereo_last[k] == 1, k
        pis = _clean_pis(groups[k])
        assert len(pis) >= 2 and all(p == pi for p in pis), (k, groups[k])
        rl, rr, rg, rst = _oracle_chain(orc_fm, x_host[k], nblk)
        assert np.array_equal(audio[k][0], rl) and np.array_equal(audio[k][1], rr), k
        assert groups_equal(groups[k], rg, keys=("a", "b", "c", "d", "errors", "block_index")), k
        assert rst[-1] == 1
    for k in (4, 24, 36):                                      # empty slots
        assert stereo_last[k] == 0 and _clean_pis(groups[k]) == [], k

    z = fm.Channelizer(sample_format="cu8", **zkw)
    audio, groups, stereo_last, _ = _band_to_engine(z, torch.from_numpy(iq8).to(dev), nblk, chunk)
    z.close()
    assert stereo_last[strong] == 1 and len(_clean_pis(groups[strong])) >= 2
    assert _clean_pis(groups[weak]) == [], groups[weak]


def test_format_arguments():
    import torch
    dev = torch.device("cuda", 0)
    L = fm.load_library()
    h = C.c_void_p()
    args = (1, 24_000_000, 100, 100)
    one = (C.c_double * 1)(-9.9e6)
    tail = (200e3, 16, 100e3, 60.0, C.byref(h))
    for bad in (-1, 3, 255):
        assert L.fmgpu_channelizer_create_format(0, bad, *args, one, *tail) == EINVAL
    assert not h.value
    with pytest.raises(ValueError):
        fm.Channelizer(sample_format="cs12")
    # create and create_multi objects are cu8
    assert L.fmgpu_channelizer_create_multi(0, *args, one, *tail) == 0
    assert L.fmgpu_channelizer_sample_format(h) == CU8
    L.fmgpu_channelizer_destroy(h)
    assert L.fmgpu_channelizer_create(0, 24_000_000, 100, 100, -9.9e6, *tail) == 0
    assert L.fmgpu_channelizer_sample_format(h) == CU8
    L.fmgpu_channelizer_destroy(h)
    assert L.fmgpu_channelizer_sample_format(None) == EINVAL

    n_in = 3200
    buf = torch.zeros(2 * (4 * n_in + 16), dtype=torch.uint8, device=dev)
    out = torch.zeros((2, 100, n_in // 100, 2), dtype=torch.float32, device=dev)
    p, o, n_out = buf.data_ptr(), out.data_ptr(), n_in // 100
    z = fm.Channelizer(first_center_hz=[-9.9e6, -9.8e6], sample_format="cs16")
    assert z.pair_bytes == 4
    assert L.fmgpu_channelizer_process_iq(z.h, p, 4 * n_in + 2, n_in, 0, 100, o, n_out, None) == EINVAL
    assert L.fmgpu_channelizer_process_iq(z.h, p, 4 * n_in - 4, n_in, 0, 100, o, n_out, None) == EINVAL
    assert L.fmgpu_channelizer_process_iq(z.h, p + 2, 4 * n_in, n_in, 0, 100, o, n_out, None) == EINVAL
    assert L.fmgpu_channelizer_process_multi(z.h, p, 4 * n_in, n_in, 0, 100, o, n_out, None) == EINVAL
    assert L.fmgpu_channelizer_process_iq(z.h, p, 4 * n_in + 4, n_in, 0, 100, o, n_out, None) == 0
    z.close()
    z = fm.Channelizer(sample_format="cs16")
    assert L.fmgpu_channelizer_process(z.h, p, n_in, 0, 100, o, n_out, None) == EINVAL
    z.close()
    z = fm.Channelizer(first_center_hz=[-9.9e6], sample_format="cs8")
    assert z.pair_bytes == 2
    assert L.fmgpu_channelizer_process(z.h, p, n_in, 0, 100, o, n_out, None) == EINVAL
    assert L.fmgpu_channelizer_process_multi(z.h, p, 2 * n_in, n_in, 0, 100, o, n_out, None) == EINVAL
    assert L.fmgpu_channelizer_process_iq(z.h, p + 1, 2 * n_in, n_in, 0, 100, o, n_out, None) == EINVAL
    assert L.fmgpu_channelizer_process_iq(z.h, p, 2 * n_in, n_in, 0, 100, o, n_out, None) == 0
    torch.cuda.synchronize()
    z.close()

    # process_iq on a cu8 object is process_multi, bit for bit
    offsets = [-9.9e6, -9.85e6]
    calls = [3200, 1500, 7300]
    n_tot = sum(calls)
    stride = 2 * n_tot + 64
    rng = np.random.default_rng(15)
    iq = torch.from_numpy(rng.integers(0, 256, (2, stride), dtype=np.uint8)).to(dev)
    za, zb = fm.Channelizer(first_center_hz=offsets), fm.Channelizer(first_center_hz=offsets)
    assert za.sample_format == "cu8" and za.pair_bytes == 2
    ya = torch.zeros((2, 100, n_tot // 100, 2), dtype=torch.float32, device=dev)
    yb = torch.zeros_like(ya)
    s0 = 0
    for n in calls:
        m0 = s0 // 100
        assert L.fmgpu_channelizer_process_iq(za.h, iq.data_ptr() + 2 * s0, stride, n, 0, 100,
                                              ya.data_ptr() + 8 * m0, n_tot // 100, None) == 0
        assert L.fmgpu_channelizer_process_multi(zb.h, iq.data_ptr() + 2 * s0, stride, n, 0, 100,
                                                 yb.data_ptr() + 8 * m0, n_tot // 100, None) == 0
        s0 += n
    torch.cuda.synchronize()
    assert torch.equal(ya, yb)
    za.close()
    zb.close()

"""Rational output rates of the channelizer (fmgpu_channelizer_create_rate / _process_stream): a
capture at wide_rate comes out at wide_rate * U / D, so 20 MS/s (HackRF) and 10 MS/s (SDRplay,
Airspy) captures reach the engine's 240 or 256 kS/s.

The outputs must follow the header's definition in both forms, with a count per call that varies and
is known before the call; splitting a capture into other calls must not change a bit; U = 1 objects
must be the integer-decimation objects; and a 20 MS/s cs8 band must decode through the engine exactly
as the oracle's reference classes decode the same channelizer output."""
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
SP = 200_000.0
# (wide_rate, output_rate, n_channels, capture offsets in Hz): U = 3, D = 250 and U = 16, D = 625
RATES = {"20M_240k": (20_000_000, 240_000, 100, [-9.9e6, -9.8e6, -9.85e6]),
         "10M_256k": (10_000_000, 256_000, 50, [-4.9e6, -4.8e6, -4.85e6])}
# ragged calls: not multiples of D, some shorter than Lin - 1, the second one completes no output
CALLS = [1, 1, 1500, 300, 4111, 777, 2600, 59]


def _model(z, first_center_hz, x, ks, n_out):
    """float64 evaluation of y_k[m] = sum_{(mD - n) = 0 mod U} h[n] x[(mD-n)/U] exp(-j 2 pi nu_k (mD-n)/U)."""
    h = z.taps().astype(np.float64)
    L, U, D = h.size, z.interpolation, z.decimation
    Lin = -(-L // U)
    xp = np.concatenate([np.zeros(Lin - 1, np.complex128), x])   # input before the first call = 0
    i = np.arange(Lin)
    nus = np.array([(first_center_hz + z.spacing_hz * k) / z.wide_rate for k in ks])
    out = np.zeros((len(ks), n_out), np.complex128)
    for m in range(n_out):
        q, s = (m * D) % U, (m * D) // U
        n = q + i * U
        ok = n < L
        idx = s - i[ok]
        v = h[n[ok]] * xp[(Lin - 1) + idx]
        out[:, m] = np.exp(-2j * np.pi * np.outer(nus, idx)) @ v
    return out


def _channelizer(form, **kw):
    if form == "direct":
        os.environ["FMGPU_CHANNELIZER_DIRECT"] = "1"
    try:
        return fm.Channelizer(**kw)
    finally:
        os.environ.pop("FMGPU_CHANNELIZER_DIRECT", None)


def _rate_channelizer(form, rate, fmt, **kw):
    wide, out_rate, Cn, offsets = RATES[rate]
    return _channelizer(form, wide_rate=wide, output_rate=out_rate, n_channels=Cn, first_center_hz=offsets,
                        spacing_hz=SP, sample_format=fmt, **kw)


def _stream(z, iq_dev, calls, row_bytes, ch_first=0, ch_count=None, fill=0.0):
    """process_stream over [W][n_tot] pairs in calls; every call's outputs appended to each row.
    Returns the [W][ch_count][ceil(n_tot U / D)] output and the per-call counts."""
    import torch
    ch_count = z.n_channels - ch_first if ch_count is None else ch_count
    n_tot = sum(calls)
    total = -(-n_tot * z.interpolation // z.decimation)
    out = torch.full((z.n_captures, ch_count, total + 16, 2), fill, dtype=torch.float32, device=iq_dev.device)
    s0, m0, counts = 0, 0, []
    for n in calls:
        want = z.outputs(n)
        got = z.process_stream(iq_dev.data_ptr() + z.pair_bytes * s0, n, out.data_ptr() + 8 * m0, total + 16,
                               ch_first, ch_count, iq_stride_bytes=row_bytes)
        assert got == want, (n, got, want)
        counts.append(got)
        s0 += n
        m0 += got
    torch.cuda.synchronize()
    assert m0 == total
    return out, counts


def _random_iq(fmt, shape, seed):
    rng = np.random.default_rng(seed)
    if fmt == "cu8":
        raw = rng.integers(0, 256, shape + (2,)).astype(np.uint8)
        x = (raw.astype(np.float64) - 127.5) / 127.5
    else:
        raw = rng.integers(-32768, 32768, shape + (2,)).astype(np.int16)
        x = raw.astype(np.float64) / 32768.0
    return raw, x[..., 0] + 1j * x[..., 1]


@pytest.mark.parametrize("form", ["polyphase", "direct"])
@pytest.mark.parametrize("fmt", ["cu8", "cs16"])
@pytest.mark.parametrize("rate", sorted(RATES))
def test_rational_rate_matches_definition_across_calls(rate, fmt, form):
    import torch
    dev = torch.device("cuda", 0)
    wide, out_rate, Cn, offsets = RATES[rate]
    z = _rate_channelizer(form, rate, fmt)
    U, D = z.interpolation, z.decimation
    assert U > 1 and np.gcd(U, D) == 1 and wide * U == out_rate * D
    assert z.output_rate == out_rate
    assert z.taps().size == D * 16
    W, n_tot = len(offsets), sum(CALLS)
    raw, x = _random_iq(fmt, (W, n_tot), 60 + U)
    iq = torch.from_numpy(raw).to(dev)
    out, counts = _stream(z, iq, CALLS, raw[0].nbytes)
    assert 0 in counts
    n_out = out.shape[2] - 16
    got = out.cpu().numpy()[:, :, :n_out]
    got = got[..., 0] + 1j * got[..., 1]
    for w, ks in ((0, [0, Cn - 1]), (1, [Cn // 3, Cn // 2]), (2, [13, Cn - 7])):
        err = np.abs(got[w, ks] - _model(z, offsets[w], x[w], ks, n_out)).max()
        assert err < 2e-5, (w, err)
    z.close()
    # a ch_first / ch_count share of the bank gives the same rows, bit for bit
    zs = _rate_channelizer(form, rate, fmt)
    part, _ = _stream(zs, iq, CALLS, raw[0].nbytes, ch_first=11, ch_count=20)
    assert torch.equal(part[:, :, :n_out], out[:, 11:31, :n_out])
    zs.close()


@pytest.mark.parametrize("form", ["polyphase", "direct"])
@pytest.mark.parametrize("rate", ["24M_240k"] + sorted(RATES))
def test_counts_sentinel_and_stream_invariance(rate, form):
    """outputs() is what process_stream writes; nothing past it is touched; one call and ragged
    calls over the same capture give the same bits (U = 1 through create_rate as well)."""
    import torch
    dev = torch.device("cuda", 0)
    if rate == "24M_240k":
        kw = dict(wide_rate=24_000_000, output_rate=240_000, n_channels=100, first_center_hz=[-9.9e6, -9.85e6],
                  spacing_hz=SP, sample_format="cs8")
    else:
        wide, out_rate, Cn, offsets = RATES[rate]
        kw = dict(wide_rate=wide, output_rate=out_rate, n_channels=Cn, first_center_hz=offsets[:2],
                  spacing_hz=SP, sample_format="cs8")
    calls = [37, 1, 2222, 501, 5003, 250, 1]
    n_tot = sum(calls)
    raw = np.random.default_rng(5).integers(-128, 128, (2, n_tot, 2)).astype(np.int8)
    iq = torch.from_numpy(raw).to(dev)
    sentinel = 1234.5
    za, zb = _channelizer(form, **kw), _channelizer(form, **kw)
    ya, ca = _stream(za, iq, [n_tot], raw[0].nbytes, fill=sentinel)
    yb, cb = _stream(zb, iq, calls, raw[0].nbytes, fill=sentinel)
    U, D = za.interpolation, za.decimation
    total = -(-n_tot * U // D)
    assert ca == [total] and sum(cb) == total
    T = 0
    for n, c in zip(calls, cb):
        assert c == -(-(T + n) * U // D) - -(-T * U // D)
        T += n
    assert torch.equal(ya, yb)
    assert bool((ya[:, :, total:] == sentinel).all())
    assert not bool((ya[:, :, :total] == sentinel).any())
    # counts are host state: asking does not advance the stream
    assert za.outputs(D) == za.outputs(D) == -(-(n_tot + D) * U // D) - total
    za.close()
    zb.close()


def test_unit_ratio_is_the_integer_decimation_object():
    import torch
    dev = torch.device("cuda", 0)
    L = fm.load_library()
    offsets = [-9.9e6, -9.8e6]
    kw = dict(wide_rate=24_000_000, n_channels=100, first_center_hz=offsets, spacing_hz=SP, sample_format="cs16")
    zr = fm.Channelizer(output_rate=240_000, **kw)
    zf = fm.Channelizer(decimation=100, **kw)
    zs = fm.Channelizer(output_rate=240_000, **kw)
    assert (zr.interpolation, zr.decimation, zr.output_rate) == (1, 100, 240_000)
    assert np.array_equal(zr.taps(), zf.taps())
    calls = [3200, 1500, 7300]
    n_tot = sum(calls)
    raw = np.random.default_rng(9).integers(-32768, 32768, (2, n_tot, 2)).astype(np.int16)
    iq = torch.from_numpy(raw).to(dev)
    n_out = n_tot // 100
    ys = [torch.zeros((2, 100, n_out, 2), dtype=torch.float32, device=dev) for _ in range(3)]
    s0 = 0
    for n in calls:
        m0 = s0 // 100
        for z, y in ((zr, ys[0]), (zf, ys[1])):
            assert L.fmgpu_channelizer_process_iq(z.h, iq.data_ptr() + 4 * s0, raw[0].nbytes, n, 0, 100,
                                                  y.data_ptr() + 8 * m0, n_out, None) == 0
        assert zs.process_stream(iq.data_ptr() + 4 * s0, n, ys[2].data_ptr() + 8 * m0, n_out,
                                 iq_stride_bytes=raw[0].nbytes) == n // 100
        s0 += n
    torch.cuda.synchronize()
    assert torch.equal(ys[0], ys[1]) and torch.equal(ys[2], ys[1])
    assert ys[0].abs().max().item() > 0.01
    for z in (zr, zf, zs):
        z.close()
    # the integer-rate calls refuse U > 1 objects
    z = fm.Channelizer(wide_rate=20_000_000, output_rate=240_000, first_center_hz=[-9.9e6])
    assert z.interpolation == 3
    buf = torch.zeros(2 * 2500, dtype=torch.uint8, device=dev)
    out = torch.zeros((100, 64, 2), dtype=torch.float32, device=dev)
    assert L.fmgpu_channelizer_process_iq(z.h, buf.data_ptr(), 5000, 2500, 0, 100, out.data_ptr(), 64, None) == EINVAL
    assert L.fmgpu_channelizer_process_multi(z.h, buf.data_ptr(), 5000, 2500, 0, 100, out.data_ptr(), 64,
                                             None) == EINVAL
    assert L.fmgpu_channelizer_process(z.h, buf.data_ptr(), 2500, 0, 100, out.data_ptr(), 64, None) == EINVAL
    z.close()


def test_rational_pass_band_and_stop_band_cs16():
    """20 MS/s -> 240 kS/s, cs16: a tone 30 kHz into carrier 5 comes out at unity gain and 30 kHz;
    every carrier but 4..6 stays below the bound the float64 model itself gives (at least 50 dB)."""
    import torch
    dev = torch.device("cuda", 0)
    z = fm.Channelizer(wide_rate=20_000_000, output_rate=240_000, first_center_hz=-9.9e6, spacing_hz=SP,
                       sample_format="cs16")
    n = 250 * 400
    t = np.arange(n)
    f5 = -9.9e6 + 5 * SP + 30_000.0
    xt = 0.7 * np.exp(2j * np.pi * f5 * t / 20e6)
    raw = np.empty((n, 2), np.int16)
    raw[:, 0] = np.clip(np.round(32768 * xt.real), -32768, 32767)
    raw[:, 1] = np.clip(np.round(32768 * xt.imag), -32768, 32767)
    x = (raw[:, 0] + 1j * raw[:, 1]) / 32768.0
    out, _ = _stream(z, torch.from_numpy(raw).to(dev), [n], raw.nbytes)
    n_out = out.shape[2] - 16
    y = out.cpu().numpy()[0, :, :n_out]
    y = y[..., 0] + 1j * y[..., 1]
    p = (np.abs(y[:, 64:]) ** 2).mean(axis=1)                  # past the filter's start-up
    assert abs(np.sqrt(p[5]) - 0.7) < 0.01
    ph = np.unwrap(np.angle(y[5, 64:]))
    assert abs((ph[-1] - ph[0]) / (2 * np.pi * (len(ph) - 1)) * 240_000 - 30_000.0) < 50.0
    others = [k for k in range(100) if k not in (4, 5, 6)]
    ym = _model(z, -9.9e6, x, [5] + others, n_out)[:, 64::8]
    pm = (np.abs(ym) ** 2).mean(axis=1)
    bound_db = 10 * np.log10(pm[1:].max() / pm[0])
    assert bound_db < -50.0, bound_db
    got_db = 10 * np.log10((np.abs(y[others, 64::8]) ** 2).mean(axis=1).max() / p[5])
    assert got_db < bound_db + 1.0, (got_db, bound_db)
    z.close()


def test_hackrf_band_to_audio_and_rds(orc_fm):
    """A 20 MS/s cs8 band (a HackRF capture) with three FM-stereo+RDS stations among 100 slots,
    12 blocks at 240 kS/s: 8,192,000 pairs, fed in ragged chunks that are not multiples of 250;
    the engine takes whole 4-block chunks of the accumulated rows."""
    import torch
    dev = torch.device("cuda", 0)
    wide, N, nblk, chunk, Cn, c0 = 20_000_000, 8192, 12, 4, 100, -49.5
    n_wide = nblk * N * 250 // 3
    assert n_wide == 8_192_000
    stations = {7: (0x2207, "CH07 FM ", 600.0, 1500.0), 50: (0x1234, "B200TEST", 1000.0, 0.0),
                93: (0x4493, "NINETY3 ", 440.0, 880.0)}
    x = np.zeros(n_wide, np.complex128)
    for k, (pi, ps, fl, fr) in stations.items():
        s = orc.Signal(fs_iq=float(wide), deviation=60_000.0, tone_l_hz=fl, tone_l_amp=0.8,
                       tone_r_hz=fr, tone_r_amp=0.8 if fr else 0.0, iq_amp=0.28,
                       freq_offset_hz=(c0 + k) * SP, seed=k,
                       rds_bits=orc.rds_encode_groups(orc.rds_groups_ps_rt(pi, ps)))
        x += generate_cf64(s, n_wide)
    iq = np.empty((n_wide, 2), np.int8)
    iq[:, 0] = np.clip(np.round(128.0 * x.real), -128, 127)
    iq[:, 1] = np.clip(np.round(128.0 * x.imag), -128, 127)
    del x
    iq_dev = torch.from_numpy(iq).to(dev)
    z = fm.Channelizer(wide_rate=wide, output_rate=240_000, n_channels=Cn, first_center_hz=c0 * SP, spacing_hz=SP,
                       sample_format="cs8")
    assert (z.interpolation, z.decimation) == (3, 250)
    stride = nblk * N
    x_dev = torch.zeros((Cn, stride, 2), dtype=torch.float32, device=dev)
    eng = fm.Engine(fm.make_config(iq_rate=240_000, decimation=1, max_blocks=chunk), Cn, 0)
    acap, gcap = eng.audio_capacity(chunk), chunk + 8
    audio = [[] for _ in range(Cn)]
    groups = [[] for _ in range(Cn)]
    stereo_last = None
    st_ = torch.cuda.current_stream().cuda_stream
    sizes = [1_000_003, 777_777, 1_234_567, 333_331, 2_010_101]
    s0, have, b0, i = 0, 0, 0, 0
    while s0 < n_wide:
        n = min(sizes[i % len(sizes)], n_wide - s0)
        i += 1
        assert n % 250 != 0
        have += z.process_stream(iq_dev.data_ptr() + 2 * s0, n, x_dev.data_ptr() + 8 * have, stride,
                                 stream=st_, iq_stride_bytes=2 * n)
        s0 += n
        while have >= (b0 + chunk) * N:
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
            b0 += chunk
    assert i > len(sizes) and have == stride and b0 == nblk
    x_host = x_dev.cpu().numpy().view(np.complex64).reshape(Cn, stride)
    eng.close()
    z.close()
    audio = [np.concatenate(a, axis=1) for a in audio]
    groups = [np.concatenate(g) for g in groups]

    def clean_pis(g):
        return [int(v["a"]) for v in g if ((int(v["errors"]) >> 6) & 3) == 0]   # block A received clean

    for k, (pi, ps, fl, fr) in stations.items():
        assert stereo_last[k] == 1, k
        pis = clean_pis(groups[k])
        assert len(pis) >= 2 and all(p == pi for p in pis), (k, groups[k])
        rl, rr, rg, rst = _oracle_chain(orc_fm, x_host[k], nblk)
        assert np.array_equal(audio[k][0], rl) and np.array_equal(audio[k][1], rr), k
        assert groups_equal(groups[k], rg, keys=("a", "b", "c", "d", "errors", "block_index")), k
        assert rst[-1] == 1
    for k in (20, 60):                                         # empty slots
        assert stereo_last[k] == 0 and clean_pis(groups[k]) == [], k


def test_rate_arguments():
    import torch
    dev = torch.device("cuda", 0)
    L = fm.load_library()
    h = C.c_void_p()
    one = (C.c_double * 1)(0.0)

    def create(wide, out_rate, cutoff=10.0):
        return L.fmgpu_channelizer_create_rate(0, 0, 1, wide, out_rate, 1, one, 1.0, 1, cutoff, 60.0, C.byref(h))

    assert create(65, 64) == 0                                 # U = 64, D = 65: the largest U
    assert (L.fmgpu_channelizer_interpolation(h), L.fmgpu_channelizer_decimation(h)) == (64, 65)
    assert L.fmgpu_channelizer_output_rate(h) == 64
    L.fmgpu_channelizer_destroy(h)
    h.value = None
    assert create(66, 65) == EINVAL                            # U = 65
    assert create(20_000_000, 240_001, 100e3) == EINVAL        # U = 240001
    assert create(240_000, 240_001, 100e3) == EINVAL           # output_rate > wide_rate
    assert create(240_000, 0, 100e3) == EINVAL
    assert create(240_000, -240_000, 100e3) == EINVAL
    assert not h.value
    assert create(240_000, 240_000, 100e3) == 0                # U = D = 1
    assert L.fmgpu_channelizer_decimation(h) == 1 and L.fmgpu_channelizer_output_rate(h) == 240_000
    L.fmgpu_channelizer_destroy(h)
    assert L.fmgpu_channelizer_outputs(None, 10) == 0
    assert L.fmgpu_channelizer_interpolation(None) == 0 and L.fmgpu_channelizer_decimation(None) == 0

    z = fm.Channelizer(wide_rate=20_000_000, output_rate=240_000, first_center_hz=[-9.9e6, -9.8e6],
                       sample_format="cs16")
    n_in = 2501
    buf = torch.zeros(2 * (4 * n_in + 16), dtype=torch.uint8, device=dev)
    out = torch.zeros((2, 100, 64, 2), dtype=torch.float32, device=dev)
    p, o = buf.data_ptr(), out.data_ptr()
    k = z.outputs(n_in)
    assert k == 31
    nout = C.c_size_t(77)
    ps = L.fmgpu_channelizer_process_stream
    assert ps(z.h, p, 4 * n_in, n_in, 0, 100, o, k - 1, C.byref(nout), None) == EINVAL
    assert ps(z.h, p, 4 * n_in + 2, n_in, 0, 100, o, k, C.byref(nout), None) == EINVAL
    assert ps(z.h, p, 4 * n_in - 4, n_in, 0, 100, o, k, C.byref(nout), None) == EINVAL
    assert ps(z.h, p + 2, 4 * n_in, n_in, 0, 100, o, k, C.byref(nout), None) == EINVAL
    assert ps(z.h, p, 4 * n_in, 0, 0, 100, o, k, C.byref(nout), None) == EINVAL
    assert ps(z.h, p, 4 * n_in, n_in, 90, 11, o, k, C.byref(nout), None) == EINVAL
    assert nout.value == 77 and z.outputs(n_in) == k           # refused calls leave the stream as it was
    assert ps(z.h, p, 4 * n_in, n_in, 0, 100, o, k, C.byref(nout), None) == 0
    assert nout.value == k
    assert ps(z.h, p, 4 * n_in, n_in, 0, 100, o, 64, None, None) == 0      # n_out may be NULL
    torch.cuda.synchronize()
    z.close()


def test_rational_polyphase_and_direct_forms_agree_and_polyphase_is_faster():
    """20 MS/s -> 240 kS/s, 100 carriers, two 8192-sample blocks per call."""
    import torch
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(21)
    n_in = 2 * 8192 * 250 // 3 + 1
    iq = torch.from_numpy(rng.integers(0, 256, 2 * n_in, dtype=np.uint8)).to(dev)
    res, ms = {}, {}
    for form in ("polyphase", "direct"):
        z = _channelizer(form, wide_rate=20_000_000, output_rate=240_000, first_center_hz=-9.9e6)
        out = torch.zeros((100, 2 * 8192 + 1, 2), dtype=torch.float32, device=dev)
        n_out = [z.process_stream(iq.data_ptr(), n_in, out.data_ptr(), out.shape[1]) for _ in range(2)]
        torch.cuda.synchronize()
        res[form] = (n_out, out.cpu().numpy())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            z.process_stream(iq.data_ptr(), n_in, out.data_ptr(), out.shape[1])
        e1.record()
        torch.cuda.synchronize()
        ms[form] = e0.elapsed_time(e1) / 5
        z.close()
    assert res["polyphase"][0] == res["direct"][0]
    err = np.abs(res["polyphase"][1] - res["direct"][1]).max()
    assert err < 2e-5, err
    print(f"channelizer 20 MS/s -> 240 kS/s, 100 channels: polyphase {ms['polyphase']:.3f} ms, "
          f"direct {ms['direct']:.3f} ms")
    assert ms["polyphase"] < 0.5 * ms["direct"], ms

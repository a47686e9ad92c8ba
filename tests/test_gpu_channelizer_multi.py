"""Many captures in one channelizer (fmgpu_channelizer_create_multi / _process_multi).

Each capture of a multi-capture object must give exactly what a single-capture object with that
capture's centre offset gives (polyphase form), the header's definition per capture (direct form),
and, for RTL-class captures with FM-stereo+RDS stations, the oracle's audio and groups bit for bit
through one engine of n_captures * n_channels channels."""
import ctypes as C
import types

import numpy as np
import pytest

import fmtuner_sdr_b200 as fm
from oracle import orc
from tests.common import groups_equal
from tests.test_gpu_channelizer import _model, _oracle_chain

pytestmark = pytest.mark.gpu
EINVAL = -1


def _capture_view(z, w):
    """What _model reads of a channelizer, with capture w's offset."""
    return types.SimpleNamespace(taps=z.taps, decimation=z.decimation, wide_rate=z.wide_rate,
                                 spacing_hz=z.spacing_hz, first_center_hz=z.first_center_hz[w])


def test_batched_equals_separate_bit_for_bit():
    import torch
    dev = torch.device("cuda", 0)
    offsets = [-9.9e6, -9.8e6, -9.85e6, -9.9e6, -9.85e6]     # c0 = -49.5 (T 2), -49 (T 1), -49.25 (T 4)
    W, D, Cn = len(offsets), 100, 100
    calls = [3200, 7300, 1500]                                 # ragged, multiples of D
    n_tot = sum(calls)
    n_out = n_tot // D
    stride = 2 * n_tot + 64                                    # rows longer than one call's input
    rng = np.random.default_rng(21)
    iq = torch.from_numpy(rng.integers(0, 256, (W, stride), dtype=np.uint8)).to(dev)
    for ch_first, ch_count in ((0, Cn), (36, 13)):
        zm = fm.Channelizer(first_center_hz=offsets)
        assert zm.n_captures == W
        zs = [fm.Channelizer(first_center_hz=f) for f in offsets]
        assert all(z.n_captures == 1 for z in zs)
        out_m = torch.zeros((W, ch_count, n_out, 2), dtype=torch.float32, device=dev)
        out_s = torch.zeros((W, ch_count, n_out, 2), dtype=torch.float32, device=dev)
        s0 = 0
        for n in calls:
            m0 = s0 // D
            zm.process(iq.data_ptr() + 2 * s0, n, out_m.data_ptr() + 8 * m0, n_out, ch_first, ch_count,
                       iq_stride_bytes=stride)
            for w, z in enumerate(zs):
                z.process(iq[w].data_ptr() + 2 * s0, n, out_s[w].data_ptr() + 8 * m0, n_out, ch_first,
                          ch_count)
            s0 += n
        torch.cuda.synchronize()
        for w in range(W):
            assert torch.equal(out_m[w], out_s[w]), (w, ch_first, ch_count)
        if ch_first == 0:
            full = out_m
        else:
            assert torch.equal(out_m, full[:, ch_first:ch_first + ch_count])
        zm.close()
        for z in zs:
            z.close()


def test_direct_form_matches_definition_per_capture():
    import torch
    dev = torch.device("cuda", 0)
    # c0 = -49.123 has no T <= 8 with c0 * T an integer: every capture takes the direct form
    offsets = [-9.9e6, -49.123 * 200e3, -9.85e6]
    z = fm.Channelizer(first_center_hz=offsets)
    W, n1, n2 = len(offsets), 3200, 4800
    n_out = (n1 + n2) // 100
    rng = np.random.default_rng(33)
    iq = rng.integers(0, 256, (W, 2 * (n1 + n2)), dtype=np.uint8)
    iq_dev = torch.from_numpy(iq).to(dev)
    out = torch.zeros((W, 100, n_out, 2), dtype=torch.float32, device=dev)
    z.process(iq_dev.data_ptr(), n1, out.data_ptr(), n_out, iq_stride_bytes=2 * (n1 + n2))
    z.process(iq_dev.data_ptr() + 2 * n1, n2, out.data_ptr() + 8 * (n1 // 100), n_out,
              iq_stride_bytes=2 * (n1 + n2))
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    got = got[..., 0] + 1j * got[..., 1]
    for w, ks in ((0, [0, 99]), (1, [0, 37, 50, 99]), (2, [13, 64])):
        ref = _model(_capture_view(z, w), iq[w], ks, n_out)
        err = np.abs(got[w, ks] - ref).max()
        assert err < 2e-5, (w, err)
    z.close()


def test_dongle_captures_to_audio_and_rds(orc_fm):
    """Three 2.4 MS/s captures, each tuned elsewhere (its carrier grid at its own offset from its
    centre), two FM-stereo+RDS stations in each -> one channelizer -> one engine of 3 x 12 channels."""
    import torch
    dev = torch.device("cuda", 0)
    # 24 blocks (0.8 s): long enough for every station to decode several groups with block A clean
    wide, D, N, nblk, chunk, Cn, sp = 2_400_000, 10, 8192, 24, 4, 12, 200_000.0
    c0s = [-5.5, -5.25, -5.75]
    W = len(c0s)
    n_wide = nblk * N * D
    z = fm.Channelizer(wide_rate=wide, decimation=D, n_channels=Cn,
                       first_center_hz=[c * sp for c in c0s], spacing_hz=sp, taps_per_phase=16)
    assert z.output_rate == 240_000 and z.n_captures == W
    # (capture, carrier): PI, PS, left tone, right tone; every station within +-0.9 MHz of its centre
    stations = {(0, 2): (0x2202, "CAP0 K2 ", 600.0, 1500.0), (0, 8): (0x2208, "CAP0 K8 ", 1000.0, 0.0),
                (1, 1): (0x3301, "CAP1 K1 ", 440.0, 880.0), (1, 9): (0x3309, "CAP1 K9 ", 700.0, 0.0),
                (2, 4): (0x4404, "CAP2 K4 ", 900.0, 300.0), (2, 10): (0x440A, "CAP2 K10", 1200.0, 0.0)}
    iq = np.empty((W, 2 * n_wide), np.uint8)
    for w in range(W):
        acc_i = np.zeros(n_wide, np.float32)
        acc_q = np.zeros(n_wide, np.float32)
        for (cw, k), (pi, ps, fl, fr) in stations.items():
            if cw != w:
                continue
            f = (c0s[w] + k) * sp
            assert abs(f) <= 900_000.0
            s = orc.Signal(fs_iq=float(wide), deviation=60_000.0, tone_l_hz=fl, tone_l_amp=0.8,
                           tone_r_hz=fr, tone_r_amp=0.8 if fr else 0.0, iq_amp=0.28,
                           freq_offset_hz=f, seed=16 * w + k,
                           rds_bits=orc.rds_encode_groups(orc.rds_groups_ps_rt(pi, ps)))
            u = s.generate(n_wide)
            acc_i += (u[0::2].astype(np.float32) - 127.5) / 127.5
            acc_q += (u[1::2].astype(np.float32) - 127.5) / 127.5
        iq[w, 0::2] = np.clip(np.round(127.5 + 127.5 * acc_i), 0, 255)
        iq[w, 1::2] = np.clip(np.round(127.5 + 127.5 * acc_q), 0, 255)

    nch = W * Cn
    iq_dev = torch.from_numpy(iq).to(dev)
    stride = nblk * N
    x_dev = torch.zeros((nch, stride, 2), dtype=torch.float32, device=dev)
    eng = fm.Engine(fm.make_config(iq_rate=240_000, decimation=1, max_blocks=chunk), nch, 0)
    acap, gcap = eng.audio_capacity(chunk), chunk + 8
    audio = [[] for _ in range(nch)]
    groups = [[] for _ in range(nch)]
    stereo_last = None
    st_ = torch.cuda.current_stream().cuda_stream
    for b0 in range(0, nblk, chunk):
        z.process(iq_dev.data_ptr() + 2 * b0 * N * D, chunk * N * D, x_dev.data_ptr() + 8 * b0 * N,
                  stride, stream=st_, iq_stride_bytes=2 * n_wide)
        a = torch.zeros((nch, 2, acap), dtype=torch.float32, device=dev)
        na = torch.zeros(nch, dtype=torch.int32, device=dev)
        g = torch.zeros((nch, gcap, 16), dtype=torch.uint8, device=dev)
        ng = torch.zeros(nch, dtype=torch.int32, device=dev)
        stt = torch.zeros((nch, chunk, 20), dtype=torch.uint8, device=dev)
        eng.process_batch_cf32(x_dev.data_ptr() + 8 * b0 * N, stride, chunk, a.data_ptr(), acap,
                               na.data_ptr(), g.data_ptr(), gcap, ng.data_ptr(), stt.data_ptr(), st_)
        torch.cuda.synchronize()
        a, na, ng = a.cpu().numpy(), na.cpu().numpy(), ng.cpu().numpy()
        gv = g.cpu().numpy().view(fm.GROUP_DTYPE).reshape(nch, gcap)
        stereo_last = stt.cpu().numpy().view(fm.STATUS_DTYPE).reshape(nch, chunk)["stereo"][:, -1]
        for c in range(nch):
            audio[c].append(a[c, :, :na[c]])
            gg = gv[c, :ng[c]].copy()
            gg["block_index"] += b0
            groups[c].append(gg)
    x_host = x_dev.cpu().numpy().view(np.complex64).reshape(nch, stride)
    eng.close()
    z.close()

    for (w, k), (pi, ps, fl, fr) in stations.items():
        row = w * Cn + k
        a = np.concatenate(audio[row], axis=1)
        g = np.concatenate(groups[row])
        assert stereo_last[row] == 1, (w, k)
        pis = [int(x["a"]) for x in g if ((int(x["errors"]) >> 6) & 3) == 0]   # block A received clean
        assert len(pis) >= 2 and all(x == pi for x in pis), (w, k, g)
        rl, rr, rg, rst = _oracle_chain(orc_fm, x_host[row], nblk)
        assert np.array_equal(a[0], rl) and np.array_equal(a[1], rr), (w, k)
        assert groups_equal(g, rg, keys=("a", "b", "c", "d", "errors", "block_index")), (w, k)
        assert rst[-1] == 1
    # empty slots stay mono and silent of RDS
    for w, k in ((0, 5), (1, 4), (2, 0)):
        row = w * Cn + k
        assert stereo_last[row] == 0 and sum(len(x) for x in groups[row]) == 0, (w, k)


def test_multi_capture_arguments():
    import torch
    dev = torch.device("cuda", 0)
    L = fm.load_library()
    h = C.c_void_p()
    args = (24_000_000, 100, 100)
    tail = (200e3, 16, 100e3, 60.0, C.byref(h))
    two = (C.c_double * 2)(-9.9e6, -9.8e6)
    assert L.fmgpu_channelizer_create_multi(0, 2, *args, None, *tail) == EINVAL
    assert L.fmgpu_channelizer_create_multi(0, 0, *args, two, *tail) == EINVAL
    assert L.fmgpu_channelizer_create_multi(0, -3, *args, two, *tail) == EINVAL
    many = (C.c_double * 65536)(*([-9.9e6] * 65536))
    assert L.fmgpu_channelizer_create_multi(0, 65536, *args, many, *tail) == EINVAL
    assert not h.value

    z = fm.Channelizer(first_center_hz=[-9.9e6, -9.8e6])
    n_in = 3200
    iq = torch.full((2, 2 * n_in + 2), 128, dtype=torch.uint8, device=dev)
    out = torch.zeros((2, 100, n_in // 100, 2), dtype=torch.float32, device=dev)
    p, o = iq.data_ptr(), out.data_ptr()
    assert L.fmgpu_channelizer_process_multi(z.h, p, 2 * n_in + 1, n_in, 0, 100, o, n_in // 100, None) == EINVAL
    assert L.fmgpu_channelizer_process_multi(z.h, p, 2 * n_in - 2, n_in, 0, 100, o, n_in // 100, None) == EINVAL
    assert L.fmgpu_channelizer_process(z.h, p, n_in, 0, 100, o, n_in // 100, None) == EINVAL
    assert L.fmgpu_channelizer_process_multi(z.h, p, 2 * n_in + 2, n_in, 0, 100, o, n_in // 100, None) == 0
    torch.cuda.synchronize()
    z.close()

    # one capture through create_multi is fmgpu_channelizer_create
    rng = np.random.default_rng(5)
    x = torch.from_numpy(rng.integers(0, 256, 2 * n_in, dtype=np.uint8)).to(dev)
    z1 = fm.Channelizer(first_center_hz=-9.85e6)
    zm = fm.Channelizer(first_center_hz=[-9.85e6])
    assert z1.n_captures == 1 and zm.n_captures == 1
    assert np.array_equal(z1.taps(), zm.taps())
    y1 = torch.zeros((100, n_in // 100, 2), dtype=torch.float32, device=dev)
    ym = torch.zeros_like(y1)
    for _ in range(2):
        z1.process(x.data_ptr(), n_in, y1.data_ptr(), n_in // 100)
        zm.process(x.data_ptr(), n_in, ym.data_ptr(), n_in // 100)
    torch.cuda.synchronize()
    assert torch.equal(y1, ym)
    z1.close()
    zm.close()

"""Stage-level C-ABI entry points, one per reference method, against the oracle's classes:
ragged and tiny block sizes, empty / null arguments, capacity limits, setters and resets."""
import ctypes as C

import numpy as np
import pytest

import fmtuner_sdr_b200 as fm
from oracle import orc
from tests.common import groups_equal

pytestmark = pytest.mark.gpu
F = C.POINTER(C.c_float)
U8 = C.POINTER(C.c_uint8)


def _f(a):
    return a.ctypes.data_as(F)


RAGGED = [1, 7, 64, 65, 1000, 8192, 3, 4097, 12288, 255, 8192]


@pytest.fixture(scope="module")
def iq8():
    return orc.config1_signal(fs_iq=2_048_000).generate(sum(RAGGED) * 8 + 64)


@pytest.mark.parametrize("factor,tpp,atten", [(8, 28, 80.0), (4, 20, 80.0), (10, 28, 80.0), (2, 12, 70.0),
                                              (3, 16, 60.0)])
def test_complex_decimator_ragged_calls(orc_fm, factor, tpp, atten):
    L = orc_fm.lib
    rng = np.random.default_rng(factor)
    iq = rng.integers(0, 256, 2 * (sum(RAGGED) * factor + 50), dtype=np.uint8)
    d = L.orc_decim_create(factor, tpp, atten)
    eng = fm.Engine(fm.make_config(iq_rate=256000 * factor, decimation=factor, block_samples=16384,
                                   max_blocks=1, decim_taps_per_phase=tpp, decim_atten_db=int(atten)), 1, 0)
    pos = 0
    for n_out in RAGGED:
        n_in = n_out * factor + (3 if n_out % 2 else 0)      # trailing partial group is ignored
        chunk = iq[2 * pos:2 * (pos + n_in)]
        ref = np.zeros(2 * n_out, np.float32)
        k = L.orc_decim_execute_complex(d, chunk.ctypes.data_as(U8), n_in, _f(ref), n_out)
        got = eng.executeComplex(chunk, n_out)
        assert k == n_out and got.size == n_out
        assert np.array_equal(got.view(np.float32), ref)
        pos += n_out * factor                                  # only whole groups were consumed
    # capacity smaller than the input: stop at capacity (liquid_primitives.cpp:484)
    chunk = iq[:2 * 100 * factor]
    assert eng.executeComplex(chunk, 10).size == 10
    # reset restores the zero-initialised window
    L.orc_decim_reset(d)
    eng.reset(fm.engine.RESET_DECIM)
    ref = np.zeros(2 * 300, np.float32)
    L.orc_decim_execute_complex(d, chunk.ctypes.data_as(U8), 100 * factor, _f(ref), 100)
    assert np.array_equal(eng.executeComplex(chunk, 100).view(np.float32), ref[:200])
    L.orc_decim_destroy(d)
    eng.close()


@pytest.mark.parametrize("agc", [0, 1, 2])
def test_fmdemod_split_paths(orc_fm, iq8, agc):
    L = orc_fm.lib
    fs = 256000
    d = L.orc_demod_create(fs, 32000)
    dc = L.orc_demod_create(fs, 32000)
    dec = L.orc_decim_create(8, 28, 80.0)
    eng_u8 = fm.Engine(fm.make_config(iq_rate=fs, decimation=1, block_samples=16384, max_blocks=1,
                                      bandwidth_hz=309000, deemphasis=1), 1, 0)
    eng_cf = fm.Engine(fm.make_config(iq_rate=fs, decimation=1, block_samples=16384, max_blocks=1,
                                      bandwidth_hz=309000, deemphasis=1), 1, 0)
    for h, e in ((d, eng_u8), (dc, eng_cf)):
        L.orc_demod_set_agc(h, agc)
        e.set_agc_mode(agc)
    pos = 0
    for i, n in enumerate(RAGGED):
        if i == 4:   # XDR 'W' + de-emphasis change in mid-stream
            for h, e in ((d, eng_u8), (dc, eng_cf)):
                L.orc_demod_set_bandwidth_hz(h, 133000)
                e.set_bandwidth_hz(133000)
                L.orc_demod_set_deemphasis(h, 50)
                e.set_deemphasis_us(50)
        if i == 7:
            for h, e in ((d, eng_u8), (dc, eng_cf)):
                L.orc_demod_reset(h)
                e.reset(fm.engine.RESET_DEMOD)
        want_mono = (i % 3) != 1
        # uint8 path (processSplit): bytes at the DSP rate
        chunk = iq8[2 * pos:2 * (pos + n)]
        mpx = np.zeros(n, np.float32)
        mono = np.zeros(n, np.float32)
        k = L.orc_demod_process_split(d, chunk.ctypes.data_as(U8), _f(mpx), _f(mono) if want_mono else None, n)
        gm, gmono = eng_u8.processSplit(chunk, want_mono)
        assert np.array_equal(gm, mpx)
        if want_mono:
            assert gmono.size == k and np.array_equal(gmono, mono[:k])
        assert eng_u8.clip_ratio() == L.orc_demod_clip_ratio(d)
        # complex path (processSplitComplex) fed by the decimator
        chunk8 = iq8[2 * pos * 8:2 * (pos + n) * 8]
        cf = np.zeros(2 * n, np.float32)
        L.orc_decim_execute_complex(dec, chunk8.ctypes.data_as(U8), n * 8, _f(cf), n)
        k = L.orc_demod_process_split_complex(dc, _f(cf), _f(mpx), _f(mono) if want_mono else None, n)
        gm, gmono = eng_cf.processSplitComplex(cf.view(np.complex64), want_mono)
        assert np.array_equal(gm, mpx)
        if want_mono:
            assert gmono.size == k and np.array_equal(gmono, mono[:k])
        pos += n
    for h in (d, dc):
        L.orc_demod_destroy(h)
    L.orc_decim_destroy(dec)
    eng_u8.close()
    eng_cf.close()


def _mpx(orc_lib, nblk=14, rate=256000, seed=0):
    decim = 8
    iq = orc.config1_signal(fs_iq=rate * decim, seed=seed).generate(nblk * 8192 * decim)
    return orc.Channel(orc_lib, orc.make_config(iq_rate=rate * decim, decimation=decim)).process(
        iq, debug=True).mpx


@pytest.mark.parametrize("blend", [0, 1, 2])
def test_stereo_decoder_blocks_and_flags(orc_fm, blend):
    L = orc_fm.lib
    fs = 256000
    mpx = _mpx(orc_fm)
    s = L.orc_stereo_create(fs)
    L.orc_stereo_set_blend(s, blend)
    eng = fm.Engine(fm.make_config(iq_rate=fs, decimation=1, block_samples=16384, max_blocks=1), 1, 0)
    eng.set_blend_mode(blend)
    sizes = [8192] * 9 + [4096, 100, 1, 8192, 12000, 8192]
    pos = 0
    for i, n in enumerate(sizes):
        if i == 10:
            L.orc_stereo_set_force_mono(s, 1)
            eng.set_force_mono(True)
        if i == 12:
            L.orc_stereo_set_force_mono(s, 0)
            eng.set_force_mono(False)
            L.orc_stereo_set_force_stereo(s, 1)
            eng.set_force_stereo(True)
        if i == 14:
            L.orc_stereo_reset(s)
            eng.reset(fm.engine.RESET_STEREO)
        x = mpx[pos:pos + n]
        l = np.zeros(n, np.float32)
        r = np.zeros(n, np.float32)
        assert L.orc_stereo_process(s, _f(x), _f(l), _f(r), n) == n
        gl, gr = eng.processAudio(x)
        assert np.array_equal(gl, l) and np.array_equal(gr, r), (i, n)
        assert eng.is_stereo() == bool(L.orc_stereo_is_stereo(s)), i     # block-count lock logic
        assert eng.pilot_tenths() == L.orc_stereo_pilot_tenths(s), i
        pos += n
    L.orc_stereo_destroy(s)
    eng.close()


@pytest.mark.parametrize("fs", [256000, 240000])
def test_afpost_capacity_and_deemphasis(orc_fm, fs):
    L = orc_fm.lib
    rng = np.random.default_rng(3)
    a = L.orc_afpost_create(fs, 32000)
    eng = fm.Engine(fm.make_config(iq_rate=fs, decimation=1, block_samples=16384, max_blocks=1,
                                   deemphasis=1), 1, 0)
    for i, (n, cap) in enumerate([(8192, 8192), (1000, 8192), (8192, 100), (5, 8192), (8192, 1024),
                                  (3000, 2), (8192, 8192)]):
        if i == 3:
            L.orc_afpost_set_deemphasis(a, 50)
            eng.set_deemphasis_us(50)
        if i == 5:
            L.orc_afpost_set_deemphasis(a, 0)
            eng.set_deemphasis_us(0)
        if i == 6:
            L.orc_afpost_reset(a)
            eng.reset(fm.engine.RESET_AFPOST)
        l = rng.normal(0, 0.2, n).astype(np.float32)
        r = rng.normal(0, 0.2, n).astype(np.float32)
        ol = np.zeros(cap, np.float32)
        orr = np.zeros(cap, np.float32)
        k = L.orc_afpost_process(a, _f(l), _f(r), n, _f(ol), _f(orr), cap)
        gl, gr = eng.afpost(l, r, cap)
        assert gl.size == k, (i, gl.size, k)
        assert np.array_equal(gl, ol[:k]) and np.array_equal(gr, orr[:k]), i
    L.orc_afpost_destroy(a)
    eng.close()


def test_rds_decoder_chunks_and_reset(orc_fm):
    L = orc_fm.lib
    fs = 256000
    mpx = _mpx(orc_fm, nblk=30)
    d = L.orc_rds_create(fs)
    eng = fm.Engine(fm.make_config(iq_rate=fs, decimation=1, block_samples=32768, max_blocks=1), 1, 0)
    sizes = [8192, 8192, 1, 999, 20000, 8192, 8192, 30000, 8192, 8192, 8192, 8192, 16384, 8192, 8192]
    pos = 0
    tot = 0
    for i, n in enumerate(sizes):
        if i == 9:
            L.orc_rds_reset(d)
            eng.reset(fm.engine.RESET_RDS)
        x = mpx[pos:pos + n]
        out = np.zeros(16, orc.GROUP_DTYPE)
        k = L.orc_rds_process(d, _f(x), n, out.ctypes.data, 16)
        got = eng.rds(x, cap=16)
        assert groups_equal(got, out[:k], keys=("a", "b", "c", "d", "errors")), i
        tot += k
        pos += n
    assert tot >= 3
    L.orc_rds_destroy(d)
    eng.close()


def test_stage_calls_chained_on_one_engine():
    """Every stage-level call carries only its own stage's halos and state: the five calls chained block
    after block on ONE engine channel give, bit for bit, what each gives on an engine of its own."""
    sizes = RAGGED + [16384, 12001, 16384, 9000] * 6
    iq = orc.config1_signal(fs_iq=2_048_000, seed=5).generate(sum(sizes) * 8)
    cfg = fm.make_config(iq_rate=2_048_000, decimation=8, block_samples=16384, max_blocks=1)
    shared = fm.Engine(cfg, 1, 0)
    own = [fm.Engine(cfg, 1, 0) for _ in range(5)]

    def chain(dec, dem, ste, afp, rds, chunk, n, cap):
        x = dec.executeComplex(chunk, n)
        mpx, mono = dem.processSplitComplex(x, want_mono=True)
        left, right = ste.processAudio(mpx)
        al, ar = afp.afpost(left, right, cap)
        return (x, mpx, mono, left, right, al, ar), rds.rds(mpx, cap=64)

    pos = n_groups = 0
    for i, n in enumerate(sizes):
        chunk = iq[2 * 8 * pos:2 * 8 * (pos + n)]
        cap = n if i % 4 else max(2, n // 10)   # a short capacity leaves part of the L/R input unused
        got, g_got = chain(*[shared] * 5, chunk, n, cap)
        ref, g_ref = chain(*own, chunk, n, cap)
        assert got[0].size == n and got[1].size == n
        for k, (a, b) in enumerate(zip(got, ref)):
            assert a.size == b.size and np.array_equal(a, b), (i, n, k)
        assert groups_equal(g_got, g_ref), i
        n_groups += len(g_ref)
        pos += n
    assert n_groups >= 3
    for e in (shared, *own):
        e.close()


def test_null_and_empty_arguments_return_zero():
    eng = fm.Engine(fm.make_config(iq_rate=256000, decimation=1, max_blocks=1), 1, 0)
    L = eng.L
    z = np.zeros(16, np.float32)
    assert L.fmgpu_stereo(eng.h, 0, None, z.ctypes.data, z.ctypes.data, 16) == 0
    assert L.fmgpu_stereo(eng.h, 0, z.ctypes.data, z.ctypes.data, z.ctypes.data, 0) == 0
    assert L.fmgpu_afpost(eng.h, 0, z.ctypes.data, z.ctypes.data, 16, z.ctypes.data, z.ctypes.data, 0) == 0
    assert L.fmgpu_rds(eng.h, 0, None, 16, None, 0) == 0
    assert L.fmgpu_demod_u8(eng.h, 0, None, z.ctypes.data, None, 8) == 0
    assert L.fmgpu_decimate(eng.h, 0, z.ctypes.data, 0, z.ctypes.data, 8) == 0
    assert L.fmgpu_stereo(eng.h, 5, z.ctypes.data, z.ctypes.data, z.ctypes.data, 16) == 0   # bad channel
    big = np.zeros(8192 * 2, np.float32)                                                     # > engine size
    assert L.fmgpu_stereo(eng.h, 0, big.ctypes.data, big.ctypes.data, big.ctypes.data, big.size) == 0
    assert "sized for" in eng.error()
    eng.close()

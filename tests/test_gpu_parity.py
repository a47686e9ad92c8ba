"""GPU engine vs CPU oracle through the C ABI, whole pipeline (the per-block body of
src/main.cpp:1232-1308). Bars (BASELINE.json north_star):
  * vs the fm-flavoured oracle (same transcendental kernels): EVERYTHING bit-exact — decimated
    IQ, MPX, DSP-rate L/R, 32 kHz audio, per-block status, RDS bits and groups;
  * vs the libm-flavoured oracle (faithful to the reference's libm call sites): audio within
    1e-4 of full scale max-abs and >= 90 dB SNR after pilot lock, stereo-lock block equal,
    pilot tenths within 1, RDS groups byte-equal.
"""
import numpy as np
import pytest

import fmtuner_sdr_b200 as fm
from oracle import orc
from tests.common import groups_equal, rates, run_engine_chunks, snr_db

pytestmark = pytest.mark.gpu


def _compare_exact(eng_audio, eng_groups, eng_status, dbg, ref, decim):
    if decim > 1:
        assert np.array_equal(dbg["dec"].view(np.float32), ref.dec.view(np.float32))
    assert np.array_equal(dbg["mpx"], ref.mpx)
    assert np.array_equal(dbg["sl"], ref.sl) and np.array_equal(dbg["sr"], ref.sr)
    assert np.array_equal(eng_audio[0], ref.left) and np.array_equal(eng_audio[1], ref.right)
    for k in ("n_audio", "stereo", "pilot_tenths", "clip_ratio", "n_groups"):
        assert np.array_equal(eng_status[k], ref.status[k]), k
    assert groups_equal(eng_groups, ref.groups)


@pytest.mark.parametrize("rate", ["240k", "256k", "1024k", "direct256k", "480k", "m2", "m16"])
def test_config2_single_channel_bit_exact(orc_fm, orc_libm, rate):
    """BASELINE config 2: the config-1 multiplex on one channel, compared per block."""
    iq_rate, decim = rates(rate)
    nblk = 16
    iq = orc.config1_signal(fs_iq=iq_rate).generate(nblk * 8192 * decim)
    kw = dict(iq_rate=iq_rate, decimation=decim)
    och = orc.Channel(orc_fm, orc.make_config(**kw))
    ref = och.process(iq, debug=True)
    eng = fm.Engine(fm.make_config(max_blocks=4, **kw), 1, 0)
    audio, groups, status, dbg = run_engine_chunks(eng, iq.reshape(1, -1), nblk, 4, debug_channel=0)
    _compare_exact(audio[0], groups[0], status[0], dbg, ref, decim)
    assert eng.launch_count() > 0
    # tolerance gate against the libm-faithful oracle
    rl = orc.Channel(orc_libm, orc.make_config(**kw)).process(iq)
    first = int(np.flatnonzero(rl.status["stereo"])[0])
    assert int(np.flatnonzero(status[0]["stereo"])[0]) == first      # pilot lock time matches
    assert np.abs(audio[0][0] - rl.left).max() <= 1e-4 and np.abs(audio[0][1] - rl.right).max() <= 1e-4
    k0 = int(rl.status["n_audio"][:first + 1].sum())
    assert snr_db(rl.left[k0:], audio[0][0][k0:]) >= 90.0
    assert np.abs(status[0]["pilot_tenths"] - rl.status["pilot_tenths"]).max() <= 1
    assert groups_equal(groups[0], rl.groups)
    eng.close()


def test_blocks_per_call_do_not_change_results(orc_fm):
    """1, 2 or 4 logical blocks per launch sequence: identical outputs (state carried exactly)."""
    iq_rate, decim = rates("240k")
    nblk = 8
    iq = orc.config1_signal(fs_iq=iq_rate, seed=3).generate(nblk * 8192 * decim).reshape(1, -1)
    outs = []
    for chunk in (1, 2, 4):
        eng = fm.Engine(fm.make_config(max_blocks=4), 1, 0)
        outs.append(run_engine_chunks(eng, iq, nblk, chunk))
        eng.close()
    for a, g, st, _ in outs[1:]:
        assert np.array_equal(a[0], outs[0][0][0])
        assert groups_equal(g[0], outs[0][1][0])
        assert np.array_equal(st, outs[0][2])


def test_pipeline_groups_do_not_change_results():
    """Channel groups on separate streams (overlap of lane / FIR kernels and host copies)."""
    iq_rate, decim = rates("240k")
    C, nblk = 70, 4
    rng = np.random.default_rng(11)
    base = np.stack([orc.config3_signal(300 + c, fs_iq=iq_rate).generate(nblk * 8192 * decim)
                     for c in range(6)])
    iq = base[rng.integers(0, 6, C)]
    ref = None
    for groups in (1, 2, 3, 8):
        eng = fm.Engine(fm.make_config(max_blocks=2, dsp_agc=1), C, 0)
        eng.set_pipeline_groups(groups)
        out = run_engine_chunks(eng, iq, nblk, 2)
        eng.close()
        if ref is None:
            ref = out
            continue
        for c in range(C):
            assert np.array_equal(out[0][c], ref[0][c]), (groups, c)
            assert groups_equal(out[1][c], ref[1][c]), (groups, c)
        assert np.array_equal(out[2], ref[2])


def test_config3_varied_channels_bit_exact(orc_fm):
    """BASELINE config 3 (reduced to 24 channels x 8 blocks so the oracle finishes in seconds):
    varied deviation / SNR / tones / RDS payload per channel, batched on one GPU."""
    iq_rate, decim = rates("240k")
    C, nblk = 24, 8
    sigs = [orc.config3_signal(c, fs_iq=iq_rate) for c in range(C)]
    iq = np.stack([s.generate(nblk * 8192 * decim) for s in sigs])
    eng = fm.Engine(fm.make_config(max_blocks=4), C, 0)
    audio, groups, status, _ = run_engine_chunks(eng, iq, nblk, 4)
    for c in range(C):
        ch = orc.Channel(orc_fm, orc.make_config())
        ref = ch.process(iq[c])
        assert np.array_equal(audio[c][0], ref.left) and np.array_equal(audio[c][1], ref.right), c
        assert np.array_equal(status[c]["stereo"], ref.status["stereo"]), c
        assert np.array_equal(status[c]["pilot_tenths"], ref.status["pilot_tenths"]), c
        assert groups_equal(groups[c], ref.groups), c
        assert np.array_equal(eng.debug_rds_bits(c), ch.rds_bits()[-eng.debug_rds_bits(c).size:]), c
    eng.close()


@pytest.mark.parametrize("agc,blend,deemph", [(1, 0, 1), (2, 2, 2), (1, 1, 0)])
def test_config5_weak_signal_settings(orc_fm, agc, blend, deemph):
    """BASELINE config 5 flavour: SNR 10-40 dB, blend soft/normal/aggressive, dsp_agc on."""
    iq_rate, decim = rates("240k")
    C, nblk = 8, 10
    rng = np.random.default_rng(50 + agc)
    iq = []
    for c in range(C):
        s = orc.config3_signal(100 + c, fs_iq=iq_rate)
        s.snr_db = float(rng.uniform(10.0, 40.0))
        iq.append(s.generate(nblk * 8192 * decim))
    iq = np.stack(iq)
    kw = dict(dsp_agc=agc, stereo_blend=blend, deemphasis=deemph)
    eng = fm.Engine(fm.make_config(max_blocks=5, **kw), C, 0)
    audio, groups, status, _ = run_engine_chunks(eng, iq, nblk, 5)
    for c in range(C):
        ch = orc.Channel(orc_fm, orc.make_config(**kw))
        ref = ch.process(iq[c])
        assert np.array_equal(audio[c][0], ref.left) and np.array_equal(audio[c][1], ref.right), c
        assert np.array_equal(status[c], ref.status), c
        assert groups_equal(groups[c], ref.groups), c
    eng.close()


def test_mono_mode_and_force_mono(orc_fm):
    iq_rate, decim = rates("256k")
    nblk = 6
    iq = orc.config1_signal(fs_iq=iq_rate).generate(nblk * 8192 * decim)
    for kw in (dict(stereo=0), dict(force_mono=1)):
        full = dict(iq_rate=iq_rate, decimation=decim, **kw)
        ref = orc.Channel(orc_fm, orc.make_config(**full)).process(iq)
        eng = fm.Engine(fm.make_config(max_blocks=3, **full), 1, 0)
        audio, groups, status, _ = run_engine_chunks(eng, iq.reshape(1, -1), nblk, 3)
        assert np.array_equal(audio[0][0], ref.left) and np.array_equal(audio[0][1], ref.right)
        assert np.array_equal(status[0]["n_audio"], ref.status["n_audio"])
        assert groups_equal(groups[0], ref.groups)
        eng.close()


def test_retune_reset_and_bandwidth_change(orc_fm):
    """dspRuntime.reset + rdsReset between blocks (main.cpp:1028-1062) and an XDR 'W' command."""
    iq_rate, decim = rates("240k")
    a = orc.config1_signal(fs_iq=iq_rate, seed=1).generate(10 * 8192 * decim)
    b = orc.config3_signal(5, fs_iq=iq_rate).generate(10 * 8192 * decim)
    och = orc.Channel(orc_fm, orc.make_config())
    eng = fm.Engine(fm.make_config(max_blocks=5), 1, 0)

    def both(iq):
        ref = och.process(iq)
        audio, groups, status, _ = run_engine_chunks(eng, iq.reshape(1, -1), 10, 5)
        assert np.array_equal(audio[0][0], ref.left) and np.array_equal(audio[0][1], ref.right)
        assert np.array_equal(status[0], ref.status)
        assert groups_equal(groups[0], ref.groups)

    both(a)
    och.reset(dsp=True, rds=True)
    eng.reset(fm.engine.RESET_ALL)
    both(b)
    och.set_bandwidth_hz(56000)
    eng.set_bandwidth_hz(56000)
    both(a)
    och.reset(dsp=True, rds=False)      # scan restore without an RDS reset
    eng.reset(fm.engine.RESET_DSP)
    both(b)
    eng.close()


def test_per_channel_settings(orc_fm):
    """Channels of one engine carry their own bandwidth / AGC / blend / de-emphasis."""
    iq_rate, decim = rates("240k")
    C, nblk = 4, 8
    iq = np.stack([orc.config3_signal(200 + c, fs_iq=iq_rate).generate(nblk * 8192 * decim)
                   for c in range(C)])
    settings = [dict(), dict(bandwidth_hz=114000, dsp_agc=1), dict(stereo_blend=2, deemphasis=1),
                dict(bandwidth_hz=42000, stereo_blend=0, deemphasis=2, dsp_agc=2)]
    eng = fm.Engine(fm.make_config(max_blocks=4), C, 0)
    for c, s in enumerate(settings):
        if "bandwidth_hz" in s:
            eng.set_bandwidth_hz(s["bandwidth_hz"], c)
        if "dsp_agc" in s:
            eng.set_agc_mode(s["dsp_agc"], c)
        if "stereo_blend" in s:
            eng.set_blend_mode(s["stereo_blend"], c)
        if "deemphasis" in s:
            eng.set_deemphasis_us({0: 50, 1: 75, 2: 0}[s["deemphasis"]], c)
    audio, groups, status, _ = run_engine_chunks(eng, iq, nblk, 4)
    for c, s in enumerate(settings):
        ref = orc.Channel(orc_fm, orc.make_config(**s)).process(iq[c])
        assert np.array_equal(audio[c][0], ref.left) and np.array_equal(audio[c][1], ref.right), c
        assert np.array_equal(status[c], ref.status), c
        assert groups_equal(groups[c], ref.groups), c
    eng.close()


def test_clipping_statistics(orc_fm):
    iq_rate, decim = rates("direct256k")
    sig = orc.config1_signal(fs_iq=iq_rate)
    sig.iq_amp = 1.2     # drives bytes to 0 / 255
    iq = sig.generate(3 * 8192)
    kw = dict(iq_rate=iq_rate, decimation=decim)
    ref = orc.Channel(orc_fm, orc.make_config(**kw)).process(iq)
    eng = fm.Engine(fm.make_config(max_blocks=3, **kw), 1, 0)
    _, _, status, _ = run_engine_chunks(eng, iq.reshape(1, -1), 3, 3)
    assert (ref.status["clip_ratio"] > 0.05).all()
    assert np.array_equal(status[0]["clip_ratio"], ref.status["clip_ratio"])
    assert eng.is_clipping(0) and eng.clip_ratio(0) == ref.status["clip_ratio"][-1]
    eng.close()


def test_one_channel_reset_leaves_the_lanes_out_of_step(orc_fm):
    """Retune of ONE channel of a batch (dspRuntime.reset + rdsReset, main.cpp:1028-1062) while its
    neighbours keep going: afterwards the lanes of a warp sit at different /24 decimation phases,
    different symbol-clock phases and different pilot-lock states, which the lane kernels (k_rds
    walks groups that end at each lane's own decimation instant) must handle per lane."""
    iq_rate, decim = rates("240k")
    C, nblk = 5, 12
    sig = [orc.config3_signal(300 + c, fs_iq=iq_rate) for c in range(C)]
    first = np.stack([s.generate(3 * 8192 * decim) for s in sig])
    rest = np.stack([s.generate(nblk * 8192 * decim, start_sample=3 * 8192 * decim) for s in sig])
    eng = fm.Engine(fm.make_config(max_blocks=4), C, 0)
    chans = [orc.Channel(orc_fm, orc.make_config()) for _ in range(C)]
    a0, g0, s0, _ = run_engine_chunks(eng, first, 3, 3)
    ref0 = [ch.process(first[c]) for c, ch in enumerate(chans)]
    for victim, what, kw in ((1, fm.engine.RESET_ALL, dict(dsp=True, rds=True)),
                             (3, fm.engine.RESET_DSP, dict(dsp=True, rds=False))):
        eng.reset(what, victim)
        chans[victim].reset(**kw)
    a1, g1, s1, _ = run_engine_chunks(eng, rest, nblk, 4)
    for c, ch in enumerate(chans):
        ref1 = ch.process(rest[c])
        assert np.array_equal(a0[c][0], ref0[c].left) and np.array_equal(a1[c][0], ref1.left), c
        assert np.array_equal(a1[c][1], ref1.right), c
        assert np.array_equal(s1[c], ref1.status), c
        assert groups_equal(g1[c], ref1.groups), c
    assert sum(len(g) for g in g1) > 0
    eng.close()

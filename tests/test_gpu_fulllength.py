"""Full-length and weak-signal parity (BASELINE configs 1, 2 and 5 at their stated lengths).

(a) configs 1/2: the 10 s single-channel multiplex at 2.4 MS/s / 10 (293 logical blocks) and at
    2.048 MS/s / 8 (313 blocks, the unmodified main.cpp's rate): the engine equals the fm-flavour
    oracle BIT FOR BIT over the whole run (hundreds of ring wrap-arounds, seconds of resampler
    phase drift, full PS/RT cycles) and stays inside north_star's tolerance against the
    reference-faithful flavour — the reference's own sources over the liquid shim
    (oracle/_ref/libfmref.so) when built, else the libm restatement, which is identical to it
    (tests/test_oracle_vs_reference.py) — with PI / PS / RT decoded from the groups and compared.
(b) config 5: 320 distinct channels, SNR 10..40 dB, 3 s each, blend mode c % 3, dsp_agc fast,
    against the reference-faithful flavour: per 5 dB bucket the RDS group exact-match rate, audio
    max-abs error and SNR after lock, lock-block equality, pilot level difference; the table is
    printed and saved as JSON (copied to profiles/ and DESIGN.md). Gate, every bucket at or
    above 20 dB: on every channel that the faithful flavour's two builds (strict -ffp-contract=off
    and stock -mfma contraction: oracle/_ref/libfmref_contract.so when the reference was built,
    else the restatement's oracle/liboracle_libm_contract.so) decode identically, the engine's
    groups are byte-equal; lock blocks equal, pilot level within 1, audio in tolerance. Groups may
    differ only on channels at the RDS decoding threshold, where any change of rounding — the
    reference's own compiler flags, the engine's last-ulp sin/cos/atan2/exp/log, the tensor-core
    decimator's single rounding — decides marginal bits; there the aligned group sequences may
    differ in no more than twice as many groups as the stock build differs from the strict
    build. With the FP32 decimator (mode 0) the
    engine additionally reproduces every group the reference decodes clean.
"""
import difflib
import json
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import fmtuner_sdr_b200 as fm
from oracle import orc
from tests.common import groups_equal, rates, run_engine_chunks, snr_db

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def faithful_lib():
    """The reference-faithful CPU flavour: the reference's own code when it was built."""
    return orc.OracleLib("ref") if orc.OracleLib.have_ref("ref") else orc.OracleLib("libm")


def stock_build_lib():
    """The faithful flavour built with gcc's default FMA contraction: the reference's own stock build
    when it was built, else the restatement's. The sweep checks that the one it uses marks as many
    threshold channels, differing in as many groups, per SNR bucket as the reference's stock build
    did (tests/golden/reference_sweep_buckets.json)."""
    return (orc.OracleLib("ref_contract") if orc.OracleLib.have_ref("ref_contract")
            else orc.OracleLib("libm_contract"))


def audio_start(status, extra_blocks=2, never=8):
    """First 32 kHz frame after PLL lock (+ settling): north_star compares audio 'after PLL lock'."""
    on = np.flatnonzero(status["stereo"])
    blk = (int(on[0]) + extra_blocks) if on.size else never
    blk = min(blk, len(status) - 16)     # a late lock still leaves half a second to compare
    return int(status["n_audio"][:blk].sum()), (int(on[0]) if on.size else -1)


@pytest.mark.parametrize("mode", [0, 1], ids=["reference-order", "fast-arithmetic"])
@pytest.mark.parametrize("rate,nblk", [("240k", 293), ("256k", 313)])
def test_config1_ten_seconds(orc_fm, rate, nblk, mode):
    """mode 0: the reference's summation order everywhere — bit for bit. mode 1: the engine's fast
    arithmetic (tensor-core decimator + scan de-emphasis, bench.py's default) — the tolerance
    gates against the faithful flavour."""
    iq_rate, decim = rates(rate)
    iq = orc.config1_signal(fs_iq=iq_rate).generate(nblk * 8192 * decim)
    eng = fm.Engine(fm.make_config(iq_rate=iq_rate, decimation=decim, max_blocks=8), 1, 0)
    eng.set_decimator_mode(mode)
    eng.set_scan_mode(mode)       # mode 1 = the engine's fast arithmetic, as bench.py runs it
    eng.set_fir_mode(mode)
    eng.set_demod_mode(mode)
    audio, groups, status, dbg = run_engine_chunks(eng, iq.reshape(1, -1), nblk, 8, debug_channel=0)
    eng.close()
    a, g, st = audio[0], groups[0], status[0]

    if mode == 0:
        ref = orc.Channel(orc_fm, orc.make_config(iq_rate=iq_rate, decimation=decim)).process(iq, debug=True)
        assert np.array_equal(dbg["mpx"], ref.mpx)
        assert np.array_equal(a[0], ref.left) and np.array_equal(a[1], ref.right)
        assert np.array_equal(st, ref.status) and groups_equal(g, ref.groups)
    assert len(g) >= 100      # 10 s of RDS: ~114 groups minus acquisition

    faith = orc.Channel(faithful_lib(), orc.make_config(iq_rate=iq_rate, decimation=decim)).process(iq)
    assert groups_equal(g, faith.groups)
    assert orc.decode_ps_rt(g) == orc.decode_ps_rt(faith.groups) == (0x1234, "B200TEST", "FM ON B200")
    assert np.array_equal(st["stereo"], faith.status["stereo"])
    assert np.abs(st["pilot_tenths"] - faith.status["pilot_tenths"]).max() <= 1
    s0, lock = audio_start(faith.status)
    assert 6 <= lock <= 8
    for x, y in ((a[0], faith.left), (a[1], faith.right)):
        assert x.size == y.size
        assert np.abs(x[s0:] - y[s0:]).max() <= 1e-4 or snr_db(y[s0:], x[s0:]) >= 90.0


def _sweep_signal(c, n_ch, iq_rate):
    # config-3 style channel (tones 400 + 37 k / 700 + 53 k Hz stay below 15 kHz for k < 256)
    s = orc.config3_signal(c % 256, fs_iq=iq_rate)
    s.seed = 7000 + c
    s.snr_db = 10.0 + 30.0 * (c + 0.5) / n_ch      # uniform over 10..40 dB
    return s


@pytest.mark.parametrize("mode", [0, 1], ids=["reference-order", "fast-arithmetic"])
def test_config5_weak_signal_sweep_vs_faithful_reference(orc_fm, mode):
    iq_rate, decim = rates("240k")
    n_ch, nblk, chunk, per_pass = 320, 88, 8, 80     # 88 blocks = 3.0 s
    faith_lib = faithful_lib()
    stock_lib = stock_build_lib()
    rows = []
    orc.config1_signal(fs_iq=iq_rate).generate(16)   # builds the generator's pulse table once

    def cpu_side(c):
        sig = _sweep_signal(c, n_ch, iq_rate)
        iq = sig.generate(nblk * 8192 * decim)
        cfg = orc.make_config(iq_rate=iq_rate, decimation=decim, dsp_agc=1, stereo_blend=c % 3)
        stock = orc.Channel(stock_lib, cfg).process(iq).groups
        return (iq, orc.Channel(faith_lib, cfg).process(iq), orc.Channel(orc_fm, cfg).process(iq),
                sig.snr_db, stock)

    with ThreadPoolExecutor(max_workers=os.cpu_count() or 8) as pool:
        for c0 in range(0, n_ch, per_pass):
            chans = list(range(c0, min(n_ch, c0 + per_pass)))
            cpu = list(pool.map(cpu_side, chans))
            eng = fm.Engine(fm.make_config(iq_rate=iq_rate, decimation=decim, max_blocks=chunk,
                                           dsp_agc=1), len(chans), 0)
            eng.set_decimator_mode(mode)
            eng.set_scan_mode(mode)
            eng.set_fir_mode(mode)
            eng.set_demod_mode(mode)
            for i, c in enumerate(chans):
                eng.set_blend_mode(c % 3, i)
            audio, groups, status, _ = run_engine_chunks(eng, np.stack([x[0] for x in cpu]), nblk, chunk)
            eng.close()
            for i, c in enumerate(chans):
                _, faith, exact, snr, stock = cpu[i]
                a, g, st = audio[i], groups[i], status[i]
                if mode == 0:
                    # the engine's own arithmetic flavour: everything bit for bit, weak signals included
                    assert np.array_equal(a[0], exact.left) and np.array_equal(a[1], exact.right), c
                    assert np.array_equal(st, exact.status) and groups_equal(g, exact.groups), c
                s0, lock = audio_start(faith.status)
                _, lock_gpu = audio_start(st)
                def same_at(x, k):
                    return k < len(x) and all(x[k][f] == faith.groups[k][f]
                                              for f in ("a", "b", "c", "d", "errors", "block_index"))

                def unmatched(x):
                    """groups of the reference sequence without a partner in x, after aligning the
                    two sequences (a dropped or late group must not count every later one)"""
                    key = lambda g: tuple(int(g[f]) for f in ("a", "b", "c", "d", "errors"))
                    ra, xa = [key(g) for g in faith.groups], [key(g) for g in x]
                    m = difflib.SequenceMatcher(a=ra, b=xa, autojunk=False)
                    return max(len(ra), len(xa)) - sum(blk.size for blk in m.get_matching_blocks())

                nref = len(faith.groups)
                same = sum(same_at(g, k) for k in range(nref))
                clean = [k for k in range(nref) if faith.groups[k]["errors"] == 0]
                clean_same = sum(same_at(g, k) for k in clean)
                gpu_diff = unmatched(g)
                stock_diff = unmatched(stock)
                err = max(float(np.abs(a[0][s0:] - faith.left[s0:]).max()),
                          float(np.abs(a[1][s0:] - faith.right[s0:]).max()))
                rows.append(dict(
                    c=c, snr_db=snr, groups_ref=int(len(faith.groups)), groups_gpu=int(len(g)),
                    groups_same=int(same), groups_equal=bool(groups_equal(g, faith.groups)),
                    clean_ref=len(clean), clean_same=int(clean_same), stock_build_diff=stock_diff,
                    gpu_diff=int(gpu_diff),
                    # "robust": the faithful flavour's two builds decode this channel identically
                    robust=bool(stock_diff == 0),
                    lock_ref=lock, lock_gpu=lock_gpu,
                    stereo_flags_equal=bool(np.array_equal(st["stereo"], faith.status["stereo"])),
                    pilot_diff=int(np.abs(st["pilot_tenths"] - faith.status["pilot_tenths"]).max()),
                    audio_maxabs=err,
                    audio_snr_db=float(min(snr_db(faith.left[s0:], a[0][s0:]),
                                           snr_db(faith.right[s0:], a[1][s0:])))))

    table = []
    for lo in range(10, 40, 5):
        b = [r for r in rows if lo <= r["snr_db"] < lo + 5]
        table.append(dict(
            snr_bucket_db=f"{lo}-{lo + 5}", channels=len(b),
            groups_ref=sum(r["groups_ref"] for r in b),
            groups_gpu=sum(r["groups_gpu"] for r in b),
            group_exact_match_rate=(sum(r["groups_same"] for r in b) / sum(r["groups_ref"] for r in b)
                                    if sum(r["groups_ref"] for r in b) else
                                    float(sum(r["groups_gpu"] for r in b) == 0)),
            groups_different=sum(r["gpu_diff"] for r in b),
            reference_stock_build_groups_different=sum(r["stock_build_diff"] for r in b),
            clean_groups_ref=sum(r["clean_ref"] for r in b),
            clean_group_match_rate=(sum(r["clean_same"] for r in b) / sum(r["clean_ref"] for r in b)
                                    if sum(r["clean_ref"] for r in b) else 1.0),
            channels_all_groups_equal=sum(r["groups_equal"] for r in b) / len(b),
            robust_channels=sum(r["robust"] for r in b),
            robust_channels_all_groups_equal=(sum(r["groups_equal"] for r in b if r["robust"]) /
                                              max(1, sum(r["robust"] for r in b))),
            lock_block_equal=sum(r["lock_ref"] == r["lock_gpu"] and r["stereo_flags_equal"] for r in b) / len(b),
            locked_channels=sum(r["lock_ref"] >= 0 for r in b),
            pilot_tenths_maxdiff=max(r["pilot_diff"] for r in b),
            audio_maxabs=max(r["audio_maxabs"] for r in b),
            audio_snr_db_min=min(r["audio_snr_db"] for r in b)))
    out = dict(config="BASELINE config 5: 320 channels x 3 s, SNR 10-40 dB, blend c%3, dsp_agc fast",
               reference_flavour=faith_lib.math, stock_build_flavour=stock_lib.math,
               arithmetic=("fast: tensor-core int8 decimator, fused tensor-core channel filter + discriminator "
                           "(AGC elided), tensor-core pilot / low-pass FIRs, scans (modes 1)" if mode else
                           "reference order everywhere (modes 0)"),
               buckets=table)
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    with open(os.path.join(ROOT, "gpurun_out", f"parity_sweep_mode{mode}.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))
    # The reference side of the table as the reference's own two builds computed it: the faithful
    # flavour's groups and locks, and which channels its stock build decodes differently (the
    # channels the gate below treats as threshold channels) must be what the reference gave.
    with open(os.path.join(ROOT, "tests", "golden", "reference_sweep_buckets.json")) as f:
        recorded = json.load(f)["buckets"]
    assert len(recorded) == len(table)
    for t, r in zip(table, recorded):
        assert {k: t[k] for k in r} == r, (t, r)
    for t in table:
        if int(t["snr_bucket_db"].split("-")[0]) >= 20:
            # bit-exact wherever the reference is bit-stable under its own build variation
            assert t["robust_channels"] >= 40 and t["robust_channels_all_groups_equal"] == 1.0, t
            if mode == 0:
                assert t["clean_groups_ref"] > 1000 and t["clean_group_match_rate"] == 1.0, t
                assert t["group_exact_match_rate"] >= 0.99, t
            # threshold channels: no further from the strict reference than its own stock build
            # (aligned sequences; twice its count leaves room for which marginal bits flip)
            assert t["groups_different"] <= max(2, 2 * t["reference_stock_build_groups_different"]), t
            assert t["lock_block_equal"] == 1.0 and t["pilot_tenths_maxdiff"] <= 1, t
            assert t["audio_maxabs"] <= 1e-4 or t["audio_snr_db_min"] >= 90.0, t

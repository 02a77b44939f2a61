"""Pins the plain-C oracle port (oracle/modes_oracle.c) against the UNMODIFIED reference objects (the reference's
lib/*.cc compiled against oracle/shim into oracle/_ref), as recorded in tests/golden/ref_results.json.xz. CPU only."""
import numpy as np
import pytest

from gr_air_modes_b200 import synth
from oracle import cpu_oracle as co

from helpers import chips_digest, load_golden, parse_msg

KNOWN = [("8D4840D6202CC371C32CE0576098", 0x576098), ("8D40621D58C382D690C8AC2863A7", 0x2863A7)]


def test_crc_known_answers(port):
    for hexs, want in KNOWN:
        b = bytes.fromhex(hexs)
        assert port.crc24(b[:11]) == want
        assert synth.crc24(b[:11]) == want


def test_crc_port_equals_reference(port, ref):
    rng = np.random.default_rng(0)
    for length in (4, 11):
        for _ in range(200):
            b = rng.integers(0, 256, length, dtype=np.uint8).tobytes()
            assert port.crc24(b) == ref.crc24(b)
    assert ref.crc24(bytes([0, 0, 1])) == 0xFFF409  # crc_table[1] == POLY (modes_crc.cc:57)


@pytest.mark.parametrize("rate,thr", [(2e6, 7.0), (4e6, 7.0), (10e6, 3.5), (20e6, 7.0), (3e6, 7.0), (5e6, 9.0), (2.4e6, 7.0)])
def test_params_match_reference(port, ref, rate, thr):
    p = port.params(rate, thr)
    r, t, h = ref.preamble_params(rate, thr)
    assert (float(p.rate_int), p.threshold_db, p.history) == (r, t, h)


@pytest.mark.parametrize("rate,n,nb,pmf,thr,seed", [
    (2e6, 400_000, 30, True, 7.0, 1), (4e6, 400_000, 30, True, 7.0, 2), (4e6, 400_000, 30, False, 7.0, 3),
    (10e6, 600_000, 20, True, 7.0, 4), (20e6, 1_000_000, 16, True, 7.0, 5), (4e6, 400_000, 30, True, 4.0, 6),
    (5e6, 300_000, 20, True, 7.0, 7), (3e6, 300_000, 20, True, 7.0, 8), (2.4e6, 300_000, 20, True, 6.0, 9),
    (4e6, 300_000, 300, True, 6.0, 10), (10e6, 500_000, 20, False, 7.0, 11), (7e6, 400_000, 20, True, 7.0, 12),
])
def test_port_matches_reference_on_scenes(port, ref, rate, n, nb, pmf, thr, seed):
    sc = synth.make_scene(rate, n, nb, seed, garble_frac=0.2 if nb > 100 else 0.0, fruit=50 if nb > 100 else 0)
    bb, avg = port.frontend(sc.iq, rate, pmf, co.MA_CANONICAL)
    r = ref.run_streams(bb, avg, rate, thr)
    p = port.run_streams(bb, avg, rate, thr)
    assert len(r.index) > 0
    assert np.array_equal(r.index, p.index)
    assert np.array_equal(r.secs, p.secs) and np.array_equal(r.frac, p.frac)
    assert r.chips_sha256 == chips_digest(p.chips)   # bit-exact 240-chip packets
    assert r.msgs == p.msgs                           # incl. the sticky-precision quirk
    assert r.calls == p.calls
    q = port.run_iq(sc.iq, rate, thr, pmf, co.MA_CANONICAL)
    assert q.msgs == r.msgs


def test_end_of_stream_rules(port, ref):
    """Bursts cut off by the end of the file exercise the 'no room' path (preamble_impl.cc:212-216)."""
    rate = 4e6
    for cut in range(0, 700, 37):
        sc = synth.make_scene(rate, 60_000, 0, 11, starts=[20_000.3, 59_200.0 - cut], amplitude=0.3)
        bb, avg = port.frontend(sc.iq, rate, True, co.MA_CANONICAL)
        r = ref.run_streams(bb, avg, rate, 7.0)
        p = port.run_streams(bb, avg, rate, 7.0)
        assert np.array_equal(r.index, p.index) and r.msgs == p.msgs and r.calls == p.calls


def test_empty_and_tiny_streams(port, ref):
    for n in (0, 1, 2, 3, 5, 17, 239, 481):
        z = np.zeros(n, np.float32)
        r = ref.run_streams(z, z, 4e6, 7.0)
        p = port.run_streams(z, z, 4e6, 7.0)
        assert len(r.index) == len(p.index) == 0 and r.calls == p.calls


def test_slicer_only_matches_reference(port, ref):
    rng = np.random.default_rng(5)
    chips = rng.normal(0.0, 0.3, (300, 240)).astype(np.float32)
    chips[:, [0, 2, 7, 9]] += 1.0
    chips[::3, 16:240:2] += 1.0     # plenty of ones
    secs = np.arange(300, dtype=np.uint64)
    frac = rng.random(300)
    r = ref.run_slicer(chips, secs, frac)
    p = port.run_slicer(chips, secs, frac)
    assert r.msgs == p.msgs and len(r.msgs) > 0


def test_moving_average_schedules_do_not_change_frames(port, ref):
    """SURVEY 7.3-2: GR's fp32 running sum (chunk dependent) vs the canonical fp64 window."""
    sc = synth.make_scene(4e6, 500_000, 60, 21)
    base = port.run_iq(sc.iq, 4e6, 7.0, True, co.MA_CANONICAL).msgs
    for mode, chunk in ((co.MA_GR_FLOAT, 4096), (co.MA_GR_FLOAT, 1024), (co.MA_SLIDING64, 0)):
        other = port.run_iq(sc.iq, 4e6, 7.0, True, mode, chunk).msgs
        assert [m.split()[:2] for m in other] == [m.split()[:2] for m in base]
        for a, b in zip(other, base):
            assert abs(10 * np.log10(parse_msg(a)[2]) - 10 * np.log10(parse_msg(b)[2])) < 1e-3


def test_golden_fixtures_reproduce(port):
    """The committed reference-generated goldens (tests/golden) are what the port computes."""
    meta, scenes = load_golden()
    for e in meta["crc"]:
        b = bytes.fromhex(e["frame"])
        assert "%06x" % port.crc24(b[:11]) == e["crc_first_11"] and e["syndrome"] == "000000"
    for s, iq in scenes:
        r = port.run_iq(iq, s["rate"], s["threshold_db"], s["use_pmf"], co.MA_CANONICAL)
        assert [int(x) for x in r.index] == s["det_index"], s["name"]
        assert r.msgs == s["msgs"], s["name"]
        sent = set(s["sent"])
        assert len(sent & {m.split()[0] for m in r.msgs}) >= 1


def test_golden_fixtures_against_live_reference(port, ref):
    meta, scenes = load_golden()
    for s, iq in scenes:
        bb, avg = port.frontend(iq, s["rate"], s["use_pmf"], co.MA_CANONICAL)
        r = ref.run_streams(bb, avg, s["rate"], s["threshold_db"])
        assert r.msgs == s["msgs"]
        assert r.chips_sha256 == s["chips_sha256"]


def test_rx_time_tag_at_stream_start(port, ref):
    """tag_to_timestamp with an rx_time tag at item 0 (preamble_impl.cc:100-137), incl. the `> 1.0f` carry."""
    sc = synth.make_scene(4e6, 400_000, 30, 3)
    bb, avg = port.frontend(sc.iq, 4e6, True, co.MA_CANONICAL)
    for st in ((1234567, 0.25), (7, 0.9999999), (0, 0.5)):
        r = ref.run_streams(bb, avg, 4e6, 7.0, start_time=st)
        port.set_start_time(*st)
        try:
            p = port.run_streams(bb, avg, 4e6, 7.0)
        finally:
            port.set_start_time(0, 0.0)
        assert r.msgs == p.msgs and np.array_equal(r.secs, p.secs) and np.array_equal(r.frac, p.frac)


def test_dc_blocker_restatement_sanity(port):
    """a2 (rx_path.py:39-41) is GNU Radio code that is not in the reference tree: parity UNPINNED. What can be
    checked: the canonical (fp64 window) and the GNU Radio recursive-fp32 formulations agree to rounding, a
    constant offset is removed after the 2(D-1)-sample transient, the delay is D-1, and both formulations
    decode the same payloads."""
    rate, D = 4e6, 200
    sc = synth.make_scene(rate, 300_000, 30, 3)
    iq = sc.iq.copy(); iq[0::2] += np.float32(0.05); iq[1::2] -= np.float32(0.03)
    y0 = port.dc_blocker(iq, D, co.MA_CANONICAL)
    y1 = port.dc_blocker(iq, D, co.MA_GR_FLOAT)
    assert np.abs(y0 - y1).max() < 1e-5
    assert abs(y0[2 * 5000::2].mean()) < 1e-4 and abs(y0[2 * 5000 + 1::2].mean()) < 1e-4
    imp = np.zeros(2 * 1000, np.float32); imp[2 * 10] = 1.0
    h = port.dc_blocker(imp, D, co.MA_CANONICAL)[0::2]
    assert np.argmax(h) == 10 + D - 1 and abs(h.sum()) < 1e-5            # delayed impulse minus a unit-area triangle
    a = port.run_iq(iq, rate, 7.0, True, co.MA_CANONICAL, use_dcblock=True).msgs
    b = port.run_iq(iq, rate, 7.0, True, co.MA_GR_FLOAT, 4096, use_dcblock=True).msgs
    assert [m.split()[:2] for m in a] == [m.split()[:2] for m in b] and len(a) > 0


def test_port_matches_reference_random_sweep(port, ref):
    """Seeded sweep over rates (integer and fractional samples/chip), thresholds, PMF on/off, burst density, garble and
    FRUIT: detection indices, 240-chip packets, timestamps, message text and the number of general_work calls of the
    port equal the unmodified reference's."""
    rng = np.random.default_rng(2024)
    rates = [2e6, 2.4e6, 2.5e6, 3e6, 3.2e6, 4e6, 5e6, 6e6, 8e6, 10e6, 12e6, 12.5e6, 16e6, 20e6]
    total = 0
    for k in range(28):
        rate = rates[k % len(rates)]
        thr = float(rng.choice([3.0, 4.5, 6.0, 7.0, 8.5, 10.0]))
        pmf = bool(rng.integers(0, 2))
        n = int(60_000 * rate / 2e6 / 2) + int(rng.integers(0, 999))
        nb = int(rng.choice([3, 12, 60]))
        sc = synth.make_scene(rate, n, nb, 7000 + k, garble_frac=0.3 if nb > 20 else 0.0, fruit=20 if nb > 20 else 0,
                              snr_db=(4.0, 28.0), df_choices=(0, 4, 5, 11, 16, 17, 20, 21, 24))
        bb, avg = port.frontend(sc.iq, rate, pmf, co.MA_CANONICAL)
        r = ref.run_streams(bb, avg, rate, thr)
        p = port.run_streams(bb, avg, rate, thr)
        where = (k, rate, thr, pmf, n, nb)
        assert np.array_equal(r.index, p.index), where
        assert np.array_equal(r.secs, p.secs) and np.array_equal(r.frac, p.frac), where
        assert r.chips_sha256 == chips_digest(p.chips), where
        assert r.msgs == p.msgs and r.calls == p.calls, where
        total += len(r.index)
    assert total > 300


def test_port_matches_reference_on_pathological_inputs(port, ref):
    """Same inputs tests/tools/stress_parity.py throws at the GPU: 1e-17 / 1e-21 / 3e14 amplitude scales (denormals, near
    overflow), NaN/Inf samples, silence, a DC offset, dense garbled traffic. (1500 such cases were run offline while
    building this; 80 here.)"""
    rng = np.random.default_rng(31337)
    tot = 0
    for case in range(80):
        rate = float(rng.choice([2e6, 2.4e6, 3e6, 4e6, 5e6, 8e6, 10e6, 16e6, 20e6, 4e6, 7e6]))
        pmf = bool(rng.random() < 0.8)
        thr = float(rng.choice([0.5, 3.0, 7.0, 7.0, 12.0, 20.0]))
        n, nb = int(rng.integers(12_000, 120_000)), int(rng.integers(0, 40))
        sigma = float(rng.choice([0.0, 1e-3, 0.01, 0.05]))
        kind = ["plain", "scale_small", "scale_big", "silence", "naninf", "dc", "dense", "denorm"][case % 8]
        sc = synth.make_scene(rate, n, nb * (10 if kind == "dense" else 1), int(rng.integers(1 << 30)), noise_sigma=sigma,
                              snr_db=(3.0, 40.0), garble_frac=0.2, fruit=int(rng.integers(0, 40)),
                              amplitude=None if sigma > 0 else 0.3, df_choices=(0, 4, 5, 11, 16, 17, 18, 20, 21, 24))
        iq = sc.iq.copy()
        if kind == "scale_small":
            iq *= np.float32(1e-17)
        elif kind == "denorm":
            iq *= np.float32(1e-21)
        elif kind == "scale_big":
            iq *= np.float32(3e14)
        elif kind == "silence":
            a = int(rng.integers(0, n))
            iq[2 * a: 2 * min(n, a + int(rng.integers(1, n)))] = 0
        elif kind == "naninf":
            for _ in range(3):
                iq[int(rng.integers(0, 2 * n))] = rng.choice([np.nan, np.inf, -np.inf, 3e38])
        elif kind == "dc":
            iq[0::2] += np.float32(0.02)
        with np.errstate(all="ignore"):
            bb, avg = port.frontend(iq, rate, pmf, co.MA_CANONICAL)
        r = ref.run_streams(bb, avg, rate, thr)
        p = port.run_streams(bb, avg, rate, thr)
        where = (case, kind, rate, pmf, thr, n)
        assert np.array_equal(r.index, p.index) and r.msgs == p.msgs and r.calls == p.calls, where
        assert r.chips_sha256 == chips_digest(p.chips), where
        tot += len(r.index)
    assert tot > 500

"""The hot path's sparse kernels WITH their launchers (gr_air_modes_b200/csrc/amb_kernels.cu minus the TMA scan kernel:
candidate bitmap from float streams, compaction, exact preamble tests, sequential and parallel resolver, slicer, CRC)
executed on the host by the SIMT emulator of tests/simt and compared with the oracle - the same comparison the GPU
tests make through amb_preamble_process / amb_slicer_process / amb_device_crc, here without a GPU. Catches
hardware-independent bugs in the warp-level logic and in the launch configuration; the GPU tests remain the gate."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from gr_air_modes_b200 import synth
from oracle import cpu_oracle as co

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("ksimt") / "libkernels_emul.so")
    subprocess.run(["g++", "-std=c++17", "-O1", "-U_FORTIFY_SOURCE", "-ffp-contract=off", "-Wno-unknown-pragmas", "-Wno-psabi", "-shared", "-fPIC",
                    "-Wl,-Bsymbolic", "-o", out, os.path.join(ROOT, "tests", "simt", "kernels_emul.cc")], check=True)   # see test_library_simt.py
    lib = C.CDLL(out)
    lib.emul_preamble.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int, C.c_void_p,
                                  C.c_void_p, C.c_int, C.c_void_p]
    lib.emul_process_iq.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_int, C.c_int, C.c_int,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    lib.emul_counts.argtypes = [C.c_void_p]
    lib.emul_dcblock.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.emul_slicer.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    lib.emul_crc.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_void_p]
    return lib


def _preamble(lib, bb, avg, rate, thr, resolver):
    n = bb.size
    max_det = n // 200 + 16
    chips = np.zeros((max_det, 240), np.float32)
    idx = np.zeros(max_det, np.uint64)
    stats = np.zeros(3, np.uint32)
    nd = lib.emul_preamble(bb.ctypes.data, avg.ctypes.data, n, rate, thr, resolver, 2, chips.ctypes.data, idx.ctypes.data,
                           max_det, stats.ctypes.data)
    assert nd >= 0, nd
    return idx[:nd], chips[:nd], stats


@pytest.mark.parametrize("rate,n,nb,pmf,thr,seed", [
    (4e6, 60_000, 12, True, 7.0, 1), (2e6, 40_000, 10, True, 7.0, 2), (10e6, 120_000, 8, True, 7.0, 3),
    (20e6, 200_000, 6, True, 7.0, 4), (5e6, 60_000, 8, True, 6.0, 5), (4e6, 60_000, 120, False, 5.0, 6),
])
def test_split_form_chain_under_the_emulator_matches_the_oracle(emul, port, rate, n, nb, pmf, thr, seed):
    dense = nb > 50
    sc = synth.make_scene(rate, n, nb, 900 + seed, garble_frac=0.3 if dense else 0.0, fruit=30 if dense else 0,
                          df_choices=(0, 4, 5, 11, 16, 17, 20, 21))
    bb, avg = port.frontend(sc.iq, rate, pmf, co.MA_CANONICAL)
    want = port.run_streams(bb, avg, rate, thr)
    assert len(want.index) >= (20 if dense else 5)
    for resolver in (1, 2):                                  # sequential walk, parallel walk (cluster walk + buckets)
        idx, chips, stats = _preamble(emul, bb, avg, rate, thr, resolver)
        assert [int(x) for x in idx] == [int(x) for x in want.index], (resolver, stats)
        assert np.array_equal(chips, np.asarray(want.chips, np.float32).reshape(-1, 240)), resolver
        assert stats[1] <= stats[0] and stats[1] >= len(want.index)


@pytest.mark.parametrize("rate,n,nb,pmf,thr,seed", [
    (4e6, 60_001, 12, True, 7.0, 1), (2e6, 30_000, 10, False, 6.0, 2), (10e6, 120_777, 8, True, 7.0, 3),
    (20e6, 200_300, 6, True, 7.0, 4), (5e6, 70_000, 8, True, 7.0, 5), (2.4e6, 40_000, 8, True, 6.0, 6),
    (4e6, 50_000, 100, True, 5.0, 7),
])
def test_fused_iq_chain_under_the_emulator_matches_the_oracle(emul, port, rate, n, nb, pmf, thr, seed):
    """amb_process's kernels on IQ, all of them: the streaming scan kernel (its seven PTX helpers - mbarrier, 2-D TMA tile
    copy - are emulated, the kernel source is the product's), prologue (tail staging), compaction, the exact and slice
    kernels in their IQ form (canonical |x|^2 / PMF / noise-floor arithmetic from the carry ++ main ++ tail segments),
    both resolvers. Detection indices, 240-chip packets and the message text equal the oracle's run over the same IQ;
    the scan kernel's candidates are a superset of the exact ones."""
    from gr_air_modes_b200 import _lib, blocks
    dense = nb > 50
    sc = synth.make_scene(rate, n, nb, 700 + seed, garble_frac=0.3 if dense else 0.0, fruit=30 if dense else 0)
    bb, avg = port.frontend(sc.iq, rate, pmf, co.MA_CANONICAL)
    want = port.run_iq(sc.iq, rate, thr, pmf, co.MA_CANONICAL)
    assert len(want.index) >= (2 if rate == 2.4e6 else 5)
    md = n // 200 + 16
    # (resolver, bitmap source): the REAL scan kernel (TMA tile copies with the 128-byte swizzle and mbarriers emulated,
    # kernel source unchanged) with the parallel resolver, and the stream-candidate stand-in with both resolvers
    for resolver, use_scan in ((2, True), (1, False), (2, False)):
        # the exact stage has two kernels: rows + one lane per candidate (dense traffic; the harness default) and one
        # warp per candidate (sparse traffic); the middle pass runs the latter
        if resolver == 1:
            os.environ["AMB_TEST_EXACT_DENSE"] = "1000000000"
        else:
            os.environ.pop("AMB_TEST_EXACT_DENSE", None)
        chips = np.zeros((md, 240), np.float32)
        idx = np.zeros(md, np.uint64)
        frames = (_lib.Frame * md)()
        nd = emul.emul_process_iq(sc.iq.ctypes.data, n, None if use_scan else bb.ctypes.data, None if use_scan else avg.ctypes.data,
                                  rate, thr, int(pmf), resolver, 2, chips.ctypes.data, idx.ctypes.data, C.cast(frames, C.c_void_p), md)
        assert nd >= 0, nd
        cnt = np.zeros(3, np.uint32)
        emul.emul_counts(cnt.ctypes.data)
        if use_scan:
            scan_cand, scan_real = int(cnt[0]), int(cnt[1])
        else:                                                # the scan kernel's conservative filter: a superset, nothing real lost
            assert scan_real == int(cnt[1]) and scan_cand >= int(cnt[0]) == int(cnt[1])
        assert [int(x) for x in idx[:nd]] == [int(x) for x in want.index], resolver
        assert np.array_equal(chips[:nd], want.chips), resolver
        ri, msgs, first = int(rate), [], True
        for k in range(nd):                                  # stamp as amb_poll_frames does (tag_to_timestamp, no rx_time tag)
            frames[k].secs, frames[k].frac = int(idx[k]) // ri, (int(idx[k]) % ri) / float(ri)
            if frames[k].passed:
                msgs.append(blocks.format_message(frames[k], first))
                first = False
        assert msgs == want.msgs, resolver


def test_end_of_stream_and_empty_streams_under_the_emulator(emul, port):
    rate = 4e6
    for cut in (0, 111, 333, 640):
        sc = synth.make_scene(rate, 30_000, 0, 11, starts=[9_000.3, 29_200.0 - cut], amplitude=0.3)
        bb, avg = port.frontend(sc.iq, rate, True, co.MA_CANONICAL)
        want = port.run_streams(bb, avg, rate, 7.0)
        idx, chips, _ = _preamble(emul, bb, avg, rate, 7.0, 2)
        assert [int(x) for x in idx] == [int(x) for x in want.index], cut
    z = np.zeros(3000, np.float32)
    idx, _, _ = _preamble(emul, z, z, rate, 7.0, 2)
    assert idx.size == 0


def test_slicer_and_crc_kernels_under_the_emulator(emul, port):
    from gr_air_modes_b200 import _lib, blocks
    rng = np.random.default_rng(5)
    n = 200
    chips = rng.normal(0.0, 0.3, (n, 240)).astype(np.float32)
    chips[:, [0, 2, 7, 9]] += 1.0
    chips[::3, 16:240:2] += 1.0
    secs = np.arange(n, dtype=np.uint64)
    frac = rng.random(n)
    want = port.run_slicer(chips, secs, frac).msgs
    frames = (_lib.Frame * n)()
    assert emul.emul_slicer(chips.ctypes.data, n, C.cast(frames, C.c_void_p)) == 0
    got, first = [], True
    for k in range(n):
        frames[k].secs, frames[k].frac = int(secs[k]), float(frac[k])
        if frames[k].passed:
            got.append(blocks.format_message(frames[k], first))
            first = False
    assert got == want and len(want) > 0
    for length in (4, 11):
        data = rng.integers(0, 256, (64, length), dtype=np.uint8)
        out = np.zeros(64, np.uint32)
        assert emul.emul_crc(data.tobytes(), 64, length, out.ctypes.data) == 0
        assert [int(x) for x in out] == [port.crc24(bytes(r)) for r in data]


def test_scan_kernel_under_the_emulator_on_pathological_inputs(emul, port):
    """The scan kernel is a conservative fp32 FILTER (FMA |x|^2, prefix-sum windows, lowered thresholds); whatever it
    is fed - 1e-17 / 1e-21 / 3e14 amplitude scales, NaN/Inf samples, silence, a DC offset, dense garble - the chain's
    result must still be the oracle's."""
    from gr_air_modes_b200 import _lib
    rng = np.random.default_rng(4242)
    kinds = ["scale_small", "denorm", "scale_big", "silence", "naninf", "dc", "dense", "zeros"]
    for case, kind in enumerate(kinds):
        rate = [4e6, 2e6, 10e6, 4e6, 5e6, 20e6, 4e6, 4e6][case]
        pmf = case % 3 != 1
        n = int(rng.integers(20_000, 50_000)) * (2 if rate >= 10e6 else 1)
        sc = synth.make_scene(rate, n, 150 if kind == "dense" else 10, 5000 + case, garble_frac=0.3 if kind == "dense" else 0.0,
                              snr_db=(6.0, 35.0), fruit=20 if kind == "dense" else 0)
        iq = sc.iq.copy()
        if kind == "scale_small":
            iq *= np.float32(1e-17)
        elif kind == "denorm":
            iq *= np.float32(1e-21)
        elif kind == "scale_big":
            iq *= np.float32(3e14)
        elif kind == "silence":
            a = int(rng.integers(0, n))
            iq[2 * a: 2 * min(n, a + n // 3)] = 0
        elif kind == "naninf":
            for v in (np.nan, np.inf, -np.inf, 3e38):
                iq[int(rng.integers(0, 2 * n))] = v
        elif kind == "dc":
            iq[0::2] += np.float32(0.02)
        elif kind == "zeros":
            iq[:] = 0
        with np.errstate(all="ignore"):
            want = port.run_iq(iq, rate, 7.0, pmf, co.MA_CANONICAL)
        md = n // 200 + 16
        chips = np.zeros((md, 240), np.float32)
        idx = np.zeros(md, np.uint64)
        frames = (_lib.Frame * md)()
        nd = emul.emul_process_iq(iq.ctypes.data, n, None, None, rate, 7.0, int(pmf), 2, 2, chips.ctypes.data, idx.ctypes.data,
                                  C.cast(frames, C.c_void_p), md)
        assert nd >= 0, (kind, nd)
        assert [int(x) for x in idx[:nd]] == [int(x) for x in want.index], kind
        assert np.array_equal(chips[:nd], want.chips, equal_nan=True), kind


def test_dc_blocker_kernels_under_the_emulator(emul, port):
    """amb_dcblock_kernel (one pass: raw tile -> MA -> MA -> output; exact fp64 prefix sums per tile, literal sums where
    the exponent spread forbids them; 1024-output tiles up to D = 256, 2048 beyond): output bit-identical to the CPU
    restatement, on ordinary samples and on tiles that force the literal path in the first or the second average."""
    rng = np.random.default_rng(9)
    for D, n, kind in ((200, 5000, "plain"), (500, 6000, "plain"), (1000, 7000, "plain"), (200, 4000, "spread"),
                       (500, 5000, "spread"), (200, 3000, "naninf")):
        iq = (rng.standard_normal(2 * n) * 0.01).astype(np.float32)
        iq[0::2] += np.float32(0.05)
        if kind == "spread":
            iq[2 * 1500: 2 * 1600] *= np.float32(1e12)          # > 18 binades inside one tile: literal sums
        if kind == "naninf":
            iq[777], iq[2222] = np.nan, np.inf
        with np.errstate(all="ignore"):
            want = port.dc_blocker(iq, D, co.MA_CANONICAL)
        got = np.zeros(2 * n, np.float32)
        assert emul.emul_dcblock(iq.ctypes.data, n, D, got.ctypes.data) == 0
        assert np.array_equal(got, want, equal_nan=True), (D, n, kind)


def test_random_thread_interleavings(emul, port):
    """The emulator normally resumes the threads of a block in index order; with a shuffle seed every scheduling round
    uses another order. A kernel that only works because of an accidental execution order (a missing barrier) stops
    getting away with it. Whole IQ chain incl. the scan kernel, three seeds."""
    from gr_air_modes_b200 import _lib
    emul.simt_set_shuffle.argtypes = [C.c_ulonglong]
    rate, n = 4e6, 50_000
    sc = synth.make_scene(rate, n, 100, 31, garble_frac=0.3, fruit=30)
    want = port.run_iq(sc.iq, rate, 6.0, True, co.MA_CANONICAL)
    md = n // 200 + 16
    try:
        for seed in (1, 2, 3):
            emul.simt_set_shuffle(seed)
            chips = np.zeros((md, 240), np.float32)
            idx = np.zeros(md, np.uint64)
            frames = (_lib.Frame * md)()
            nd = emul.emul_process_iq(sc.iq.ctypes.data, n, None, None, rate, 6.0, 1, 2, 2, chips.ctypes.data, idx.ctypes.data,
                                      C.cast(frames, C.c_void_p), md)
            assert nd == len(want.index) and [int(x) for x in idx[:nd]] == [int(x) for x in want.index], seed
            assert np.array_equal(chips[:nd], want.chips), seed
    finally:
        emul.simt_set_shuffle(0)

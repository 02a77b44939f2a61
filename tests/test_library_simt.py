"""The WHOLE library on the CPU box: tests/simt/library_emul.cc compiles the library's own three translation units
(kernels, host orchestration + C ABI, decoder) against the SIMT emulator and CUDA-runtime stand-ins of tests/simt, and
this module drives that build through the ordinary Python package - the same scenarios the GPU parity tests run,
scaled down: streaming vs one-shot, end-of-stream rules, setters and the state machine, a recording time-sharded over
several contexts (hand-over chain and speculative resolution), the split-form blocks, the DC blocker option, the
front-end dumps, two contexts side by side, and the batch decoder through its C ABI.

TEST INFRASTRUCTURE ONLY: the emulated build exists in a pytest temp directory for the duration of this module; the
package itself only ever binds gr_air_modes_b200/libairmodes_b200.so and has no CPU path (tests/test_host_logic.py).
It is not thread-safe (one emulated device, global fiber state): everything here is sequential.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import gr_air_modes_b200 as am
from gr_air_modes_b200 import _lib, synth
from oracle import cpu_oracle as co

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module", autouse=True)
def emulated_library(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("libsimt") / "libairmodes_b200_emulated.so")
    # -Bsymbolic: the library's calls into its own C ABI (amb_create -> amb_destroy, ...) must stay inside the emulated
    # build even when the real libairmodes_b200.so was loaded RTLD_GLOBAL into this process by an earlier test
    subprocess.run(["g++", "-std=c++17", "-O1", "-U_FORTIFY_SOURCE", "-ffp-contract=off", "-Wno-unknown-pragmas", "-Wno-psabi", "-shared", "-fPIC",
                    "-Wl,-Bsymbolic", "-o", out, os.path.join(ROOT, "tests", "simt", "library_emul.cc")], check=True)
    saved = (_lib.LIB_PATH, _lib._lib)
    _lib.LIB_PATH, _lib._lib = out, None
    try:
        yield out
    finally:
        _lib.LIB_PATH, _lib._lib = saved


def run(iq, rate, thr, pmf, chunks=None, resolver=0, dcblock=False, exact_dense=None):
    q = am.msg_queue()
    rx = am.rx_path(rate, thr, q, use_pmf=pmf, use_dcblock=dcblock)
    rx._ctx.call("amb_set_option", b"resolver", resolver)
    if exact_dense is not None:        # 0: every call is decided by the row-based exact kernel (dense-traffic regime)
        rx.set_option("exact_dense", exact_dense)
    frames, pos, n = [], 0, iq.size // 2
    for c in (chunks or []) + [n]:
        c = int(min(c, n - pos))
        last = pos + c >= n
        rx.process(iq[2 * pos: 2 * (pos + c)], flush=last)
        frames += rx.frames
        pos += c
        if last:
            break
    st = rx.stats()
    rx.close()
    return q.strings(), frames, st


@pytest.mark.parametrize("rate,n,nb,pmf,thr", [(4e6, 50_000, 12, True, 7.0), (2e6, 30_000, 10, False, 6.0), (10e6, 90_000, 8, True, 7.0),
                                               (20e6, 150_000, 6, True, 7.0), (5e6, 50_000, 8, True, 7.0)])
def test_streaming_equals_one_shot_equals_oracle(port, rate, n, nb, pmf, thr):
    sc = synth.make_scene(rate, n, nb, int(rate / 1e6) + 300)
    want = port.run_iq(sc.iq, rate, thr, pmf, co.MA_CANONICAL)
    assert len(want.msgs) >= 2
    msgs, frames, st = run(sc.iq, rate, thr, pmf)
    assert msgs == want.msgs and [f.sample_index for f in frames] == [int(x) for x in want.index]
    assert st.kernel_launches >= 6 and st.samples_in == n
    rng = np.random.default_rng(1)
    for resolver in (0, 1):
        chunks = [int(x) for x in rng.integers(1, n // 3, 3)] + [1, 511, 513]
        msgs2, frames2, _ = run(sc.iq, rate, thr, pmf, chunks=chunks, resolver=resolver, exact_dense=0 if resolver else None)
        assert msgs2 == want.msgs and [f.sample_index for f in frames2] == [int(x) for x in want.index], resolver
    for f, g in zip(frames, want.frames):
        assert bytes(f.data) == bytes(g.data) and f.ref_level == g.ref_level and f.crc == g.crc and f.numlowconf == g.numlowconf


def test_end_of_stream_rules_and_tiny_inputs(port):
    rate = 4e6
    for cut in (0, 150, 333, 480, 640):
        sc = synth.make_scene(rate, 30_000, 0, 11, starts=[9_000.3, 29_200.0 - cut], amplitude=0.3)
        want = port.run_iq(sc.iq, rate, 7.0, True, co.MA_CANONICAL)
        msgs, frames, _ = run(sc.iq, rate, 7.0, True)
        assert msgs == want.msgs and [f.sample_index for f in frames] == [int(x) for x in want.index], cut
    for n in (0, 1, 3, 17, 239, 481, 2000):
        msgs, frames, _ = run(np.zeros(2 * n, np.float32), rate, 7.0, True)
        assert msgs == [] and frames == []


def test_setters_errors_and_state_machine(port):
    q = am.msg_queue()
    rx = am.rx_path(4e6, 7.0, q, use_pmf=True)
    assert rx.get_threshold() == 7.0 and rx.get_pmf() is True
    with pytest.raises(RuntimeError):
        rx.set_rate(1e6)                                    # below 2 Msps: preamble_impl would divide by zero (:150)
    with pytest.raises(RuntimeError):
        am.rx_path(30e6, 7.0, q)
    rx.process(np.zeros(2000, np.float32), flush=True)
    with pytest.raises(RuntimeError):
        rx.process(np.zeros(2000, np.float32))              # flushed stream needs reset()
    rx.reset()
    sc = synth.make_scene(4e6, 40_000, 10, 77)
    lo = port.run_iq(sc.iq, 4e6, 4.0, True, co.MA_CANONICAL).msgs
    hi = port.run_iq(sc.iq, 4e6, 12.0, True, co.MA_CANONICAL).msgs
    rx.set_threshold(4.0)
    rx.process(sc.iq, flush=True)
    assert q.strings() == lo
    q.flush(); rx.reset(); rx._slicer._first = True
    rx.set_threshold(12.0)
    rx.process(sc.iq, flush=True)
    assert q.strings() == hi and hi != lo
    rx.set_rate(10e6)                                       # re-tune (rx_path.py:67-72): a new stream at the new rate
    sc10 = synth.make_scene(10e6, 80_000, 8, 78)
    q.flush(); rx._slicer._first = True
    rx.set_threshold(7.0)
    rx.process(sc10.iq, flush=True)
    assert q.strings() == port.run_iq(sc10.iq, 10e6, 7.0, True, co.MA_CANONICAL).msgs
    rx.close()


def test_rx_time_start_tag(port):
    sc = synth.make_scene(4e6, 40_000, 10, 3)
    q = am.msg_queue()
    rx = am.rx_path(4e6, 7.0, q, use_pmf=True)
    rx.set_start_time(1234567, 0.9999999)
    rx.process(sc.iq, flush=True)
    port.set_start_time(1234567, 0.9999999)
    try:
        want = port.run_iq(sc.iq, 4e6, 7.0, True, co.MA_CANONICAL).msgs
    finally:
        port.set_start_time(0, 0.0)
    assert q.strings() == want
    rx.close()


def _time_sharded_chain(iq, rate, thr, pmf, plan, resolver=0):
    q = am.msg_queue()
    rxs = [am.rx_path(rate, thr, q, use_pmf=pmf) for _ in plan]
    for rx, sp in zip(rxs, plan):
        rx._ctx.call("amb_set_option", b"resolver", resolver)
        rx.defer_resolve(True)
        rx.seek(sp.first_sample, sp.first_decision)
        rx.process(iq[2 * sp.first_sample: 2 * sp.end], flush=sp.flush, collect=False)
    frames, state, queued = [], (0, 0), 0
    for rx, sp in zip(rxs, plan):
        rx.resolve(state)
        if not sp.flush:
            state = rx.walk_state()
        rx._slicer._first = queued == 0
        queued += rx.drain()
        frames += rx.frames
    for rx in rxs:
        rx.close()
    return q.strings(), frames


def _time_sharded_speculative(iq, rate, thr, pmf, plan):
    """shard.process_time_sharded_speculative for every rank, sequentially (the emulated device is not thread-safe)."""
    from gr_air_modes_b200 import shard
    qs = [am.msg_queue() for _ in plan]
    rxs = [am.rx_path(rate, thr, q, use_pmf=pmf) for q in qs]
    last = len(plan) - 1
    mines = []
    for rank, (rx, sp) in enumerate(zip(rxs, plan)):
        rx.defer_resolve(True)
        rx.seek(sp.first_sample, sp.first_decision)
        rx.process(iq[2 * sp.first_sample: 2 * sp.end], flush=sp.flush, collect=False)
        mine = [0] * 6
        if rank < last:
            rx.resolve(None)
            s = rx.walk_summary()
            mine = [s.pos, s.p, s.first_real, s.first_packet, s.exact_span, s.frames_passed]
        mines.append(mine)
    entries, queued, bad = shard.compose_entries(plan, mines)
    frames, handed = [], None
    for rank, (rx, sp) in enumerate(zip(rxs, plan)):
        if rank < bad:
            qd = queued[rank]
        else:
            if rank == bad:
                (pos, p), qd = entries[rank], queued[rank]
            else:
                pos, p, qd = handed
            rx.resolve((pos, p))
        rx._slicer._first = qd == 0
        if rank >= bad and not sp.flush:
            state = rx.walk_state()
            n = rx.drain()
            handed = state + (qd + n,)
        else:
            rx.drain()
        frames += rx.frames
        rx.close()
    return [m for q in qs for m in q.strings()], frames, bad


def test_one_recording_time_sharded_over_several_contexts(port):
    from gr_air_modes_b200 import shard
    rate, n = 4e6, 120_000
    sc = synth.make_scene(rate, n, 45, 74)
    want = port.run_iq(sc.iq, rate, 7.0, True, co.MA_CANONICAL)
    idx = [int(x) for x in want.index]
    geo = am.query_geometry(rate, 7.0, True)
    for spans in (2, 3):
        plan = shard.time_shard_plan(n, spans, geo)
        for resolver in ((0, 1) if spans == 2 else (0,)):
            msgs, frames = _time_sharded_chain(sc.iq, rate, 7.0, True, plan, resolver)
            assert [f.sample_index for f in frames] == idx and msgs == want.msgs, (spans, resolver)
        msgs, frames, bad = _time_sharded_speculative(sc.iq, rate, 7.0, True, plan)
        assert bad == spans - 1 and [f.sample_index for f in frames] == idx and msgs == want.msgs
    # cuts right behind accepted preambles: the hand-over matters, speculation must fall back to the chain
    mid = [x for x in idx if 30_000 < x < 105_000]
    fell_back = 0
    for a, b, d in ((2, 9, 3), (1, 11, 1)):
        cuts = [mid[a] + d, mid[b] + d + 1]
        plan = shard.time_shard_plan(n, 3, geo, boundaries=cuts)
        msgs, frames = _time_sharded_chain(sc.iq, rate, 7.0, True, plan)
        assert [f.sample_index for f in frames] == idx and msgs == want.msgs, cuts
        msgs, frames, bad = _time_sharded_speculative(sc.iq, rate, 7.0, True, plan)
        fell_back += bad < 2
        assert [f.sample_index for f in frames] == idx and msgs == want.msgs, cuts
    assert fell_back > 0


def test_time_shard_api_errors():
    q = am.msg_queue()
    rx = am.rx_path(4e6, 7.0, q, use_pmf=True)
    g = am.query_geometry(4e6, 7.0, True)
    with pytest.raises(RuntimeError):
        rx.seek(4096, 4096 + g.shard_back - 1)
    with pytest.raises(RuntimeError):
        rx.resolve((0, 0))
    rx.defer_resolve(True)
    rx.seek(0, 0)
    iq = synth.make_scene(4e6, 30_000, 5, 3).iq
    rx.process(iq, flush=False, collect=False)
    with pytest.raises(RuntimeError):
        rx.process(iq, flush=False, collect=False)
    with pytest.raises(RuntimeError):
        rx.walk_state()
    rx.resolve((0, 0))
    rx.walk_state()
    rx.defer_resolve(False)
    rx.reset()
    assert rx.process(iq, flush=True) >= 4
    rx.close()


def test_split_form_blocks(port):
    rng = np.random.default_rng(3)
    for rate in (4e6, 10e6):
        sc = synth.make_scene(rate, 60_000, 12, 56)
        bb, avg = port.frontend(sc.iq, rate, True, co.MA_CANONICAL)
        want = port.run_streams(bb, avg, rate, 7.0)
        pre = am.preamble(rate, 7.0)
        assert pre.get_rate() == rate and pre.get_threshold() == 7.0
        chips, tags, pos, n = [], [], 0, bb.size
        for c in list(rng.integers(1, 25_000, 5)) + [n]:
            c = int(min(c, n - pos))
            last = pos + c >= n
            ch, tg = pre.process(bb[pos:pos + c], avg[pos:pos + c], flush=last)
            chips.append(ch)
            tags += tg
            pos += c
            if last:
                break
        assert [t[0] for t in tags] == [int(x) for x in want.index]
        assert np.array_equal(np.concatenate(chips), want.chips)
        q = am.msg_queue()
        am.slicer(q).process(np.concatenate(chips), [(t[1], t[2]) for t in tags])
        assert q.strings() == want.msgs


def test_dc_blocker_option_and_front_end_dumps(port):
    rate = 4e6
    sc = synth.make_scene(rate, 40_000, 12, 5)
    iq = sc.iq.copy()
    iq[0::2] += np.float32(0.05)
    want = port.run_iq(iq, rate, 7.0, True, co.MA_CANONICAL, use_dcblock=True)
    msgs, frames, _ = run(iq, rate, 7.0, True, chunks=[9_000, 7, 12_000], dcblock=True)
    assert msgs == want.msgs and len(msgs) >= 1            # the 50 us blocker distorts 120 us bursts, as in the reference
    q = am.msg_queue()
    rx = am.rx_path(rate, 7.0, q, use_pmf=True, use_dcblock=True)
    small = iq[: 2 * 6000]
    assert np.array_equal(rx.dump_stage("dc", small), port.dc_blocker(small, 200, co.MA_CANONICAL))
    rx.close()
    for r, pmf in ((4e6, True), (10e6, True), (2e6, False)):
        rx = am.rx_path(r, 7.0, q, use_pmf=pmf)
        x = synth.make_scene(r, 5000, 2, 9).iq
        bb, avg = port.frontend(x, r, pmf, co.MA_CANONICAL)
        assert np.array_equal(rx.dump_stage("bb", x), bb) and np.array_equal(rx.dump_stage("avg", x), avg)
        rx.close()


def test_two_contexts_and_device_crc(port):
    import ctypes as C
    a, b = synth.make_scene(4e6, 40_000, 10, 1), synth.make_scene(10e6, 80_000, 8, 2)
    qa, qb = am.msg_queue(), am.msg_queue()
    ra, rb = am.rx_path(4e6, 7.0, qa, use_pmf=True), am.rx_path(10e6, 7.0, qb, use_pmf=True)
    ra.process(a.iq[: 2 * 20_000]); rb.process(b.iq[: 2 * 30_000])
    ra.process(a.iq[2 * 20_000:], flush=True); rb.process(b.iq[2 * 30_000:], flush=True)
    assert qa.strings() == port.run_iq(a.iq, 4e6, 7.0, True, co.MA_CANONICAL).msgs
    assert qb.strings() == port.run_iq(b.iq, 10e6, 7.0, True, co.MA_CANONICAL).msgs
    out = (C.c_uint32 * 1)()
    ra._ctx.call("amb_device_crc", bytes.fromhex("8D4840D6202CC371C32CE0"), 1, 11, out)
    assert out[0] == 0x576098
    ra.close(); rb.close()


def test_decoder_does_not_pair_with_reports_of_an_earlier_stream():
    """A persistent decoder, a new recording whose timestamps restart at 0: a stored report that is LATER than the
    current message belongs to the earlier stream and must count as expired (the reference's wall clock would have
    weeded it long ago, cpr.py:196-204) instead of producing a position out of two unrelated reports."""
    from gr_air_modes_b200 import decode
    even, odd = "8d40621d58c382d690c8ac2863a7", "8d40621d58c386435cc412692ad6"
    d = decode.batch_decoder(None)
    a = d.decode_messages([(even, 0, 100, 0.0), (odd, 0, 101, 0.0)])
    assert (a["status"][0] & decode.FS_CPR_NO_POS) and (a["status"][1] & decode.FS_HAS_POS)
    assert abs(a["lat"][1] - 52.26) < 0.02 and abs(a["lon"][1] - 3.93) < 0.03         # the textbook pair (odd frame latest)
    b = d.decode_messages([(odd, 0, 1, 0.0)])                 # new stream: t restarts; the even report of t = 100 is "later"
    assert (b["status"][0] & decode.FS_CPR_NO_POS) and not (b["status"][0] & decode.FS_HAS_POS)
    c = d.decode_messages([(even, 0, 2, 0.0)])                # ... and pairs normally within the new stream
    assert c["status"][0] & decode.FS_HAS_POS
    d.close()


def test_decoder_through_its_c_abi():
    from gr_air_modes_b200 import decode, report
    from helpers import compare_decode, load_decode_golden
    import decode_cases
    case = load_decode_golden()[0]
    msgs = [tuple(m) for m in case["msgs"]][:600]
    d = decode.batch_decoder(case["location"])
    one = [decode.record_to_dict(r) for r in d.decode_messages(msgs)]
    assert d.stats()[0] == 7          # fields + the five bucket-partition pairing kernels + resolve
    texts = decode_cases.message_strings([tuple(m) for m in case["msgs"]])[:600]
    for k, (rec, ref) in enumerate(zip(one, case["ref"])):
        compare_decode(rec, ref, 0.0, "msg %d" % k, tol_libm=1e-13)
        assert report.format_report(texts[k], rec) == case["lines"][k]
    d.reset()
    got = []
    for a, b in ((0, 1), (1, 33), (33, 400), (400, 600)):          # the report table carries over from batch to batch
        got += [decode.record_to_dict(r) for r in d.decode_messages(msgs[a:b])]
    assert [g["status"] for g in got] == [o["status"] for o in one]
    assert all(g["lat"] == o["lat"] or (g["lat"] != g["lat"] and o["lat"] != o["lat"]) for g, o in zip(got, one))
    d.close()


def test_graft_entry_smoke_rehearsal(capsys):
    """__graft_entry__.smoke() - what the driver runs on the B200 before the bench - against the emulated build."""
    sys.path.insert(0, ROOT)
    import __graft_entry__ as entry
    entry.smoke()
    assert "smoke ok" in capsys.readouterr().out


def test_candidate_flood_does_not_overflow(port):
    """Input whose |x|^2 is denormal: the scan kernel's filter (absolute 1e-42 slack) passes every non-zero sample,
    more than n / 8 candidates. Calls of up to 2^25 samples size the candidate list for every position, so the exact
    stage simply weeds them out and the result is still the oracle's (found by fuzzing the emulated chain)."""
    rate, n = 2.5e6, 60_000
    sc = synth.make_scene(rate, n, 30, 1234, noise_sigma=0.05, snr_db=(3.0, 40.0))
    iq = sc.iq * np.float32(1e-21)
    want = port.run_iq(iq, rate, 0.5, True, co.MA_CANONICAL)
    q = am.msg_queue()
    rx = am.rx_path(rate, 0.5, q, use_pmf=True)
    rx.process(iq, flush=True)
    st = rx.stats()
    assert st.candidates > n // 8                         # the flood is real ...
    assert q.strings() == want.msgs and len(want.msgs) > 20   # ... and harmless
    rx.close()


# ---- host ingest pipeline (amb_process with host memory): chunk ring, gathering of small calls, 16-bit IQ, polls ----
def test_ingest_ring_small_calls_and_nonblocking_poll(port):
    """GNU Radio-sized calls are gathered in the ring's pinned buffer and dispatched every `coalesce` samples; a tiny
    chunk size forces many ring wrap-arounds. Results = one shot = oracle, whichever way they are collected."""
    rate = 4e6
    sc = synth.make_scene(rate, 120_000, 24, 901)
    want = port.run_iq(sc.iq, rate, 7.0, True, co.MA_CANONICAL)
    assert len(want.msgs) >= 10
    for chunk, coalesce, call in ((4096, 1024, 700), (8192, 8192, 3001), (1 << 22, 1 << 18, 8192)):
        q = am.msg_queue()
        rx = am.rx_path(rate, 7.0, q, use_pmf=True)
        rx.set_option("ingest_chunk", chunk)
        rx.set_option("coalesce", coalesce)
        n, pos, early = sc.iq.size // 2, 0, 0
        while pos < n:
            c = min(call, n - pos)
            rx.process(sc.iq[2 * pos: 2 * (pos + c)], flush=False, collect=False)
            early += rx.poll_ready()                       # non-blocking: whatever has completed
            pos += c
        rx.process(sc.iq[:0], flush=True, collect=True)    # closes the stream, forces the rest out
        assert q.strings() == want.msgs, (chunk, coalesce, call)
        assert rx.stats().samples_in == n
        if coalesce < 100_000:
            assert early > 0                               # messages did arrive through the non-blocking poll
        rx.close()


def test_ingest_large_pageable_call_is_cut_into_chunks(port):
    rate = 10e6
    sc = synth.make_scene(rate, 200_000, 16, 902)
    want = port.run_iq(sc.iq, rate, 7.0, True, co.MA_CANONICAL)
    q = am.msg_queue()
    rx = am.rx_path(rate, 7.0, q, use_pmf=True)
    rx.set_option("ingest_chunk", 16384)                   # 13 chunks, ring of 4
    rx.process(sc.iq, flush=True)
    assert q.strings() == want.msgs and [f.sample_index for f in rx.frames] == [int(x) for x in want.index]
    # and again on the same context after a reset, now complex64 and in two uneven calls
    q.flush(); rx.reset(); rx._slicer._first = True
    c = sc.iq.view(np.complex64)
    rx.process(c[:77_777], collect=False)
    rx.process(c[77_777:], flush=True)
    assert q.strings() == want.msgs
    rx.close()


def test_sc16_input_equals_its_float32_widening(port):
    """16-bit IQ is widened on the device with x * 2^-15: identical to feeding the float32 a host-side conversion
    (radio.py:163-173, cpu_format fc32) would have produced - every message, bit for bit."""
    rate = 4e6
    sc = synth.make_scene(rate, 100_000, 20, 903, noise_sigma=0.01)
    i16 = np.clip(np.rint(sc.iq * 32768.0), -32768, 32767).astype(np.int16)
    f32 = i16.astype(np.float32) * np.float32(1.0 / 32768.0)
    want = port.run_iq(f32, rate, 7.0, True, co.MA_CANONICAL)
    assert len(want.msgs) >= 8
    for chunk in (8192, 1 << 22):
        q = am.msg_queue()
        rx = am.rx_path(rate, 7.0, q, use_pmf=True)
        rx.set_option("ingest_chunk", chunk)
        rx.process(i16[:60_002], collect=False)
        rx.process(i16[60_002:], flush=True)
        assert q.strings() == want.msgs, chunk
        rx.close()
    with pytest.raises(TypeError):
        am.rx_path(rate, 7.0, am.msg_queue()).process(np.zeros(64, np.float64))
    q = am.msg_queue()
    rx = am.rx_path(rate, 7.0, q, use_pmf=True)
    rx.process(f32.view(np.complex64).astype(np.complex128), flush=True)   # complex128 is narrowed, not reinterpreted
    assert q.strings() == want.msgs


def test_mid_stream_rx_time_tag(port):
    rate = 4e6
    sc = synth.make_scene(rate, 80_000, 16, 904)
    plain = port.run_iq(sc.iq, rate, 7.0, True, co.MA_CANONICAL)
    T = 40_000
    q = am.msg_queue()
    rx = am.rx_path(rate, 7.0, q, use_pmf=True)
    rx.set_start_time(100, 0.25)
    rx.add_time_tag(T, 200, 0.5)
    rx.process(sc.iq, flush=True)
    assert [f.sample_index for f in rx.frames] == [int(x) for x in plain.index]
    ri = int(rate)
    for f in rx.frames:
        i = int(f.sample_index)
        base, off = ((200, 0.5), T) if i >= T else ((100, 0.25), 0)
        secs, frac = base[0] + (i - off) // ri, base[1] + ((i - off) % ri) / float(ri)
        if frac > 1.0:
            frac -= 1.0; secs += 1
        assert (f.secs, f.frac) == (secs, frac)
    with pytest.raises(RuntimeError):
        rx.add_time_tag(T - 1, 1, 0.0)                      # ascending offsets only


# ---- GNU Radio adapters (gr_adapter.py) against a stand-in gnuradio.gr: the test is the scheduler ---------------------
def _import_gr_adapter():
    stubs = os.path.join(ROOT, "tests", "stubs")
    if stubs not in sys.path:
        sys.path.insert(0, stubs)
    import importlib
    import gr_air_modes_b200.gr_adapter as ga
    return importlib.reload(ga)


def _drive_sink(blk, items, cuts, tags=()):
    """Hand `items` to a sink block's work() in ragged pieces; honours partial consumption."""
    from gnuradio import gr
    blk._in_tags[0] = [gr.tag_t(o, k, v) for (o, k, v) in tags]
    pos, n, k = 0, len(items), 0
    blk._nread[0] = 0
    blk.start()
    while pos < n:
        c = min(int(cuts[k % len(cuts)]), n - pos); k += 1
        c -= c % blk.output_multiple if c >= blk.output_multiple and pos + c < n else 0
        used = blk.work([items[pos:pos + c]], [])
        assert 0 <= used <= c
        if used == 0 and pos + c >= n:
            break
        if used == 0:
            cuts = [x + 240 for x in cuts]                      # give it more next time, as a scheduler would
        blk._nread[0] += used
        pos += used
    blk.stop()


def test_gr_adapter_rx_path_sink_with_ragged_work_calls_and_restart(port):
    ga = _import_gr_adapter()
    rate = 4e6
    sc = synth.make_scene(rate, 150_000, 30, 905)
    want = port.run_iq(sc.iq, rate, 7.0, True, co.MA_CANONICAL)
    q = am.msg_queue()
    blk = ga.rx_path(rate, 7.0, q, use_pmf=True)
    blk._impl.set_option("coalesce", 20_000)
    c64 = sc.iq.view(np.complex64)
    _drive_sink(blk, c64, [8191, 4096, 1, 32768, 777])
    assert q.strings() == want.msgs
    assert blk.get_threshold() == 7.0 and blk.get_pmf() is True
    q.flush()
    _drive_sink(blk, c64, [32768])                              # stop() + start(): the flowgraph was restarted
    assert q.strings() == want.msgs                             # a new stream incl. the first-message precision quirk
    # rx_time tags from a UHD source: item 0 = start time, a later one = after an overflow
    import pmt
    q.flush()
    key = pmt.string_to_symbol("rx_time")
    tags = [(0, key, pmt.make_tuple(pmt.from_uint64(1000), pmt.from_double(0.5))),
            (70_000, key, pmt.make_tuple(pmt.from_uint64(2000), pmt.from_double(0.125)))]
    _drive_sink(blk, c64, [30_000], tags)
    secs = [int(m.split()[3]) for m in q.strings()]
    idx = [int(f) for f in want.index[[i for i, f in enumerate(want.frames) if f.passed]]]
    assert len(secs) == len(idx) and all((s >= 2000) == (i >= 70_000) for s, i in zip(secs, idx)) and min(secs) >= 1000


def test_gr_adapter_split_blocks_preamble_then_slicer(port, ref):
    """The reference's own wiring of the two blocks (rx_path.py:57-65) with the adapters in their place: float streams
    -> preamble adapter (240 items + preamble_found tag per detection) -> slicer adapter -> queue."""
    from helpers import chips_digest
    ga = _import_gr_adapter()
    from gnuradio import gr
    rate = 4e6
    sc = synth.make_scene(rate, 120_000, 24, 906)
    bb, avg = port.frontend(sc.iq, rate, True, co.MA_CANONICAL)
    want = ref.run_streams(bb, avg, rate, 7.0)
    pre = ga.preamble(rate, 7.0)
    assert pre.get_rate() == 4e6 and pre.get_threshold() == 7.0
    stream, pos, cuts, k = [], 0, [4096, 9999, 1, 30000], 0
    while pos < bb.size:
        c = min(cuts[k % len(cuts)], bb.size - pos); k += 1
        out = np.zeros(240 * 3, np.float32)                      # deliberately small: packets must queue up inside
        pre._consumed = [0, 0]
        produced = pre.general_work([bb[pos:pos + c], avg[pos:pos + c]], [out])
        assert pre._consumed == [c, c] and produced % 240 == 0
        stream.append(out[:produced].copy()); pre._nwritten[0] += produced
        pos += c
        while pre._out:                                          # the scheduler keeps calling while forecast() says 0 inputs
            need = [1, 1]; pre.forecast(240, need); assert need == [0, 0]
            produced = pre.general_work([bb[:0], avg[:0]], [out])
            stream.append(out[:produced].copy()); pre._nwritten[0] += produced
    pre.stop()
    out = np.zeros(240 * max(1, len(pre._out)), np.float32)
    produced = pre._emit(out); stream.append(out[:produced].copy())
    items = np.concatenate(stream)
    assert items.size == 240 * len(want.index)
    assert chips_digest(items.reshape(-1, 240)) == want.chips_sha256
    assert [t.offset for t in pre.out_tags] == [240 * i for i in range(len(want.index))]
    q = am.msg_queue()
    sl = ga.slicer(q)
    _drive_sink(sl, items, [240 * 5, 240, 240 * 17 + 100], [(t.offset, t.key, t.value) for t in pre.out_tags])
    assert q.strings() == want.msgs


# ---- device-side drain (amb_drain_device): stream order + stamps without the host -------------------------------------
def _feed(rx, iq, cuts):
    pos, n = 0, iq.size // 2
    for c in list(cuts) + [n]:
        c = int(min(c, n - pos))
        last = pos + c >= n
        rx.process(iq[2 * pos: 2 * (pos + c)], flush=last, collect=False)
        pos += c
        if last:
            break


@pytest.mark.parametrize("tile", [2048, 16, 2])
def test_device_side_drain_equals_host_poll(port, tile):
    """amb_drain_device hands out, in device memory, byte for byte the records amb_poll_frames copies to the host: same
    order (sorting network over the work-list order of several calls; small tiles force its global stages), same stamps
    (start time + a later rx_time tag)."""
    import ctypes as C
    rate = 4e6
    sc = synth.make_scene(rate, 260_000, 150, 907, garble_frac=0.2)
    cuts = [70_000, 33_333, 90_001]

    def ctx():
        q = am.msg_queue()
        rx = am.rx_path(rate, 7.0, q, use_pmf=True)
        rx.set_option("order_tile", tile)
        rx.set_start_time(1000, 0.75)
        rx.add_time_tag(120_000, 5000, 0.999)
        return rx

    rx = ctx()
    _feed(rx, sc.iq, cuts)
    buf, got = rx._ctx.poll_array()
    want = bytes(buf)[:got * 80]
    rx.close()
    assert got > 64                                   # several tiles of 16: the global stages run
    idx = [int(buf[k].sample_index) for k in range(got)]
    assert idx == sorted(idx) and idx == [int(x) for x in port.run_iq(sc.iq, rate, 7.0, True, co.MA_CANONICAL).index]

    rx = ctx()
    _feed(rx, sc.iq, cuts)
    n = rx._ctx.call("amb_drain_device", None, 0)
    assert n == got
    with pytest.raises(RuntimeError):
        rx._ctx.call("amb_drain_device", (am.Frame * n)(), n - 1)      # too small: nothing consumed
    out = (am.Frame * n)()
    assert rx._ctx.call("amb_drain_device", out, n) == n
    assert bytes(out) == want
    assert rx._ctx.call("amb_drain_device", None, 0) == 0 and rx._ctx.call("amb_pending_frames") == 0
    rx.close()

    # frames that a non-blocking poll already moved to the host stay there; the device drain hands out the rest
    rx = ctx()
    rx.set_option("coalesce", 4096)                   # dispatch the first call at once instead of gathering 2^18 samples
    rx.process(sc.iq[: 2 * 100_000], flush=False, collect=False)
    hb, hgot = rx._ctx.poll_ready_array(4096)
    head = bytes(hb)[:hgot * 80]
    rx.process(sc.iq[2 * 100_000:], flush=True, collect=False)
    n2 = rx._ctx.call("amb_drain_device", None, 0)
    out2 = (am.Frame * max(n2, 1))()
    assert rx._ctx.call("amb_drain_device", out2, n2) == n2
    assert hgot > 0 and n2 > 0 and head + bytes(out2)[:n2 * 80] == want
    rx.close()


def test_frames_go_from_the_slicer_to_the_decoder_in_device_memory():
    """amb_drain_device -> amb_decode_frames_device (the whole chain without a host copy of the frames) gives the records
    of the host-driven chain (amb_poll_frames -> amb_decode_frames), byte for byte."""
    import ctypes as C
    from gr_air_modes_b200 import decode
    rate = 4e6
    sc = synth.make_scene(rate, 200_000, 110, 911)

    def ctx():
        rx = am.rx_path(rate, 7.0, am.msg_queue(), use_pmf=True)
        rx.set_start_time(500, 0.5)
        return rx

    rx = ctx()
    rx.process(sc.iq, flush=True)
    frames = list(rx.frames)
    rx.close()
    d = decode.batch_decoder([45.0, 9.0])
    want = d.decode(frames).tobytes()
    d.close()

    rx = ctx()
    _feed(rx, sc.iq, [90_000, 50_000])
    n = rx._ctx.call("amb_drain_device", None, 0)
    assert n == len(frames) > 50
    fr = (am.Frame * n)()
    assert rx._ctx.call("amb_drain_device", fr, n) == n
    rx.close()
    d = decode.batch_decoder([45.0, 9.0])
    rec = (C.c_uint8 * (144 * n))()
    d._check(d._lib.amb_decode_frames_device(d._h, fr, n, rec))
    d.close()
    assert bytes(rec) == want

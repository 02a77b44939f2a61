"""SURVEY.md 8 row f4 (field decode: parse.py / altitude.py / cpr.py) - CPU side.

  * oracle/decode_oracle.py against the committed golden produced by the UNMODIFIED reference modules
    (tests/golden/make_decode_golden.py), bit-exact incl. every float;
  * the same on further seeds and unconstrained message bytes, against what the reference computed for them
    (tests/golden/make_decode_ref_golden.py);
  * the product's per-message device code (gr_air_modes_b200/csrc/amb_decode_core.h, the `__host__ __device__`
    functions the CUDA kernels call) compiled for the host by tests/decode_host_shim.cc - a test-only harness, not a
    product path - against the golden, so the decode arithmetic is checked even where no GPU is present.
"""
import os
import sys

import pytest

from helpers import compare_decode, load_decode_golden, load_decode_ref_golden

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def test_decode_oracle_matches_reference_golden():
    from oracle import decode_oracle as do
    n = 0
    for ci, case in enumerate(load_decode_golden()):
        recs = do.decode_batch([tuple(m) for m in case["msgs"]], case["location"])
        assert len(recs) == len(case["ref"])
        for k, (rec, ref) in enumerate(zip(recs, case["ref"])):
            compare_decode(rec, ref, 0.0, "case %d msg %d" % (ci, k))
            n += 1
    assert n > 5000


def test_decode_oracle_matches_live_reference_on_fresh_seeds():
    import decode_cases
    from oracle import decode_oracle as do
    for case in load_decode_ref_golden()["fresh"]:
        seed = case["seed"]
        loc, msgs = decode_cases.make_case(seed, location=case["location"], seconds=30.0, surface_share=0.4)
        recs = do.decode_batch(msgs, loc)
        assert len(recs) == len(case["ref"])
        for k, (rec, r) in enumerate(zip(recs, case["ref"])):
            compare_decode(rec, r, 0.0, "seed %d msg %d" % (seed, k))


# ---- the product's decode arithmetic, compiled for the host by a test-only shim -------------------------------------
@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    import ctypes as C
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = str(tmp_path_factory.mktemp("shim") / "libdecode_shim.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-o", out,
                    os.path.join(root, "tests", "decode_host_shim.cc")], check=True)
    lib = C.CDLL(out)
    lib.shim_decode.restype = C.c_int
    lib.shim_decode.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p]
    lib.shim_nl.restype = C.c_int
    lib.shim_nl.argtypes = [C.c_double]
    return lib


def _shim_decode(lib, msgs, location):
    import ctypes as C
    import numpy as np
    from gr_air_modes_b200 import decode
    arr, n = decode.frames_from_messages(msgs)
    out = np.zeros(n, dtype=decode.FIELDS_DTYPE)
    have, lat, lon = (0, 0.0, 0.0) if location is None else (1, location[0], location[1])
    assert lib.shim_decode(C.cast(arr, C.c_void_p), n, have, lat, lon, C.c_void_p(out.ctypes.data)) == 0
    return [decode.record_to_dict(r) for r in out]


def test_product_decode_core_on_host_matches_reference_golden(shim):
    assert shim.shim_sizeof_fields() == 144
    n = 0
    for ci, case in enumerate(load_decode_golden()):
        recs = _shim_decode(shim, [tuple(m) for m in case["msgs"]], case["location"])
        for k, (rec, ref) in enumerate(zip(recs, case["ref"])):
            # lat/lon bit-exact; hypot-based values to 1e-14 (CPython's math.hypot is its own routine, not libm's)
            compare_decode(rec, ref, 0.0, "case %d msg %d" % (ci, k), tol_libm=1e-14)
            n += 1
    assert n > 5000


def test_product_decode_core_equals_oracle_record_for_record(shim):
    """Every member of struct amb_fields, not only what the reference's consumers read."""
    import math
    import decode_cases
    from oracle import decode_oracle as do
    for seed in (201, 202):
        loc, msgs = decode_cases.make_case(seed, location=(None if seed == 202 else (-12.0, 130.9)), seconds=25.0,
                                           surface_share=0.5, n_random=500)
        want = do.decode_batch(msgs, loc)
        got = _shim_decode(shim, msgs, loc)
        for k, (g, w) in enumerate(zip(got, want)):
            for key, wv in w.items():
                gv = g[key]
                near = key in ("val", "range", "bearing")          # hypot & co: last-place differences allowed
                for a, b in (zip(gv, wv) if isinstance(wv, list) else [(gv, wv)]):
                    if isinstance(b, float) and math.isnan(b):
                        assert math.isnan(a), (seed, k, key, g, w)
                    elif near:
                        assert abs(a - b) <= 1e-14 * max(1.0, abs(b)), (seed, k, key, g, w)
                    else:
                        assert a == b, (seed, k, key, g, w)


def test_nl_table_equals_formula(shim):
    """amb_nl() (transition table built from the host libm) against cpr.py:46-51 evaluated directly."""
    import numpy as np
    from oracle import decode_oracle as do
    rng = np.random.default_rng(5)
    lats = np.concatenate([rng.uniform(-90, 90, 20000), [0.0, 86.999, 87.0, -87.0, 89.9, 10.4704713, -10.4704713]])
    # and a fine sweep across every transition
    for k in range(2, 60):
        lo, hi = 0.0, 87.0
        for _ in range(60):
            mid = (lo + hi) / 2
            if do.nl(mid) >= k:
                lo = mid
            else:
                hi = mid
        lats = np.concatenate([lats, lo + np.arange(-50, 51) * 1e-13, -(lo + np.arange(-50, 51) * 1e-13)])
    bad = [x for x in lats if shim.shim_nl(float(x)) != int(do.nl(float(x)))]
    # only latitudes within a few ulp of a transition may differ (libm is not monotone to the last bit there)
    assert len(bad) <= 20, bad[:10]
    for x in bad:
        assert any(abs(do.nl(x + d) - do.nl(x - d)) == 1 for d in (1e-12,)), x


def test_report_lines_match_reference_printer(shim):
    """gr_air_modes_b200.report (the text apps/modes_rx prints by default) against the lines the UNMODIFIED
    python/msprint.py printed for the same messages (golden 'lines'); records from the host build of the product's
    decode arithmetic."""
    import decode_cases
    from gr_air_modes_b200 import report
    n = printed = 0
    for ci, case in enumerate(load_decode_golden()):
        msgs = [tuple(m) for m in case["msgs"]]
        recs = _shim_decode(shim, msgs, case["location"])
        for k, (text, rec, want) in enumerate(zip(decode_cases.message_strings(msgs), recs, case["lines"])):
            got = report.format_report(text, rec)
            assert got == want, (ci, k, text, got, want)
            n += 1
            printed += want is not None
    assert n > 5000 and printed > 4000


def test_fuzz_oracle_core_and_reports_against_live_reference(shim):
    """Unconstrained message bytes (incl. what no slicer emits: long DFs in 56 bits, short DFs in 112 bits) through
    the UNMODIFIED parse.py / altitude.py / cpr.py / msprint.py, the oracle, the host build of the product's decode
    arithmetic, and report.py: all four agree message by message. The whole stream is decoded (CPR state carries
    across messages); the reference's results are stored for a fixed sample of 1500 of its 12000 messages."""
    import decode_cases
    from gr_air_modes_b200 import report
    from oracle import decode_oracle as do
    msgs = decode_cases.fuzz_messages()
    keep = decode_cases.fuzz_sample(len(msgs))
    texts = decode_cases.message_strings(msgs)
    stored = load_decode_ref_golden()["fuzz"]
    assert [c["location"] for c in stored] == list(decode_cases.FUZZ_LOCATIONS)
    for case in stored:
        loc = case["location"]
        want = do.decode_batch(msgs, loc)
        got = _shim_decode(shim, msgs, loc)
        for k, r, line in zip(keep, case["ref"], case["lines"]):
            compare_decode(want[k], r, 0.0, "oracle %d %s" % (k, msgs[k][0]))
            compare_decode(got[k], r, 0.0, "core %d %s" % (k, msgs[k][0]), tol_libm=1e-13)
            assert report.format_report(texts[k], got[k]) == line, (k, texts[k])
        assert sum("pos" in r for r in case["ref"]) > 40


class _ShimBackend:
    """Stands in for decode.batch_decoder in CPU tests: same decode()/set_location() surface, arithmetic from the host
    build of the product's decode core (tests/decode_host_shim.cc), state kept across calls like the device table."""

    def __init__(self, lib, location):
        import ctypes as C
        lib.shim_new.restype = C.c_void_p
        lib.shim_step.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p]
        self._lib, self._h, self._loc = lib, lib.shim_new(), location

    def set_location(self, loc):
        self._loc = loc

    def decode(self, frames, n):
        import ctypes as C
        import numpy as np
        from gr_air_modes_b200 import decode
        out = np.zeros(n, dtype=decode.FIELDS_DTYPE)
        have, lat, lon = (0, 0.0, 0.0) if self._loc is None else (1, self._loc[0], self._loc[1])
        self._lib.shim_step(self._h, C.cast(frames, C.c_void_p), n, have, lat, lon, C.c_void_p(out.ctypes.data))
        return out


def test_cpr_decoder_dropin_class_against_the_reference_class(shim):
    """decode.cpr_decoder (same methods, return list and exceptions as python/cpr.py:183-240) against what the
    UNMODIFIED reference class returned on the reference's own self-test procedure (cpr.py:264-331: sweep of
    positions, even then odd report) plus surface reports, expiry and a moving receiver location, on one injected
    clock (decode_cases.cpr_class_script)."""
    import decode_cases as dc
    from gr_air_modes_b200 import decode
    from gr_air_modes_b200.errors import CPRBoundaryStraddleError, CPRNoPositionError
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_decode_golden as mg
    stored = load_decode_ref_golden()["cpr_class"]
    clock = mg.Clock()
    ok = straddle = nopos = 0
    for surface, (loc, events) in dc.cpr_class_script().items():
        ours = decode.cpr_decoder(list(loc), clock=clock.time, _backend=_ShimBackend(shim, list(loc)))
        wants = iter(stored[str(surface)])
        for ev in events:
            if ev[0] == "loc":
                ours.set_location(list(ev[1]))
                continue
            _, clock.now, icao, la, lo, odd = ev
            want = next(wants)
            try:
                got = ours.decode(icao, la, lo, odd, surface)
            except CPRBoundaryStraddleError:
                got = "straddle"
            except CPRNoPositionError:
                got = "nopos"
            if isinstance(want, str):
                assert got == want, (surface, ev, got, want)
                straddle += want == "straddle"
                nopos += want == "nopos"
            else:
                assert got[0] == want[0] and got[1] == want[1], (surface, ev, got, want)     # lat/lon bit-exact
                assert abs(got[2] - want[2]) <= 1e-12 * max(1, want[2]) and abs(got[3] - want[3]) <= 1e-10
                ok += 1
        assert next(wants, None) is None
    assert ok > 2500 and nopos >= 2 * 1500 and straddle > 0

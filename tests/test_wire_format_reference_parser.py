"""SURVEY.md 8 row f2: the message strings we emit are consumed by the reference's UNMODIFIED parser
(python/parse.py make_parser, :422-436). What the parser published for each message of tests/golden/golden.json is
stored by tests/golden/make_decode_ref_golden.py (the reference files imported in place behind a stub `air_modes`
package, never copied); the messages themselves are what the oracle port computes for the golden scenes."""
import math

from oracle import cpu_oracle as co

from helpers import load_decode_ref_golden, load_golden


def test_reference_parser_accepts_our_messages(port):
    meta, scenes = load_golden()
    parsed = load_decode_ref_golden()["parser"]
    seen = 0
    for s, iq in scenes:
        msgs = port.run_iq(iq, s["rate"], s["threshold_db"], s["use_pmf"], co.MA_CANONICAL).msgs
        assert msgs == s["msgs"], s["name"]
        for m in msgs:
            rep = parsed[m]
            data, ecc, ref, secs, frac = m.split()
            if rep is None:                 # the parser drops types it has no handler for (ADSBError)
                continue
            assert rep["ecc"] == int(ecc, 16)
            assert abs(rep["rssi"] - 10.0 * math.log10(max(1e-8, float(ref)))) < 1e-12
            assert rep["secs"] == int(secs) and rep["frac_secs"] == float(frac)
            df = int(data[:2], 16) >> 3
            assert rep["df"] == df and rep["typed"]
            if df in (11, 17) and data in s["sent"]:
                assert rep["aa"] == int(data[2:8], 16)      # ICAO address straight from our payload
                seen += 1
    assert seen >= 20

"""Generates tests/golden/decode_ref_golden.json.xz: what the UNMODIFIED reference modules (python/parse.py, altitude.py,
cpr.py, msprint.py, modes_types.py, loaded where they lie as in make_decode_golden.py) compute for the inputs of
tests/test_decode_cpu.py and tests/test_wire_format_reference_parser.py that are not in decode_golden.json.gz:

  fresh      run_reference records of three further make_case() seeds
  fuzz       run_reference records and msprint lines of decode_cases.fuzz_messages() at three receiver locations,
             kept at the indices decode_cases.fuzz_sample() picks
  cpr_class  the outcome of every decode() of the reference's cpr_decoder class on decode_cases.cpr_class_script()
  parser     per message of tests/golden/golden.json, the modes_report make_parser (parse.py:422-436) published

Nothing in the output is hand-edited.

    python tests/golden/make_decode_ref_golden.py
"""
import json
import lzma
import math
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
import make_decode_golden as mg  # noqa: E402  (puts the repository and tests/ on sys.path)

FRESH = [(seed, None if seed == 102 else (40.0 + seed % 7, -70.0)) for seed in (101, 102, 103)]


def fresh(mods):
    import decode_cases
    out = []
    for seed, loc in FRESH:
        loc, msgs = decode_cases.make_case(seed, location=loc, seconds=30.0, surface_share=0.4)
        out.append({"seed": seed, "location": loc, "ref": mg.run_reference(loc, msgs, mods)})
    return out


def fuzz(mods):
    import decode_cases
    msgs = decode_cases.fuzz_messages()
    keep = decode_cases.fuzz_sample(len(msgs))
    out = []
    for loc in decode_cases.FUZZ_LOCATIONS:
        ref = mg.run_reference(loc, msgs, mods)
        lines = mg.run_reference_printer(loc, msgs, mods)
        out.append({"location": loc, "ref": [ref[k] for k in keep], "lines": [lines[k] for k in keep]})
    return out


def cpr_class(mods):
    import decode_cases
    exc, alt, parse, cpr = mods
    clock = mg.Clock()
    cpr.time = type("T", (), {"time": staticmethod(clock.time)})
    out = {}
    for surface, (loc, events) in decode_cases.cpr_class_script().items():
        dec = cpr.cpr_decoder(list(loc))
        got = []
        for ev in events:
            if ev[0] == "loc":
                dec.set_location(list(ev[1]))
                continue
            _, clock.now, icao, la, lo, odd = ev
            try:
                got.append([float(x) for x in dec.decode(icao, la, lo, odd, surface)])
            except exc.CPRBoundaryStraddleError:
                got.append("straddle")
            except exc.CPRNoPositionError:
                got.append("nopos")
        out[str(surface)] = got
    return out


def parser(mods):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import load_golden
    exc, alt, parse, cpr = mods
    meta, _ = load_golden()
    out = {}
    for s in meta["scenes"]:
        for m in s["msgs"]:
            pub = {}
            parse.make_parser(pub)(m)
            if "modes_dl" not in pub:       # the parser drops types it has no handler for (ADSBError)
                out[m] = None
                continue
            rep = pub["modes_dl"]
            df = rep.data.get_type()
            out[m] = {"ecc": rep.ecc, "rssi": rep.rssi, "secs": rep.timestamp.secs, "frac_secs": rep.timestamp.frac_secs,
                      "df": df, "typed": ("type%i_dl" % df) in pub,
                      "aa": rep.data["aa"] if df in (11, 17) else None}
    return out


def main():
    mods = mg.load_reference()
    data = {"fresh": fresh(mods), "fuzz": fuzz(mods), "cpr_class": cpr_class(mods), "parser": parser(mods)}
    mg.unload_reference()

    def clean(o):
        if isinstance(o, float) and (math.isnan(o) or math.isinf(o)):
            return None
        if isinstance(o, dict):
            return {k: clean(v) for k, v in o.items()}
        if isinstance(o, (list, tuple)):
            return [clean(v) for v in o]
        return o
    path = os.path.join(HERE, "decode_ref_golden.json.xz")
    with lzma.open(path, "wb", preset=9) as f:
        f.write(json.dumps(clean(data), separators=(",", ":")).encode())
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()

import fcntl
import hashlib
import json
import lzma
import os
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_RESULTS = os.path.join(HERE, "golden", "ref_results.json.xz")


def chips_digest(chips):
    """SHA-256 of 240-chip packets (float32), every NaN in one canonical form: equal digests = np.array_equal(equal_nan)."""
    a = np.array(chips, dtype=np.float32)
    a[np.isnan(a)] = np.nan
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


class RecordedRef:
    """The unmodified reference objects (oracle/_ref: preamble_impl.cc, slicer_impl.cc, modes_crc.cc) as the tests see
    them, replayed from tests/golden/ref_results.json.xz: every call the tests make is keyed by a hash of its arguments,
    so an input the reference was never shown has no answer and the test fails. Results carry the chip packets as
    `chips_sha256` (see chips_digest). tests/golden/make_ref_golden.py records the file by running the tests against
    the live objects (`live`), where the reference sources exist."""

    def __init__(self, live=None):
        self.live, self.new = live, {}
        if live is None:
            with lzma.open(REF_RESULTS, "rt") as f:
                self.table = json.load(f)

    @staticmethod
    def _key(name, *args):
        h = hashlib.sha256(name.encode())
        for a in args:
            if isinstance(a, np.ndarray):
                h.update(b"a" + str(a.dtype).encode() + np.ascontiguousarray(a).tobytes())
            else:
                h.update(b"s" + repr(a).encode())
        return h.hexdigest()

    def _call(self, key, compute):
        if self.live is None:
            if key not in self.table:
                raise KeyError("no recorded reference result for this input: rerun tests/golden/make_ref_golden.py")
            return self.table[key]
        self.new[key] = compute()
        return self.new[key]

    def save(self):
        """Record mode: merge this session's calls into the file (several pytest processes may record at once)."""
        if self.live is None or not self.new:
            return
        with open(os.path.join(tempfile.gettempdir(), "amb_ref_results.lock"), "w") as lock:
            fcntl.flock(lock, fcntl.LOCK_EX)
            table = {}
            if os.path.exists(REF_RESULTS):
                with lzma.open(REF_RESULTS, "rt") as f:
                    table = json.load(f)
            table.update(self.new)
            with lzma.open(REF_RESULTS, "wb", preset=9) as f:
                f.write(json.dumps(table, sort_keys=True, separators=(",", ":")).encode())

    @staticmethod
    def _result(d):
        from oracle.cpu_oracle import Result
        r = Result(np.array(d["index"], np.uint64), np.array(d["secs"], np.uint64), np.array(d["frac"], np.float64),
                   None, d["msgs"], None, d["calls"])
        r.chips_sha256 = d["chips_sha256"]
        return r

    @staticmethod
    def _record(r):
        return {"index": [int(x) for x in r.index], "secs": [int(x) for x in r.secs], "frac": [float(x) for x in r.frac],
                "chips_sha256": chips_digest(r.chips), "msgs": r.msgs, "calls": r.calls}

    def crc24(self, data: bytes) -> int:
        data = bytes(data)
        return self._call(self._key("crc24", data), lambda: self.live.crc24(data))

    def preamble_params(self, rate, threshold_db):
        rate, thr = float(rate), float(threshold_db)
        return tuple(self._call(self._key("preamble_params", rate, thr), lambda: list(self.live.preamble_params(rate, thr))))

    def run_streams(self, bb, avg, rate, threshold_db, slice_=True, start_time=None):
        bb, avg = np.ascontiguousarray(bb, np.float32), np.ascontiguousarray(avg, np.float32)
        rate, thr = float(rate), float(threshold_db)
        st = None if start_time is None else (int(start_time[0]), float(start_time[1]))
        key = self._key("run_streams", bb, avg, rate, thr, bool(slice_), st)
        return self._result(self._call(key, lambda: self._record(self.live.run_streams(bb, avg, rate, thr, slice_, st))))

    def run_slicer(self, chips, secs, frac):
        chips = np.ascontiguousarray(chips, np.float32)
        secs, frac = np.ascontiguousarray(secs, np.uint64), np.ascontiguousarray(frac, np.float64)
        key = self._key("run_slicer", chips, secs, frac)
        return self._result(self._call(key, lambda: self._record(self.live.run_slicer(chips, secs, frac))))


def load_golden():
    with open(os.path.join(HERE, "golden", "golden.json")) as f:
        meta = json.load(f)
    z = np.load(os.path.join(HERE, "golden", "scenes.npz"))
    scenes = []
    for s in meta["scenes"]:
        iq = z[s["name"]].astype(np.float32) / np.float32(2048.0)
        scenes.append((s, iq))
    return meta, scenes


def parse_msg(m):
    """'<hex> <crc> <ref> <secs> <frac>' (slicer_impl.cc:186-192, parse.py:425)."""
    data, crc, ref, secs, frac = m.split()
    return data, int(crc, 16), float(ref), int(secs), float(frac)


def first_four(bb, avg, rate, threshold_db, port):
    """Indices (reported coordinates) passing preamble_impl.cc:173-179, vectorised in float32."""
    p = port.params(rate, threshold_db)
    H = p.history - 1
    n = bb.size
    pad = 16 * int(np.ceil(p.spc)) + 8
    a = np.concatenate([np.zeros(H, np.float32), bb, np.zeros(pad, np.float32)])
    v = np.concatenate([np.zeros(H, np.float32), avg, np.zeros(pad, np.float32)])
    m = n + H
    thr = (v[:m] * np.float32(p.threshold)).astype(np.float32)
    ok = a[:m] > thr
    ok &= ~(a[1:m + 1] > a[:m])
    for k in (1, 2, 3):
        ok &= ~(a[p.po[k]:m + p.po[k]] < thr)
    return np.nonzero(ok)[0]


# ---- field-decode parity (SURVEY.md 8 row f4) -----------------------------------------------------
def load_decode_golden():
    import gzip
    with gzip.open(os.path.join(HERE, "golden", "decode_golden.json.gz"), "rt") as f:
        return json.load(f)["cases"]


def load_decode_ref_golden():
    """What the unmodified reference modules computed for the inputs of tests/golden/make_decode_ref_golden.py."""
    with lzma.open(os.path.join(HERE, "golden", "decode_ref_golden.json.xz"), "rt") as f:
        return json.load(f)


def compare_decode(rec, ref, tol=0.0, where="", tol_libm=None):
    """rec: one decoded record (dict with the members of struct amb_fields); ref: what the unmodified reference
    computed for the same message (tests/golden/make_decode_golden.py). Integers and strings must be equal.
    Latitude/longitude/ground track (+, -, *, /, floor, fmod only) are compared with relative tolerance `tol`
    (0 = bit-exact); velocity, heading, range and bearing go through hypot/atan2/sin/cos/pow, where CPython's own
    hypot and each libm differ in the last place: `tol_libm` (default = tol)."""
    import math
    NO_HANDLER, METRIC, NOPOS, STRADDLE, HASPOS, HASRNG = 0x01, 0x02, 0x04, 0x08, 0x10, 0x20

    if tol_libm is None:
        tol_libm = tol

    def close(a, b, t=None):
        t = tol if t is None else t
        if b is None:
            return a is None or math.isnan(a)
        if t == 0.0:
            return a == b
        return abs(a - b) <= t * max(1.0, abs(b))

    st = rec["status"]
    if "dropped" in ref:
        assert st & NO_HANDLER, (where, rec, ref)
        return
    assert not (st & NO_HANDLER), (where, rec, ref)
    assert rec["df"] == ref["df"], (where, rec, ref)
    for k in ("vs", "ri", "sl", "fs", "ca", "icao", "squawk", "ftc", "cat", "eps", "tti", "ast", "subtype"):
        if k in ref:
            assert rec[k] == ref[k], (where, k, rec, ref)
    if "bds" in ref:
        assert rec["bds"] == ref["bds"], (where, rec, ref)
    if "metric_alt" in ref:
        assert st & METRIC, (where, rec, ref)
    elif "altitude" in ref:
        assert not (st & METRIC) and rec["altitude"] == ref["altitude"], (where, rec, ref)
    if "ident" in ref:
        assert rec["ident"] == ref["ident"], (where, rec, ref)
    if "aux" in ref:
        assert list(rec["aux"]) == ref["aux"], (where, rec, ref)
    if "ara" in ref:
        assert rec["aux"][0] == ref["ara"] and rec["aux"][1] == ref["rac"], (where, rec, ref)
        assert rec["aux"][2] == (ref["rat"] | (ref["mte"] << 1)), (where, rec, ref)
    if "tid" in ref:
        assert rec["aux"][3] == ref["tid"], (where, rec, ref)
    if "tidr" in ref:
        assert rec["aux"][3] == (ref["tidr"] | (ref["tidb"] << 8)) and rec["threat_alt"] == ref["threat_alt"], (where, rec, ref)
        assert not (st & 0x40), (where, rec, ref)
    if "threat_metric_alt" in ref:
        assert st & 0x40, (where, rec, ref)          # AMB_FS_METRIC_THREAT
    if "cpr" in ref:
        assert [rec["cpr_format"], rec["cpr_lat"], rec["cpr_lon"]] == ref["cpr"], (where, rec, ref)
    if "ground_track" in ref:
        assert close(rec["val"][0], ref["ground_track"]), (where, rec, ref)
    if "val" in ref:
        for a, b in zip(rec["val"], ref["val"]):
            assert close(a, b, tol_libm), (where, rec, ref)
    if ref.get("cpr_error") == "straddle":
        assert (st & STRADDLE) and (st & NOPOS) and not (st & HASPOS), (where, rec, ref)
    elif ref.get("cpr_error") == "nopos":
        assert (st & NOPOS) and not (st & (STRADDLE | HASPOS)), (where, rec, ref)
    elif "pos" in ref:
        lat, lon, rng, brg = ref["pos"]
        assert (st & HASPOS) and not (st & NOPOS), (where, rec, ref)
        assert close(rec["lat"], lat) and close(rec["lon"], lon), (where, rec, ref)
        if rng is None:
            assert not (st & HASRNG), (where, rec, ref)
        else:
            assert st & HASRNG, (where, rec, ref)
            assert close(rec["range"], rng, tol_libm) and close(rec["bearing"], brg, tol_libm), (where, rec, ref)

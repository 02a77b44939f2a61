"""Seeded Mode S message sets for the field-decode tests (SURVEY.md 8 row f4). Tool-local generator: frames are
assembled bit by bit, parity from the Mode S CRC (modes_crc.cc:31), positions from a plain CPR encoder
(DO-260 formulas; the reference's own cpr_encode is cpr.py:243-262)."""
from __future__ import annotations

import math

import numpy as np

from gr_air_modes_b200.synth import crc24


def _nl(lat):
    if abs(lat) >= 87.0:
        return 1
    return int(math.floor(2.0 * math.pi / math.acos(
        1.0 - (1.0 - math.cos(math.pi / 30.0)) / math.cos(math.pi / 180.0 * abs(lat)) ** 2)))


def cpr_encode(lat, lon, odd, surface=False):
    scale = 2.0 ** 19 if surface else 2.0 ** 17
    dlat = 360.0 / (60 - odd)
    yz = math.floor(scale * ((lat % dlat) / dlat) + 0.5)
    rlat = dlat * (yz / scale + math.floor(lat / dlat))
    dlon = 360.0 / max(_nl(rlat) - odd, 1)
    xz = math.floor(scale * ((lon % dlon) / dlon) + 0.5)
    return int(yz) & 0x1FFFF, int(xz) & 0x1FFFF


def enc_alt12(feet):
    """25 ft Q-bit altitude code as carried in BDS0,5 (12 bits)."""
    n = (int(feet) + 1000) // 25
    return ((n & 0x7F0) << 1) | 0x10 | (n & 0x0F)


def enc_alt13(feet):
    """13-bit AC field, Q=1, M=0."""
    n = (int(feet) + 1000) // 25
    return ((n & 0x7E0) << 2) | ((n & 0x10) << 1) | 0x10 | (n & 0x0F)


class Bits:
    def __init__(self, nbits):
        self.v, self.n = 0, nbits

    def put(self, start, num, val):
        """1-based start from the MSB, like parse.py get_bits."""
        sh = self.n - start - num + 1
        self.v |= (int(val) & ((1 << num) - 1)) << sh
        return self

    def bytes(self):
        return self.v.to_bytes(self.n // 8, "big")


def finish(body: bytes, address: int = 0):
    """body = frame without the last 3 bytes. Returns (frame bytes, ecc) with AP/PI = parity ^ address."""
    par = crc24(body) ^ (address & 0xFFFFFF)
    return body + par.to_bytes(3, "big"), address & 0xFFFFFF


def df17(aa, me56, ca=5):
    b = Bits(88).put(1, 5, 17).put(6, 3, ca).put(9, 24, aa).put(33, 56, me56)
    return finish(b.bytes())


def me_airborne(ftc, alt12, odd, lat17, lon17, ss=0, saf=0, t=0):
    return Bits(56).put(1, 5, ftc).put(6, 2, ss).put(8, 1, saf).put(9, 12, alt12).put(21, 1, t).put(22, 1, odd) \
        .put(23, 17, lat17).put(40, 17, lon17).v


def me_surface(ftc, mvt, gts, gtk, odd, lat17, lon17):
    return Bits(56).put(1, 5, ftc).put(6, 7, mvt).put(13, 1, gts).put(14, 7, gtk).put(22, 1, odd) \
        .put(23, 17, lat17).put(40, 17, lon17).v


def me_ident(ftc, cat, text):
    v = 0
    for ch in (text + " " * 8)[:8]:
        if "A" <= ch <= "Z":
            d = ord(ch) - ord("A") + 1
        elif "0" <= ch <= "9":
            d = ord(ch)
        else:
            d = 32
        v = (v << 6) | d
    return Bits(56).put(1, 5, ftc).put(6, 3, cat).put(9, 48, v).v


def short_frame(df, rng, address):
    b = Bits(32).put(1, 5, df).put(6, 27, int(rng.integers(0, 1 << 27)))
    return finish(b.bytes(), address)


def long_frame(df, rng, address, mb=None):
    b = Bits(88).put(1, 5, df).put(6, 27, int(rng.integers(0, 1 << 27)))
    b.put(33, 56, int(rng.integers(0, 1 << 56, dtype=np.uint64)) if mb is None else mb)
    return finish(b.bytes(), address)


def raw_message(rng):
    """(frame bytes, ecc) with unconstrained contents; the DF and a few sub-type fields are steered so that every
    branch of the parser is reached often."""
    nb = 14 if rng.random() < 0.6 else 7
    raw = bytearray(rng.integers(0, 256, nb, dtype=np.uint8).tobytes())
    r = rng.random()
    if r < 0.45:
        raw[0] = (17 << 3) | (raw[0] & 7)
        raw[1], raw[2], raw[3] = 0, 0, int(rng.integers(0, 40))
        if nb == 14 and rng.random() < 0.7:
            ftc = int(rng.choice([1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 16, 17, 18, 19, 28]))
            raw[4] = (ftc << 3) | (raw[4] & 7)
    elif r < 0.5:
        raw[0], raw[1] = 0, 0                           # small value: modes_reply.is_long (parse.py:222-223)
    elif r < 0.75:
        raw[0] = (int(rng.choice([0, 4, 5, 11, 16, 20, 21, 24])) << 3) | (raw[0] & 7)
        if nb == 14 and rng.random() < 0.8:
            raw[4] = int(rng.integers(0, 4)) << 4       # MB register 0..3 / 0
    return bytes(raw), int(rng.integers(0, 1 << 24))


def make_case(seed, n_aircraft=6, seconds=40.0, location=(37.4, -122.1), surface_share=0.2, n_random=150):
    """Returns (location or None, [(hex, ecc, secs, frac), ...]) in time order."""
    rng = np.random.Generator(np.random.PCG64(seed))
    ev = []                                             # (t, frame, ecc)
    lat0, lon0 = location if location is not None else (48.0, 11.0)
    for a in range(n_aircraft):
        aa = int(rng.integers(1, 1 << 24))
        surface = rng.random() < surface_share
        lat = lat0 + rng.uniform(-1.5, 1.5)
        lon = lon0 + rng.uniform(-1.5, 1.5)
        if a == 1:
            lat = 10.4704713 + rng.uniform(-2e-3, 2e-3)  # next to an NL transition: boundary straddles
        if a == 2:
            lat, lon = -33.9 + rng.uniform(-1, 1), 151.2 + rng.uniform(-1, 1)   # southern / eastern hemisphere
        dlat, dlon = rng.uniform(-2e-3, 2e-3), rng.uniform(-2e-3, 2e-3)
        alt = int(rng.integers(0, 1600)) * 25
        t = rng.uniform(0, 1.0)
        odd = int(rng.integers(0, 2))
        quiet_from = rng.uniform(5, seconds) if a % 3 == 0 else 1e9            # a gap > 10 s: reports expire
        while t < seconds:
            if not (quiet_from < t < quiet_from + rng.uniform(11, 27)):
                if surface:
                    la, lo = cpr_encode(lat, lon, odd, True)
                    me = me_surface(int(rng.integers(5, 9)), int(rng.integers(0, 128)), 1, int(rng.integers(0, 128)), odd, la, lo)
                else:
                    la, lo = cpr_encode(lat, lon, odd, False)
                    ftc = int(rng.choice([9, 10, 11, 12, 13, 14, 16, 17, 18]))
                    me = me_airborne(ftc, enc_alt12(alt), odd, la, lo)
                ev.append((t, *df17(aa, me)))
                if rng.random() < 0.5:
                    odd ^= 1
            if rng.random() < 0.3:                      # velocity, all subtypes incl. the unhandled 5-7
                sub = int(rng.integers(0, 8))
                me = Bits(56).put(1, 5, 19).put(6, 3, sub).put(9, 48, int(rng.integers(0, 1 << 48))).v
                ev.append((t + 0.01, *df17(aa, me)))
            if rng.random() < 0.1:
                ev.append((t + 0.02, *df17(aa, me_ident(int(rng.integers(1, 5)), int(rng.integers(0, 7)), "TEST%03dX" % a))))
            if rng.random() < 0.05:
                ev.append((t + 0.03, *df17(aa, Bits(56).put(1, 5, 28).put(9, 3, int(rng.integers(0, 8))).v)))
            if rng.random() < 0.2:
                ev.append((t + 0.04, *short_frame(int(rng.choice([0, 4, 5])), rng, aa)))
            if rng.random() < 0.1:
                b = Bits(32).put(1, 5, 11).put(6, 3, 5).put(9, 24, aa)
                ev.append((t + 0.05, *finish(b.bytes(), int(rng.integers(0, 16)))))
            step = rng.uniform(0.4, 0.6)
            t += step
            lat += dlat * step
            lon += dlon * step
            alt = max(0, alt + int(rng.integers(-2, 3)) * 25)
    for _ in range(n_random):                           # anything the slicer could queue, random contents
        t = rng.uniform(0, seconds)
        kind = int(rng.integers(0, 8))
        addr = int(rng.integers(0, 1 << 24))
        if kind == 0:
            ev.append((t, *df17(addr, int(rng.integers(0, 1 << 56, dtype=np.uint64)))))
        elif kind == 1:
            ev.append((t, *short_frame(int(rng.choice([0, 4, 5, 11])), rng, addr)))
        elif kind == 2:
            ev.append((t, *long_frame(int(rng.choice([16, 20, 21])), rng, addr)))
        elif kind == 3:                                  # MB with a handled register
            mb = Bits(56).put(1, 4, int(rng.integers(0, 4))).put(9, 48, int(rng.integers(0, 1 << 48))).v
            ev.append((t, *long_frame(int(rng.choice([20, 21])), rng, addr, mb)))
        elif kind == 4:                                  # DFs the parser has no table for (sliced as short / long)
            df = int(rng.choice([1, 2, 3, 6, 7, 12, 18, 19, 22, 23, 24, 25, 31]))
            ev.append((t, *short_frame(df, rng, addr)))
        elif kind == 5:                                  # 13-bit AC with Q=1, and with the M bit set
            ac = enc_alt13(int(rng.integers(0, 2000)) * 25) | (0x40 if rng.random() < 0.3 else 0)
            b = Bits(32).put(1, 5, int(rng.choice([0, 4]))).put(6, 14, int(rng.integers(0, 1 << 14))).put(20, 13, ac)
            ev.append((t, *finish(b.bytes(), addr)))
        elif kind == 6:                                  # Gillham (Q=0) altitude, raw CPR bits
            me = me_airborne(int(rng.integers(9, 19)), int(rng.integers(0, 1 << 12)) & ~0x10, int(rng.integers(0, 2)),
                             int(rng.integers(0, 1 << 17)), int(rng.integers(0, 1 << 17)))
            ev.append((t, *df17(addr & 0xFF, me)))       # few addresses: random even/odd pairs do meet
        else:
            me = me_surface(int(rng.integers(5, 9)), int(rng.integers(0, 128)), 1, int(rng.integers(0, 128)),
                            int(rng.integers(0, 2)), int(rng.integers(0, 1 << 17)), int(rng.integers(0, 1 << 17)))
            ev.append((t, *df17(addr & 0xFF, me)))
    for _ in range(n_random // 3):                      # what no slicer emits but a message string can carry: free bytes,
        t = rng.uniform(0, seconds)                     # long DFs in 56 bits (sub-fields read 0), short DFs in 112 bits
        ev.append((t, *raw_message(rng)))
    ev.sort(key=lambda e: e[0])
    base = 1_700_000_000 if seed % 2 else 0             # UTC-sized seconds lose no precision in secs + frac? (they do: tested)
    msgs = []
    for t, frame, ecc in ev:
        secs = int(t)
        msgs.append((frame.hex(), ecc, base + secs, float(np.float64(t - secs))))
    return (list(location) if location is not None else None), msgs


def message_strings(msgs):
    """(hex, ecc, secs, frac) -> the slicer's message text (slicer_impl.cc:186-192) with a made-up reference level."""
    return ["%s %06x %r %d %r" % (h, e, 10.0 ** (-((7 * k) % 61) / 10.0), s, f) for k, (h, e, s, f) in enumerate(msgs)]


def fuzz_messages(n=12000, seed=77):
    """Unconstrained message bytes (raw_message), arrival gaps exponential with a rare 12 s silence."""
    rng = np.random.default_rng(seed)
    msgs, t = [], 0.0
    for _ in range(n):
        frame, ecc = raw_message(rng)
        t += float(rng.exponential(0.02)) + (12.0 if rng.random() < 0.001 else 0.0)
        msgs.append((frame.hex(), ecc, int(t), t - int(t)))
    return msgs


FUZZ_LOCATIONS = ([37.4, -122.1], None, [-45.0, 170.0])


def fuzz_sample(n, k=1500, seed=78):
    """The fixed indices of fuzz_messages() whose reference results are stored (all of them would exceed 500 kB)."""
    return sorted(int(x) for x in np.random.default_rng(seed).choice(n, k, replace=False))


def cpr_class_script(rounds=1500):
    """The reference's cpr.py self-test procedure (cpr.py:264-331: sweep of positions, even then odd report) plus
    surface reports, expiry and a moving receiver location, for a cpr_decoder class on an injected clock.
    -> {surface: (first location, [("loc", [lat, lon]) | ("decode", now, icao, lat_cpr, lon_cpr, odd), ...])}"""
    out = {}
    for surface in (0, 1):
        ev = []
        for i in range(rounds):
            lat = i / (rounds / 170.) - 85 if not surface else 35.0 + (i % 50) * 1e-3
            if not surface and 100 <= i < 160:
                lat = 10.4704713 - 7e-4 + (i - 100) * 2.5e-5          # across an NL transition: boundary straddles
            lon = i / (rounds / 360.) - 180 if not surface else -100.0 + (i % 70) * 1e-3
            icao = (i * 7919) & 0xFFFFFF
            now = 1000.0 + i * 0.37 + (30.0 if i == 700 else 0.0)
            if i == 900:
                ev.append(("loc", [34.5, -99.5]))
            for odd, dl in ((0, 0.0), (1, 1e-3)):
                la, lo = cpr_encode(lat + dl, min(lon + dl, 180), odd, bool(surface))
                now += 0.01
                ev.append(("decode", now, icao, la, lo, odd))
        out[surface] = ([35.0, -100.0], ev)
    return out


CASES = [
    dict(seed=11, location=(37.4, -122.1)),
    dict(seed=12, location=None),
    dict(seed=13, location=(-33.9, 151.2), surface_share=0.5),
    dict(seed=14, location=(51.5, -0.1), seconds=70.0, n_aircraft=10, n_random=400),
]

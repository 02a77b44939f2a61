"""The decoder's KERNEL SOURCE (gr_air_modes_b200/csrc/amb_decode_kernels.cuh: fields / pairing / resolve kernels, plus
the experimental pairing variants behind AMB_PAIR_V2 / AMB_PAIR_V3) executed on the host by a small SIMT emulator
(tests/simt/simt_emul.h: cooperative fibers, real barrier semantics for __syncthreads / __syncwarp / shuffles / votes /
match) and compared with the sequential host replay of the same arithmetic and with the oracle. A CPU-side check of the
warp-level logic - match/ballot ordering inside a 32-frame step, table hand-over between steps and batches, the stable
partition of variant 3 - for hardware-independent bugs; the GPU tests remain the parity gate."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def libs(tmp_path_factory):
    d = tmp_path_factory.mktemp("simt")
    emul, shim = str(d / "libdecode_emul.so"), str(d / "libdecode_shim.so")
    flags = ["g++", "-std=c++17", "-O1", "-U_FORTIFY_SOURCE", "-ffp-contract=off", "-Wno-unknown-pragmas", "-shared", "-fPIC",
             "-Wl,-Bsymbolic"]                                                   # see test_library_simt.py
    subprocess.run(flags + ["-o", emul, os.path.join(ROOT, "tests", "simt", "decode_emul.cc")], check=True)
    subprocess.run(flags + ["-o", shim, os.path.join(ROOT, "tests", "decode_host_shim.cc")], check=True)
    e, s = C.CDLL(emul), C.CDLL(shim)
    e.emul_new.restype = C.c_void_p
    e.emul_new.argtypes = [C.c_int]
    e.emul_free.argtypes = [C.c_void_p]
    e.emul_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p]
    s.shim_new.restype = C.c_void_p
    s.shim_step.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p]
    return e, s


def _traffic(n, seed, n_aircraft):
    """Position-heavy traffic of few aircraft with SMALL addresses (the emulated report table has 2^17 slots), several
    reports of one aircraft inside one 32-frame step, equal timestamps, an expiry gap, some other message types."""
    import decode_cases as dc
    from gr_air_modes_b200 import decode
    rng = np.random.default_rng(seed)
    craft = [(int(a), float(rng.uniform(-60, 60)), float(rng.uniform(-170, 170))) for a in rng.choice(np.arange(1, 1 << 15), n_aircraft, replace=False)]
    msgs, t = [], 0.0
    for k in range(n):
        aa, lat, lon = craft[int(rng.integers(0, n_aircraft))]
        r = rng.random()
        if r < 0.8:
            odd = int(rng.integers(0, 2))
            surface = rng.random() < 0.2
            la, lo = dc.cpr_encode(lat + 1e-4 * rng.standard_normal(), lon + 1e-4 * rng.standard_normal(), odd, surface)
            me = dc.me_surface(6, 10, 1, 5, odd, la, lo) if surface else dc.me_airborne(11, dc.enc_alt12(20000), odd, la, lo)
            frame, ecc = dc.df17(aa, me)
        elif r < 0.9:
            frame, ecc = dc.df17(aa, dc.me_ident(2, 3, "SIMT%d" % (k % 10)))
        else:
            frame, ecc = dc.short_frame(int(rng.choice([0, 4, 5, 11])), rng, aa)
        t += float(rng.choice([0.0, 1e-4, 0.05])) + (30.0 if k == n // 2 else 0.0)
        msgs.append((frame.hex(), ecc, int(t), t - int(t)))
    arr, _ = decode.frames_from_messages(msgs)
    return arr, msgs


def _run(e, s, arr, n, variant, warps, splits, loc):
    from gr_air_modes_b200 import decode
    have, lat, lon = (0, 0.0, 0.0) if loc is None else (1, loc[0], loc[1])
    he, hs = e.emul_new(17), s.shim_new()
    got = np.zeros(n, dtype=decode.FIELDS_DTYPE)
    want = np.zeros(n, dtype=decode.FIELDS_DTYPE)
    base = C.addressof(arr)
    pos = 0
    for c in splits + [n]:
        c = min(c, n - pos)
        if c <= 0:
            break
        fr = C.c_void_p(base + 80 * pos)
        assert e.emul_decode(he, fr, c, variant, warps, have, lat, lon, C.c_void_p(got.ctypes.data + 144 * pos)) == 0
        s.shim_step(hs, fr, c, have, lat, lon, C.c_void_p(want.ctypes.data + 144 * pos))
        pos += c
    e.emul_free(he)
    return got, want


@pytest.mark.parametrize("variant,warps", [(1, 4), (1, 12), (2, 4), (2, 8), (3, 0)])
def test_kernel_source_under_the_emulator_equals_sequential_replay(libs, variant, warps):
    e, s = libs
    n = 2500
    arr, msgs = _traffic(n, 40 + variant, 5)
    for splits in ([], [1, 31, 32, 33, 700]):
        got, want = _run(e, s, arr, n, variant, warps, splits, [40.0, -3.0])
        assert got.tobytes() == want.tobytes(), (variant, warps, splits)      # every byte of every record
    st = want["status"]
    assert ((st & 0x10) != 0).sum() > 1200 and ((st & 0x04) != 0).sum() > 5


def test_variant3_partition_across_tiles(libs):
    """More than one 8192-frame tile: the stable counting sort of variant 3 must keep stream order inside every bucket."""
    from oracle import decode_oracle as do
    e, s = libs
    n = 9000
    arr, msgs = _traffic(n, 77, 40)
    got, want = _run(e, s, arr, n, 3, 0, [8191], None)
    assert got.tobytes() == want.tobytes()
    orc = do.decode_batch(msgs, None)
    assert [w["status"] for w in orc] == want["status"].tolist()

"""The "%g" formatter of the jf_aligner coords lines (mrfmt::fmt_general, pacbio_b200/csrc/records_common.hpp),
shared by the host and the device printer, against glibc's printf("%g") across the whole double range."""
import ctypes as C
import os
import random
import struct

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def H():
    h = C.CDLL(os.path.join(ROOT, "pacbio_b200", "libmegareads_host.so"))
    h.mrh_general_format_pair.argtypes = [C.c_double, C.c_char_p, C.c_char_p]
    return h


def f(bits):
    return struct.unpack("<d", struct.pack("<Q", bits & 0xFFFFFFFFFFFFFFFF))[0]


def bits(x):
    return struct.unpack("<Q", struct.pack("<d", x))[0]


def check(H, xs):
    mine, libc = C.create_string_buffer(64), C.create_string_buffer(64)
    for x in xs:
        for v in (x, -x):
            assert H.mrh_general_format_pair(v, mine, libc), (repr(v), mine.value, libc.value)


def around(x):
    """x and its two neighbouring doubles"""
    b = bits(abs(x))
    return [x] + [f(b + d) for d in (-1, 1) if 0 < b + d < 0x7FF0000000000000]


def test_special_values(H):
    check(H, [0.0, float("inf"), float("nan"), f(0x7FF8000000000000 | (1 << 63)), f(0x7FF0000000000001),
              5e-324, 1e-323, 2.2250738585072014e-308, 2.225073858507201e-308, 1.7976931348623157e308])


def test_every_decade_and_the_values_that_round_across_it(H):
    """10^k for k in -323..308 with its neighbours, and the values just below a decade that round up into it
    (9.999995 10^k, the tie itself, and its neighbours)."""
    xs = []
    for k in range(-323, 309):
        for mant in ("1", "9.999995", "9.9999949999999", "9.99999500000001", "1.000005", "9.99999"):
            x = float(mant + "e%d" % k)
            if x != 0 and x != float("inf"):
                xs += around(x)
    check(H, xs)


def test_notation_boundaries(H):
    """X = -5 / -4 (0.0001 against 1e-05) and X = 5 / 6 (999999.5 against 1e+06), both sides."""
    xs = [1e-4, 1e-5, 9.999995e-05, 9.9999949e-05, 0.000099999, 0.00010000049, 999999.4, 999999.5, 999999.6, 100000.0,
          99999.95, 99999.949999, 123456.0, 1234567.0, 999999.0, 1e6, 0.5, 1.0, 10.0]
    check(H, [y for x in xs for y in around(x)])


def test_ties_at_the_sixth_digit(H):
    """Exact binary ties: ties go to the even digit, on the exact value (1234565 -> 1.23456e+06, 1234575 ->
    1.23458e+06)."""
    xs = [1234565.0, 1234575.0, 12345.25, 12345.75, 0.1234565, 2.5, 1.5, 100000.5, 999998.5, 999999.5, 1234565.0 * 2 ** 20]
    xs += [(2 * i + 1) * 0.5 for i in range(100000, 100400)]                 # 6-digit integers and a half
    xs += [(2 * i + 1) * 5.0 for i in range(100000, 100400)]                 # 7 digits ending in 5
    xs += [(2 * i + 1) * 0.5 ** 8 for i in range(12345 * 128, 12345 * 128 + 400)]
    check(H, xs)


def test_random_bit_patterns_and_coords_values(H):
    """About 10^5 random doubles over the whole range, and values of the size stretch, offset and avg_err take."""
    rng = random.Random(7)
    xs = [f(rng.getrandbits(64)) for _ in range(100000)]
    xs += [rng.uniform(0.5, 1.5) for _ in range(30000)]                     # stretch
    xs += [rng.uniform(-20000, 20000) for _ in range(30000)]                # offset
    xs += [rng.uniform(0, 10) for _ in range(30000)]                        # avg_err
    xs += [round(rng.uniform(-20000, 20000), rng.randrange(0, 7)) for _ in range(30000)]   # short decimals
    check(H, xs)

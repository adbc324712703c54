"""The pieces of the mega-read printer that the host and the device share (pacbio_b200/csrc/records_common.hpp),
checked on the CPU: the port of libstdc++'s std::sort that orders the tiling candidates on the device, and the
fixed-point number formatter of the record lines."""
import ctypes as C
import os
import random
import struct

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def H():
    h = C.CDLL(os.path.join(ROOT, "pacbio_b200", "libmegareads_host.so"))
    h.mrh_selftest_sort.restype = C.c_uint64
    h.mrh_selftest_sort.argtypes = [C.c_int, C.POINTER(C.c_double), C.c_uint64]
    h.mrh_fixed_format_pair.argtypes = [C.c_double, C.c_int, C.c_char_p, C.c_char_p]
    return h


def sort_mismatches(H, kind, keys):
    a = np.ascontiguousarray(keys, dtype=np.float64)
    return H.mrh_selftest_sort(kind, a.ctypes.data_as(C.POINTER(C.c_double)), len(a))


@pytest.mark.parametrize("kind", [0, 1, 2], ids=["greedy_lpath", "maximal_tiling_end", "weighted_weight"])
def test_sort_port_gives_the_permutation_of_std_sort(H, kind):
    """Same permutation as std::sort, ties included: every size 0-40 with keys of 1-4 distinct values, then random
    sizes up to 5000 (introsort, heap fallback and the final insertion sort all run there)."""
    rng = random.Random(1234 + kind)
    for n in range(41):
        for distinct in (1, 2, 3, 4):
            for _ in range(20):
                keys = [rng.randrange(distinct) * (0.5 if kind == 2 else 1) for _ in range(n)]
                assert sort_mismatches(H, kind, keys) == 0, (n, distinct, keys)
    for _ in range(300):
        n = rng.randrange(41, 5001)
        distinct = rng.randrange(1, 5)
        keys = [rng.randrange(distinct) for _ in range(n)]
        assert sort_mismatches(H, kind, keys) == 0, (n, distinct)
    # adversarial orders for the median of three: sorted, reversed, organ pipe
    for n in (17, 100, 1000, 4999):
        for keys in (list(range(n)), list(range(n, 0, -1)), [min(i, n - i) for i in range(n)]):
            assert sort_mismatches(H, kind, keys) == 0, n


def fixed_pair(H, x, d):
    mine, libc = C.create_string_buffer(400), C.create_string_buffer(400)
    same = H.mrh_fixed_format_pair(x, d, mine, libc)
    return bool(same), mine.value.decode(), libc.value.decode()


def test_fixed_formatter_prints_every_double_as_printf(H):
    """"%.2f" / "%.4f" of the shared formatter equal glibc's for huge values (the multi-word path), values around
    2^53 and 2^64 (the 128-bit path), subnormals, signed zeros, infinities and NaNs of both signs."""
    def f(bits):
        return struct.unpack("<d", struct.pack("<Q", bits))[0]
    xs = [0.0, -0.0, 1e11, 1e12, 1e15, 1e300, 1e308, 1.7976931348623157e308, 5e-324, 2.2250738585072014e-308,
          1e-310, float("inf"), float("-inf"), float("nan"), f(0xfff8000000000000), f(0x7ff0000000000001)]
    for e in (52, 53, 54, 63, 64, 65):
        for delta in (-2, -1, 0, 1, 2):
            xs.append(2.0 ** e + delta * 2.0 ** max(0, e - 52))
    e = 11.0
    while e <= 308:
        xs += [10 ** e, 1.5 * 10 ** e] if e < 308 else [10 ** e]
        e += 0.5
    rng = random.Random(5)
    for _ in range(20000):
        xs.append(f(rng.getrandbits(64)))
        xs.append(rng.uniform(1e11, 1e20))
        xs.append(2.0 ** rng.uniform(-1074, 1023))
    for x in xs:
        for v in (x, -x):
            for d in (2, 4):
                same, mine, libc = fixed_pair(H, v, d)
                assert same, (v, d, mine, libc)

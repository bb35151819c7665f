"""The exact-sum accumulator of the deposition profile (torj_jl_b200/csrc/torj_exactsum.cuh), checked on the CPU.

The header's pure functions are compiled with g++ and compared against an exact model in Python integers and fractions:
a booking v is the integer q = round_half_even(v * 2^160); a bin holds sum(q) exactly; its double is
float(Fraction(sum(q), 2^160)), which Python rounds correctly (nearest, ties to even)."""
import ctypes as C
import os
import random
import subprocess
from fractions import Fraction

import numpy as np
import pytest

from conftest import ROOT

CSRC = os.path.join(ROOT, "torj_jl_b200", "csrc")
SHIM = r"""
#include "torj_exactsum.cuh"
extern "C" {
int xs_split(double v, int* k, long long* d) {
    TorjXsSplit s = torj_xs_split(v);
    *k = s.k; d[0] = s.d[0]; d[1] = s.d[1]; d[2] = s.d[2];
    return s.ok;
}
// books v[i] for i in order[0..n) into w[8]; returns the number refused
long long xs_book_many(long long* w, const double* v, const long long* order, long long n) {
    long long bad = 0;
    for (long long i = 0; i < n; ++i) {
        TorjXsSplit s = torj_xs_split(v[order[i]]);
        if (s.ok) torj_xs_add(w, s); else ++bad;
    }
    return bad;
}
double xs_to_double(const long long* w) { return torj_xs_to_double(w); }
void xs_normalize(long long* w) { torj_xs_normalize(w); }
int xs_valid(long long bookings, long long refused) { return torj_xs_valid(bookings, refused); }
double xs_vmax(void) { return TORJ_XS_VMAX; }
long long xs_max_bookings(void) { return TORJ_XS_MAX_BOOKINGS; }
long long xs_buffer_words(long long n) { return (long long)torj_xs_buffer_words((size_t)n); }
}
"""
Q = 160
DIGIT = 28
NW = 8
TWO64 = 2.0 ** 64


@pytest.fixture(scope="module")
def xs(tmp_path_factory):
    d = tmp_path_factory.mktemp("exactsum")
    src = d / "shim.cpp"
    src.write_text(SHIM)
    so = str(d / "libexactsum.so")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-shared", "-fPIC", "-I" + CSRC, "-o", so,
                           str(src)])
    L = C.CDLL(so)
    i64p = np.ctypeslib.ndpointer(np.int64, flags="C")
    L.xs_split.argtypes, L.xs_split.restype = [C.c_double, C.POINTER(C.c_int), i64p], C.c_int
    L.xs_book_many.argtypes = [i64p, np.ctypeslib.ndpointer(np.float64, flags="C"), i64p, C.c_longlong]
    L.xs_book_many.restype = C.c_longlong
    L.xs_to_double.argtypes, L.xs_to_double.restype = [i64p], C.c_double
    L.xs_normalize.argtypes, L.xs_normalize.restype = [i64p], None
    L.xs_valid.argtypes, L.xs_valid.restype = [C.c_longlong, C.c_longlong], C.c_int
    L.xs_vmax.restype = C.c_double
    L.xs_max_bookings.restype = C.c_longlong
    L.xs_buffer_words.argtypes, L.xs_buffer_words.restype = [C.c_longlong], C.c_longlong
    return L


def quantize(v):
    """The model of one booking: v in quanta, rounded half to even."""
    return round(Fraction(v) * 2 ** Q)


def split(L, v):
    k = C.c_int(-1)
    d = np.zeros(3, dtype=np.int64)
    ok = L.xs_split(float(v), C.byref(k), d)
    return ok, k.value, [int(x) for x in d]


def book(L, vals, order=None):
    v = np.ascontiguousarray(vals, dtype=np.float64)
    o = np.arange(len(v), dtype=np.int64) if order is None else np.ascontiguousarray(order, dtype=np.int64)
    w = np.zeros(NW, dtype=np.int64)
    bad = L.xs_book_many(w, v, o, len(o))
    return w, bad


def words_value(w):
    return sum(int(x) << (DIGIT * k) for k, x in enumerate(w))


def random_doubles(rng, n, lo_exp=-215, hi_exp=63, signed=True):
    out = []
    for _ in range(n):
        e = rng.randint(lo_exp, hi_exp)
        m = rng.getrandbits(52) | (1 << 52)
        v = float(Fraction(m, 1 << 52) * Fraction(2) ** e)
        if signed and rng.random() < 0.5:
            v = -v
        out.append(v)
    return out


EDGES = [
    0.0, -0.0, 2.0 ** -Q, 2.0 ** -(Q + 1), 3 * 2.0 ** -(Q + 1), 5 * 2.0 ** -(Q + 1), 2.0 ** -(Q + 1) * (1 + 2.0 ** -52),
    5 * 2.0 ** -(Q + 2), 7 * 2.0 ** -(Q + 2), 2.0 ** -(Q + 54), 2.0 ** -(Q + 53), 2.0 ** -(Q + 53) * (1 + 2.0 ** -52),
    5e-324, 2.2250738585072014e-308, np.nextafter(TWO64, 0.0), 2.0 ** 63, 2.0 ** 40, 1.0, 0.5, 1.0 / 3.0,
    (2.0 ** 53 - 1) * 2.0 ** -(Q + 1), (2.0 ** 53 - 1) * 2.0 ** -(Q + 3),
] + [2.0 ** (DIGIT * k - Q + r) * (1 + 2.0 ** -52) for k in range(NW) for r in (-1, 0, 1, 27)]


def test_split_is_exact_over_the_range_and_at_the_edges(xs):
    rng = random.Random(1)
    vals = EDGES + [-v for v in EDGES] + random_doubles(rng, 20000)
    for v in vals:
        if not abs(v) < TWO64:
            continue
        ok, k, d = split(xs, v)
        assert ok == 1, v
        assert 0 <= k <= NW - 3
        assert all(abs(x) < 2 ** DIGIT for x in d), (v, d)
        assert all(x == 0 or (x < 0) == (v < 0) for x in d), (v, d)
        assert sum(x << (DIGIT * (k + j)) for j, x in enumerate(d)) == quantize(v), v


def test_split_rounds_half_even_below_the_quantum(xs):
    qt = 2.0 ** -Q
    for v, q in [(qt / 2, 0), (3 * qt / 2, 2), (5 * qt / 2, 2), (7 * qt / 2, 4), (qt / 2 * (1 + 2.0 ** -52), 1),
                 (5 * qt / 4, 1), (7 * qt / 4, 2), (qt / 4, 0), (2.0 ** -1074, 0)]:
        for s in (1, -1):
            ok, k, d = split(xs, s * v)
            assert ok == 1 and sum(x << (DIGIT * (k + j)) for j, x in enumerate(d)) == s * q, (v, d)


def test_values_beyond_the_range_are_refused(xs):
    assert xs.xs_vmax() == TWO64
    for v in (TWO64, -TWO64, 2.0 ** 70, -1e300, float("inf"), float("-inf"), float("nan")):
        ok, _, d = split(xs, v)
        assert ok == 0 and d == [0, 0, 0], v
    w, bad = book(xs, [1.0, float("nan"), TWO64, 2.0])
    assert bad == 2 and xs.xs_to_double(w) == 3.0


def test_sum_is_independent_of_the_order_with_carry_chains(xs):
    rng = random.Random(2)
    # digits of all ones: every add of the chain values carries through several words once normalised
    chain = [float((2 ** 53 - 1) * Fraction(2) ** (DIGIT * k - Q - 1)) for k in range(1, 6)] * 40
    vals = chain + random_doubles(rng, 3000, lo_exp=-170, hi_exp=40, signed=False) + EDGES[:14]
    exact = sum(quantize(v) for v in vals)
    ref, bad = book(xs, vals)
    assert bad == 0 and words_value(ref) == exact
    for _ in range(30):
        order = list(range(len(vals)))
        rng.shuffle(order)
        w, _ = book(xs, vals, order)
        assert np.array_equal(w, ref)
    n = ref.copy()
    xs.xs_normalize(n)
    assert words_value(n) == exact and all(0 <= int(x) < 2 ** DIGIT for x in n[:-1])


def test_conversion_is_correctly_rounded(xs):
    rng = random.Random(3)
    cases = []
    for _ in range(3000):  # random sums, some with heavy cancellation (signed bookings)
        cases.append(random_doubles(rng, rng.randint(1, 40), lo_exp=rng.randint(-215, 0), hi_exp=rng.randint(0, 63)))
    big = 2.0 ** 60
    u = 2.0 ** 8  # ulp of 2^60
    cases += [
        [big, u / 2],                      # tie: to even (down)
        [big, u / 2, 2.0 ** -Q],           # above the tie: up (sticky in a low word)
        [big, u, u / 2],                   # tie: to even (up)
        [big, -u / 4],                     # below: a borrow through every word
        [-big, -u / 2], [-big, -u, -u / 2],
        [1.0, 2.0 ** -53], [1.0, 2.0 ** -53, 2.0 ** -Q], [1.0, -2.0 ** -54], [1.0, -2.0 ** -54, -2.0 ** -Q],
        [2.0 ** -Q], [2.0 ** 63, 2.0 ** 63, 2.0 ** 63], [np.nextafter(TWO64, 0.0)] * 1000,
        [1.0, -1.0], [2.0 ** 40, -2.0 ** 40, 2.0 ** -150],
    ]
    for vals in cases:
        w, bad = book(xs, vals)
        assert bad == 0
        exact = sum(quantize(v) for v in vals)
        want = float(Fraction(exact, 2 ** Q))
        got = xs.xs_to_double(w)
        assert got == want and np.signbit(got) == np.signbit(want) or (got == 0.0 and want == 0.0), (vals[:4], got, want)


def test_booking_bound_and_buffer_layout(xs):
    nb = xs.xs_max_bookings()
    assert nb == 2 ** 34
    # headroom: nb adds of < 2^28 keep every word below 2^62, so the carries of the conversion cannot overflow
    assert nb * (2 ** DIGIT - 1) < 2 ** 62
    assert xs.xs_valid(nb, 0) == 1 and xs.xs_valid(nb + 1, 0) == 0 and xs.xs_valid(5, 1) == 0 and xs.xs_valid(0, 0) == 1
    assert xs.xs_buffer_words(10) == 10 * NW + 2
    # the extreme the bound allows: nb bookings of the largest value still convert exactly
    w = np.zeros(NW, dtype=np.int64)
    ok, k, d = split(xs, np.nextafter(TWO64, 0.0))
    for j in range(3):
        w[k + j] = d[j] * nb
    assert xs.xs_to_double(w) == float(Fraction(quantize(np.nextafter(TWO64, 0.0)) * nb, 2 ** Q))

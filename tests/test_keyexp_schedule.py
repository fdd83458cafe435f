"""Sliding windows over key-row exponents (csrc/keyexp.h) and the key-row slot orders that make them warp-uniform.

CPU: the recoder and the order builder are compiled for the host from the product header and checked directly; the merged
schedule the job kernels walk (sliding windows of base 0, 5-bit fixed windows of base 1 every fifth bit) is replayed on the
N-adic model of tests/test_nadic_model.py for the three folded job shapes of the GG20 driver and checked against `pow`,
together with the product count the kernels' work counters report.  GPU: offline batches whose sessions all use one key
row, and whose rows are interleaved, against the C twin of the oracle."""
import ctypes
import random
import subprocess

import numpy as np
import pytest

import __graft_entry__ as entry
from tests.test_nadic_model import Nadic

BITS, WINDOW = 6, 5          # KEYEXP_BITS, WINDOW_BITS

SHIM = r"""
#include "keyexp.h"
using namespace tecdsa;
extern "C" {
int k_recode(const uint32_t* e, int bits, int* lo, uint32_t* digit) {
    int n = 0;
    for (int top = keyexp_top(e, bits - 1); top >= 0; n++) { lo[n] = keyexp_window(e, top, digit[n]); top = keyexp_top(e, lo[n] - 1); }
    return n;
}
int k_count(const uint32_t* e, int bits, int* first_lo) { return keyexp_count(e, bits, *first_lo); }
size_t k_order(const uint32_t* rows, size_t units, uint32_t nrows, size_t pad, uint32_t* order) {
    uint32_t* count = new uint32_t[nrows];
    size_t n = keyexp_order(rows, units, nrows, pad, count, order);
    delete[] count;
    return n;
}
}
"""


@pytest.fixture(scope="module")
def kx(tmp_path_factory):
    d = tmp_path_factory.mktemp("keyexp")
    src, so = d / "shim.cpp", d / "libkeyexp.so"
    src.write_text(SHIM)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-I", entry.CSRC, "-shared", "-fPIC", "-o", str(so), str(src)])
    lib = ctypes.CDLL(str(so))
    lib.k_order.restype = ctypes.c_size_t
    return lib


def _limbs(v, limbs):
    return np.frombuffer(int(v).to_bytes(4 * limbs, "little"), dtype=np.uint32).copy()


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def recode(kx, e, limbs):
    bits = 32 * limbs
    lo, dg = np.zeros(bits, np.int32), np.zeros(bits, np.uint32)
    n = kx.k_recode(_ptr(_limbs(e, limbs)), bits, _ptr(lo), _ptr(dg))
    return [(int(lo[j]), int(dg[j])) for j in range(n)]


def _key_exponents():
    """(exponent, limbs) of the seven key tables of every golden key row: N, p, q, p-1, q-1, q mod (p-1), p mod (q-1)"""
    from tests.golden import fixtures
    out = []
    for keys in fixtures.load_all_keysets():
        for k in keys:
            p, q = k.dk.p, k.dk.q
            out += [(p * q, 64), (p, 32), (q, 32), (p - 1, 32), (q - 1, 32), (q % (p - 1), 32), (p % (q - 1), 32)]
    return out


EDGE = [(1, 1), (0xFFFFFFFF, 1), (1 << 31, 1), ((1 << 2048) - 1, 64), (1 << 2047, 64), ((1 << 2047) | 1, 64),
        (0x21, 1), (0x41, 1), ((1 << 37) - 1, 2), (sum(1 << (7 * j) for j in range(146)), 32), (0b101 << 1019, 32)]


@pytest.mark.parametrize("which", ["golden", "edge"])
def test_recoding_reproduces_exponent_within_bound(kx, which):
    cases = _key_exponents() if which == "golden" else EDGE
    assert which == "edge" or len(cases) == 24 * 7
    for e, limbs in cases:
        sched = recode(kx, e, limbs)
        assert sum(d << lo for lo, d in sched) == e
        assert all(d & 1 and d < 1 << BITS for _, d in sched)
        tops = [lo + d.bit_length() - 1 for lo, d in sched]
        assert all(a - b >= BITS for a, b in zip(tops, tops[1:]))       # windows start at least BITS bits apart
        assert len(sched) <= -(-e.bit_length() // BITS)
        first_lo = ctypes.c_int(0)
        assert kx.k_count(_ptr(_limbs(e, limbs)), 32 * limbs, ctypes.byref(first_lo)) == len(sched)
        assert first_lo.value == (sched[0][0] if sched else -1)
    assert recode(kx, 0, 2) == []


def straus_keyexp(A, kx, x, e_key, key_limbs, y=None, e1=None, e1_limbs=8, muls=()):
    """nadic_jobs_kernel on a keyexp class: lift, odd-power table of x, 5-bit table of y, merged loop, multipliers, exit.
    Returns (value, products, squarings) with products = table + window products (the lifts and the exit are not counted)."""
    k = A.bits // 32
    X = A.lift(x, 2 * k)
    x2 = A.mul(X, X, cross2=True)
    odd = [X]
    for _ in range(2 ** (BITS - 1) - 1):
        odd.append(A.mul(odd[-1], x2, cross2=True))
    products, squarings = 2 ** (BITS - 1), 0
    nw1 = 0
    if y is not None:
        Y = A.lift(y, 2 * k)
        tbl1 = [A.one, Y]
        for _ in range(2 ** WINDOW - 2):
            tbl1.append(A.mul(tbl1[-1], Y, cross2=True))
        products += 2 ** WINDOW - 2
        nw1 = -(-32 * e1_limbs // WINDOW)
    sched = dict(recode(kx, e_key, key_limbs))
    p = max(max(sched) if sched else -1, (nw1 - 1) * WINDOW)
    acc, first = A.one, True
    while p >= 0:
        if not first:
            acc = A.sqr(acc)
            squarings += 1
        first = False
        if p in sched:
            acc = A.mul(acc, odd[sched[p] >> 1], cross2=True)
            products += 1
        if p % WINDOW == 0 and p // WINDOW < nw1:
            acc = A.mul(acc, tbl1[(e1 >> p) & (2 ** WINDOW - 1)], cross2=True)
            products += 1
        p -= 1
    for m in muls:
        acc = A.mul(acc, A.lift(m, 2 * k), cross2=True)
    return A.plain(acc), products, squarings


def fixed_windows(A, c, e, muls, e_limbs=8):
    """the fixed-window loop of one base (nadic_jobs_kernel without keyexp), then the multipliers"""
    k = A.bits // 32
    C = A.lift(c, 2 * k)
    tbl = [A.one, C]
    for _ in range(2 ** WINDOW - 2):
        tbl.append(A.mul(tbl[-1], C, cross2=True))
    acc, nw = A.one, -(-32 * e_limbs // WINDOW)
    for w in reversed(range(nw)):
        if w < nw - 1:
            for _ in range(WINDOW):
                acc = A.sqr(acc)
        acc = A.mul(acc, tbl[(e >> (WINDOW * w)) & (2 ** WINDOW - 1)], cross2=True)
    for m in muls:
        acc = A.mul(acc, A.lift(m, 2 * k), cross2=True)
    return A.plain(acc)


def _kernel_products(kx, e_key, key_limbs, e1_limbs=None):
    """the product count of the kernels' work counter for a keyexp class (nadic.cuh / jobs.cuh): 32 table products, one per
    window, 30 table products and one per 5-bit window for base 1, and max(first window, top 5-bit window) squarings"""
    first_lo = ctypes.c_int(0)
    nwin = kx.k_count(_ptr(_limbs(e_key, key_limbs)), 32 * key_limbs, ctypes.byref(first_lo))
    products = 2 ** (BITS - 1) + nwin
    top = first_lo.value
    if e1_limbs:
        nw1 = -(-32 * e1_limbs // WINDOW)
        products += 2 ** WINDOW - 2 + nw1
        top = max(top, (nw1 - 1) * WINDOW)
    return products, max(top, 0)


@pytest.mark.parametrize("shape", ["UV", "VU21", "VU20", "p-adic", "edge"])
def test_merged_schedule_against_pow(kx, shape):
    """UV / VU21: s^N * (c^-1)^e * m mod N^2, N the prover's key exponent (sliding windows), e a 256-bit challenge (5-bit
    windows); VU20: (c^-1)^e * m1 * m2 with the 5-bit windows alone (no key exponent: the fixed-window loop); p-adic:
    b^p and b^(p-1) mod p^2; edge: extreme key exponents merged with a 5-bit base"""
    from tests.golden import fixtures
    rng = random.Random(sum(map(ord, shape)))
    keys = fixtures.load_keyset(rng.randrange(8))
    k = keys[rng.randrange(3)]
    p, q = k.dk.p, k.dk.q
    n = p * q
    if shape in ("UV", "VU21", "VU20"):
        A = Nadic(n, 64)
        nn = n * n
        s, c, m1, m2, e = rng.randrange(n), rng.randrange(nn), rng.randrange(nn), rng.randrange(nn), rng.getrandbits(256)
        if shape == "VU20":
            assert fixed_windows(A, c, e, (m1, m2)) == pow(c, e, nn) * m1 * m2 % nn
            return
        got, prods, sq = straus_keyexp(A, kx, s, n, 64, c, e, 8, (m1,))
        assert got == pow(s, n, nn) * pow(c, e, nn) * m1 % nn
        assert (prods, sq) == _kernel_products(kx, n, 64, 8)
    elif shape == "p-adic":
        A = Nadic(p, 32)
        b = rng.randrange(p * p)
        for ex in (p, p - 1):
            got, prods, sq = straus_keyexp(A, kx, b, ex, 32)
            assert got == pow(b, ex, p * p)
            assert (prods, sq) == _kernel_products(kx, ex, 32)
    else:
        A = Nadic((1 << 1024) - 105, 32)
        for ex in (1, 2, 63, 64, 1 << 1023, (1 << 1024) - 1):
            b = rng.getrandbits(2048)
            y, nn = rng.getrandbits(2048), A.n ** 2
            got, prods, sq = straus_keyexp(A, kx, b, ex, 32, y, 7, 1)
            assert got == pow(b, ex, nn) * pow(y, 7, nn) % nn
            assert (prods, sq) == _kernel_products(kx, ex, 32, 1)
            got, prods, sq = straus_keyexp(A, kx, b, ex, 32)
            assert got == pow(b, ex, nn)
            assert (prods, sq) == _kernel_products(kx, ex, 32)


def _sessions(n, n_keysets, seed):
    rng = np.random.default_rng(seed)
    pairs = [(0, 1), (0, 2), (1, 2), (1, 0), (2, 0), (2, 1)]
    pr = rng.integers(0, 6, size=n)
    s = np.zeros((n, 3), np.uint32)
    s[:, 0] = rng.integers(0, n_keysets, size=n)
    s[:, 1] = [pairs[i][0] for i in pr]
    s[:, 2] = [pairs[i][1] for i in pr]
    return s


@pytest.mark.parametrize("n,n_keysets,pad", [(8192, 8, 8), (4096, 8, 4), (3, 8, 8), (1000, 1, 16), (5, 2, 8)])
def test_key_row_orders(kx, n, n_keysets, pad):
    """offline_impl's two orders (by own and by peer key row) on session tables drawn like gg20.synthetic_batch's"""
    s = _sessions(n, n_keysets, n * 7 + pad)
    U = 2 * n
    a, b = s[:, 1].astype(np.int64), s[:, 2].astype(np.int64)
    own = np.empty(U, np.uint32)
    own[0::2] = s[:, 0] * 3 + a
    own[1::2] = s[:, 0] * 3 + b
    peer = np.empty(U, np.uint32)
    peer[0::2] = own[1::2]
    peer[1::2] = own[0::2]
    nrows = 3 * n_keysets
    cap = U + min(nrows, U) * (pad - 1)
    for rows in (own, peer):
        order = np.zeros(cap, np.uint32)
        m = kx.k_order(_ptr(rows), U, nrows, pad, _ptr(order))
        assert m % pad == 0 and m <= cap
        o = order[:m]
        live = o[o < 0x80000000]
        assert sorted(live.tolist()) == list(range(U))                    # every unit exactly once
        assert np.all(np.diff(rows[live].astype(np.int64)) >= 0)          # sorted by row, stable
        for r in np.unique(rows):
            assert np.all(np.diff(live[rows[live] == r].astype(np.int64)) > 0)
        for w in range(0, m, pad):                                        # every warp-sized run names units of one key row
            run = o[w:w + pad] & 0x7FFFFFFF
            assert np.all(run < U) and len(set(rows[run].tolist())) == 1
        for g in (4, 8, 16):                                              # smaller warps of the same order as well
            if g <= pad:
                assert all(len(set(rows[o[w:w + g] & 0x7FFFFFFF].tolist())) == 1 for w in range(0, m, g))
        assert m - U <= len(np.unique(rows)) * (pad - 1)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["one_row", "interleaved"])
def test_offline_key_row_layouts_vs_twin(engine, pkg, layout):
    """key-uniform warps from the slot orders: a batch on one key row (every warp of an ordered class on the same schedule,
    runs padded at the end) and one whose rows alternate unit by unit, both equal to the C twin"""
    from mpecdsa_b200 import gg20
    from oracle import twin
    from tests.golden import fixtures
    keysets = fixtures.load_all_keysets()
    ks = gg20.KeySets(engine, keysets)
    n = 37
    sessions, rnd = gg20.synthetic_batch(keysets, n, 0xB2000011)
    if layout == "one_row":
        sessions[:, 0], sessions[:, 1], sessions[:, 2] = 3, 2, 0
    else:
        pairs = [(0, 1), (1, 2), (2, 0), (1, 0), (2, 1), (0, 2)]
        for i in range(n):
            sessions[i] = (i % 8, *pairs[i % 6])
    res = gg20.offline_batch(engine, ks, sessions, rnd)
    want = twin.offline_batch(twin.KeyTables(keysets), sessions, rnd, 8)
    ks.free()
    assert not want.status.any() and not np.asarray(res.status).any()
    assert np.array_equal(res.R, want.R) and np.array_equal(res.sigma, want.sigma) and np.array_equal(res.digest, want.digest)

"""The guarded fast paths of csrc/rt_device.cuh (shared reciprocal, one range test per normalisation, slow paths out of
line) against the plain __fdiv_rn / __fsqrt_rn code they replace, bit for bit.

GPU: every float32 bit pattern as numerator against divisors that straddle the guard's edges, every bit pattern as a
square-root argument, seeded and built 3-vectors, and sphere roots (rt_debug_exact_fastpath of lib/librt_b200_check.so).
CPU: the division guard, read from the header, accepts no exponent pair whose quotient or residual could leave the
normal range.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
HDR = os.path.join(ROOT, "ray-tracer-s8_b200", "csrc", "rt_device.cuh")
CHECK_LIB = os.path.join(ROOT, "ray-tracer-s8_b200", "lib", "librt_b200_check.so")


def _const(name):
    src = open(HDR).read()
    m = re.search(name + r"\s*=\s*([^,;]+)[,;]", src)
    expr = m.group(1).replace("u", "")
    return int(eval(expr, {}))  # e.g. "(125 << 24) - 1"


def _guard():
    lo, span = _const("X_DIV_LO"), _const("X_DIV_SPAN")
    l2lo, l2span = _const("X_LEN2_LO"), _const("X_LEN2_SPAN")

    def mag(bits):  # x_div_mag on a bit pattern
        return ((bits << 1) - lo) & 0xFFFFFFFF <= span

    def len2(bits):
        return (bits - l2lo) & 0xFFFFFFFF <= l2span

    return mag, len2


def test_division_guard_is_conservative():
    mag, len2 = _guard()
    accepted = 0
    for ea in range(256):
        for eb in range(256):
            pats_a = [(ea << 23) | m for m in (0, 0x7FFFFF)]
            pats_b = [(eb << 23) | m for m in (0, 0x7FFFFF)]
            ok_a = [mag(p) for p in pats_a]
            ok_b = [mag(p) for p in pats_b]
            assert ok_a[0] == ok_a[1] and ok_b[0] == ok_b[1]  # the test depends on the exponent field only
            if not (ok_a[0] and ok_b[0]):
                continue
            accepted += 1
            assert 1 <= ea <= 254 and 1 <= eb <= 254
            # |a| in [2^(ea-127), 2^(ea-126)), |b| likewise: the quotient's range, with the refinement's 1-ulp slack
            q_lo = (ea - 127) - (eb - 126)
            q_hi = (ea - 126) - (eb - 127)
            assert q_lo - 1 >= -126, (ea, eb)  # the quotient stays normal
            assert q_hi + 1 <= 127, (ea, eb)  # and finite
            # t = a - b*q is a multiple of ulp(b)*ulp(q) >= 2^(ea-127-47): zero or normal
            assert (ea - 127) - 47 >= -126, (ea, eb)
            assert (254 - eb) >= 1 and (254 - eb) <= 254  # 1/b is normal
    assert accepted == 125 * 125
    # a squared length that passes x_len2_domain has its square root (the divisor) inside the division domain
    for e in range(256):
        if len2(e << 23) or len2((e << 23) | 0x7FFFFF):
            assert 27 <= e <= 226
            el = (e - 127) // 2 + 127  # exponent field of sqrt, rounded down; sqrt(2^k * 1.99..) < 2^(k/2 + 1)
            assert mag(el << 23) and mag(min(el + 1, 255) << 23)


def _divisors():
    d = []
    for e in (1, 2, 26, 27, 63, 64, 65, 66, 100, 126, 127, 128, 150, 188, 189, 190, 191, 226, 227, 253, 254):
        for m in (0, 1, 0x400000, 0x7FFFFE, 0x7FFFFF):
            for s in (0, 1):
                d.append((s << 31) | (e << 23) | m)
    d += [0, 0x80000000, 1, 0x7FFFFF, 0x80000001, 0x7F800000, 0xFF800000, 0x7FC00000, 0xFFC00000]
    f = np.array(d, dtype=np.uint32).view(np.float32)
    extra = np.array([1.0, 3.0, 0.1, 7.0, 1000.0, 639.0, 359.0, 3839.0, 2159.0, 1.0 / 3.0, 1.7320508, 16.0],
                     dtype=np.float32)
    rng = np.random.default_rng(7)
    rnd = rng.uniform(-100.0, 100.0, 20).astype(np.float32)
    return np.concatenate([f, extra, rnd]).astype(np.float32)


def _vectors():
    rng = np.random.default_rng(11)
    bits = rng.integers(0, 2 ** 32, size=(200_000, 3), dtype=np.uint64).astype(np.uint32)
    whole = bits.view(np.float32)
    # components over the whole exponent range, finite
    e = rng.integers(0, 255, size=(200_000, 3)).astype(np.uint32)
    m = rng.integers(0, 2 ** 23, size=(200_000, 3)).astype(np.uint32)
    s = rng.integers(0, 2, size=(200_000, 3)).astype(np.uint32)
    finite = ((s << 31) | (e << 23) | m).view(np.float32)
    usual = rng.normal(size=(200_000, 3)).astype(np.float32)
    mixed = usual * np.float32(2.0) ** rng.integers(-70, 70, size=(200_000, 1)).astype(np.float32)
    special = [0.0, -0.0, 1e-45, -1e-45, 1e-40, 1.1754942e-38, 1e-30, 1e-20, 1.0, -1.0, 0.5, 3e19, 1e20, 1e30, 3.4e38,
               np.inf, -np.inf, np.nan]
    grid = np.array(np.meshgrid(special, special, special), dtype=np.float32).reshape(3, -1).T
    axis = np.zeros((6, 3), np.float32)
    for i in range(3):
        axis[2 * i, i], axis[2 * i + 1, i] = 1.0, -2.5
    return np.ascontiguousarray(np.concatenate([whole, finite, usual, mixed, grid, axis]).astype(np.float32))


def _spheres():
    rng = np.random.default_rng(13)
    n = 300_000
    d = rng.normal(size=(n, 3)).astype(np.float64)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    oc = rng.normal(size=(n, 3)) * (10.0 ** rng.uniform(-3, 3, size=(n, 1)))
    r = np.abs(rng.normal(size=n)) * 10.0 ** rng.uniform(-2, 2, size=n)
    # a third of the origins on their sphere (a ray leaving the surface tests its own sphere: c is near zero)
    k = n // 3
    oc[:k] = oc[:k] / np.linalg.norm(oc[:k], axis=1, keepdims=True) * r[:k, None]
    rec = np.concatenate([d, oc, (r * r)[:, None]], axis=1).astype(np.float32)
    edge = np.array([[0, 0, 1, 0, 0, 0, 1], [1, 0, 0, -5, 0, 0, 0], [0, 1, 0, 0, -1e30, 0, 1], [0, 0, 1, 0, 0, -1e-30, 1],
                     [0, 0, 1, np.nan, 0, 0, 1], [0, 0, -1, 0, 0, np.inf, 1], [0.6, 0.8, 0, 3, 4, 0, 25],
                     [1, 0, 0, -1e20, 0, 0, 1e30]], dtype=np.float32)
    return np.ascontiguousarray(np.concatenate([rec, edge]).astype(np.float32))


@pytest.mark.gpu
def test_fast_paths_match_ieee_bit_for_bit():
    L = C.CDLL(CHECK_LIB)
    f = L.rt_debug_exact_fastpath
    fp = C.POINTER(C.c_float)
    f.argtypes = [fp, C.c_uint32, fp, C.c_uint32, fp, C.c_uint32, C.POINTER(C.c_uint64)]
    f.restype = C.c_int
    div, vec, sph = _divisors(), _vectors(), _spheres()
    out = (C.c_uint64 * 3)()
    st = f(div.ctypes.data_as(fp), len(div), vec.ctypes.data_as(fp), len(vec), sph.ctypes.data_as(fp), len(sph), out)
    assert st == 0, st
    print(f"divisors {len(div)} vectors {len(vec)} spheres {len(sph)} in-domain pairs {out[2]} "
          f"mismatches scalar {out[0]} vector/sphere {out[1]}")
    assert out[2] > 100 * 2 ** 31  # most of the divisors are inside the domain
    assert out[0] == 0
    assert out[1] == 0

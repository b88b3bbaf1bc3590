"""CPU tier: the lazily reduced Fp12 product (tower.cuh: fp4_mul_redc, fp12_mul_assign), compiled for the host from the
device source (tests/hostsim/lazy_fp12_mul.cu).  Values are passed as RAW Montgomery limbs so that every stated bound
can be hit exactly; the host build aborts if an Fp4 output reaches 2^256 or a lin9_reduce input reaches 2^262."""
import ctypes
import os
import random
import subprocess

import pytest

from oracle import bn254_py as o

HERE = os.path.dirname(os.path.abspath(__file__))
P = o.P
R = 1 << 256
RINV = pow(R, -1, P)
PINV = pow(P, -1, R)


@pytest.fixture(scope="module")
def lz(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("lazy_fp12_mul") / "liblazy_fp12_mul.so")
    subprocess.check_call(["nvcc", "-x", "cu", "-O2", "-std=c++17", "-DSYLOW_HOSTSIM", "-shared", "-Xcompiler", "-fPIC",
                           "-w", "-o", so, os.path.join(HERE, "hostsim", "lazy_fp12_mul.cu")])
    return ctypes.CDLL(so)


def _words(vals):
    out = (ctypes.c_uint32 * (8 * len(vals)))()
    for i, v in enumerate(vals):
        out[8 * i: 8 * i + 8] = [(v >> (32 * k)) & 0xffffffff for k in range(8)]
    return out


def _ints(ws, n):
    return [sum(int(ws[8 * i + k]) << (32 * k) for k in range(8)) for i in range(n)]


def _fp4_exact(x0, x1, y0, y1):
    """The four accumulators of fp4_mul_redc before reduction: C0 = X0 Y0 + xi X1 Y1, C1 = X0 Y1 + X1 Y0 over the
    integers, with the lifts the routine adds (12 p^2, p^2, 2 p^2, 0)."""
    def mul(a, b):
        return a[0] * b[0] - a[1] * b[1], a[0] * b[1] + a[1] * b[0]
    p, q = mul(x0, y0), mul(x1, y1)
    a, b = mul(x0, y1), mul(x1, y0)
    return [p[0] + 9 * q[0] - q[1] + 12 * P * P, p[1] + q[0] + 9 * q[1] + P * P,
            a[0] + b[0] + 2 * P * P, a[1] + b[1]]


EDGE = [0, 1, 2, P - 1, P - 2, (P - 1) // 2, (P + 1) // 2, 1 << 253, (1 << 254) - 1 - (1 << 200)]
EDGE = [e for e in EDGE if e < P]


def test_fp4_mul_redc_exact_at_bounds(lz):
    """Every output is exactly the Montgomery reduction (A + M p) / R of its accumulator, for operands drawn from the
    extremes of the raw limb range (all p - 1 reaches the largest accumulators) and random ones."""
    rng = random.Random(44)
    sets = [[P - 1] * 8, [0] * 8, [P - 1, 0] * 4, [0, P - 1] * 4, [P - 1] * 4 + [0] * 4, [0] * 4 + [P - 1] * 4]
    sets += [[P - 1 if (m >> k) & 1 else 0 for k in range(8)] for m in range(256)]
    sets += [[rng.choice(EDGE) for _ in range(8)] for _ in range(400)]
    sets += [[rng.randrange(P) for _ in range(8)] for _ in range(200)]
    for v in sets:
        got = _ints(_call4(lz, v), 4)
        x0, x1, y0, y1 = (v[0], v[1]), (v[2], v[3]), (v[4], v[5]), (v[6], v[7])
        for g, A in zip(got, _fp4_exact(x0, x1, y0, y1)):
            assert 0 <= A < 22 * P * P
            M = (-A * PINV) % R
            assert g == (A + M * P) // R, v
        assert max(got[:2]) < 5.16 * P and max(got[2:]) < 1.76 * P


def _call4(lz, v):
    out = (ctypes.c_uint32 * 32)()
    lz.hs_fp4_mul_redc(_words(v), out)
    return out


def test_fp12_mul_assign_against_oracle(lz):
    """a <- a b and a <- a conj(b) on ANY Fp12 values: all-zero and all-(p - 1) raw coefficients, mixtures of the two,
    other edge coefficients and random values, against the oracle's Fp12 product."""
    rng = random.Random(1212)
    pats = [[0] * 12, [P - 1] * 12, [P - 1, 0] * 6, [0, P - 1] * 6, [P - 1] * 6 + [0] * 6, [0] * 6 + [P - 1] * 6]
    pairs = [(x, y) for x in pats for y in pats]
    pairs += [([rng.choice([0, P - 1]) for _ in range(12)], [rng.choice([0, P - 1]) for _ in range(12)])
              for _ in range(100)]
    pairs += [([rng.choice(EDGE) for _ in range(12)], [rng.choice(EDGE) for _ in range(12)]) for _ in range(100)]
    pairs += [([rng.randrange(P) for _ in range(12)], [rng.randrange(P) for _ in range(12)]) for _ in range(100)]
    for ra, rb in pairs:
        fa = o.fp12_from_list([c * RINV % P for c in ra])
        fb = o.fp12_from_list([c * RINV % P for c in rb])
        for conj in (0, 1):
            out = (ctypes.c_uint32 * 96)()
            lz.hs_fp12_mul_assign(_words(ra), _words(rb), conj, out)
            want = o.fp12_mul(fa, o.fp12_conj(fb) if conj else fb)
            assert _ints(out, 12) == [c * R % P for c in o.fp12_to_list(want)], (ra, rb, conj)

"""CPU tier: the lazily reduced Granger-Scott squaring (pairing.cuh: gs_fp4_square) and the reduction of its 17-limb
accumulators (fp.cuh: fp_redc_acc, lin9_reduce), compiled for the host from the device source (tests/hostsim/lazy_fp4.cu).
Values are passed as RAW Montgomery limbs so that every stated bound can be hit exactly; the host build aborts if a
lin9_reduce input reaches 2^262 or its remainder reaches 2p."""
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
    so = str(tmp_path_factory.mktemp("lazy_fp4") / "liblazy_fp4.so")
    subprocess.check_call(["nvcc", "-x", "cu", "-O2", "-std=c++17", "-DSYLOW_HOSTSIM", "-shared", "-Xcompiler", "-fPIC",
                           "-w", "-o", so, os.path.join(HERE, "hostsim", "lazy_fp4.cu")])
    return ctypes.CDLL(so)


def _words(v, n):
    return (ctypes.c_uint32 * n)(*[(v >> (32 * i)) & 0xffffffff for i in range(n)])


def _int(ws):
    return sum(int(x) << (32 * i) for i, x in enumerate(ws))


def _call(fn, n_out, *args):
    out = (ctypes.c_uint32 * n_out)()
    fn(*args, out)
    return out


# ------------------------------------------------------------------------------------------ the two reductions
def test_redc_acc_exact(lz):
    """V = (A + M p) / R with M = -A p^-1 mod R, for accumulators up to the largest the squaring forms (45.3 p^2 < 2^513)
    and the 17-limb edges below 2^262 R."""
    rng = random.Random(17)
    top = 4 * P * P + 9 * 4 * P * P + P * R  # A0's bound: S_a + 9 S_b + p R
    cases = [0, 1, R - 1, R, P * R, P * R - 1, top - 1, top, (1 << 513) - 1, (1 << 512), (1 << 512) - 1,
             (1 << 261) * R - 1]
    cases += [k * P * R + d for k in (1, 2, 9, 27) for d in (-1, 0, 1)]
    cases += [rng.randrange(top) for _ in range(2000)] + [rng.randrange((1 << 261) * R) for _ in range(200)]
    for A in cases:
        V = _int(_call(lz.hs_redc_acc, 9, _words(A, 17)))
        M = (-A * PINV) % R
        assert V == (A + M * P) // R, hex(A)
        assert V % P == A * RINV % P


def test_lin9_reduce_quotient_edges(lz):
    """T mod p for every k p - 1, k p, k p + 1 below 2^262 (k up to 338) and the container's extremes: the quotient estimate
    from the top 32 bits may be one short, never more."""
    rng = random.Random(262)
    cases = [0, 1, P - 1, P, (1 << 256) - 1, 1 << 256, (1 << 262) - 1, (1 << 261), (1 << 262) - P]
    for k in range(1, 340):
        for d in (-2, -1, 0, 1, 2):
            T = k * P + d
            if 0 <= T < (1 << 262):
                cases.append(T)
    cases += [rng.randrange(1 << 262) for _ in range(5000)]
    for T in cases:
        assert _int(_call(lz.hs_lin9_reduce, 8, _words(T, 9))) == T % P, hex(T)


# ------------------------------------------------------------------------------------------ the squaring
def _fp2_raw(a):
    return [a[0] * RINV % P, a[1] * RINV % P]


def _to_raw(a):
    return tuple(c * R % P for c in a)


def _gs_expected(a, b, x, y, xi):
    """x <- 3 A - 2 x, y <- 3 B + 2 y (3 xi B + 2 y) with (A, B) the Fp4 square of (a, b), all on raw Montgomery limbs."""
    a, b, x, y = (tuple(_fp2_raw(v)) for v in (a, b, x, y))
    t0, t1 = o._fp4_square(a, b)
    if xi:
        t1 = o.fp2_residue_mul(t1)
    nx = o.fp2_sub(o.fp2_scale(t0, 3), o.fp2_scale(x, 2))
    ny = o.fp2_add(o.fp2_scale(t1, 3), o.fp2_scale(y, 2))
    return _to_raw(nx) + _to_raw(ny)


def test_gs_fp4_square_at_bounds(lz):
    """One Fp4 squaring with every input coefficient drawn from the extremes of the raw limb range (0, 1, p - 1, ...),
    both forms (plain and times xi): the accumulators and lin9_reduce inputs reach their stated maxima here."""
    rng = random.Random(4)
    edge = [0, 1, 2, P - 1, P - 2, (P - 1) // 2, (P + 1) // 2, (1 << 253), (1 << 254) - 1 - (1 << 200)]
    edge = [e for e in edge if e < P]
    sets = [[P - 1] * 8, [0] * 8, [P - 1, 0] * 4, [0, P - 1] * 4, [P - 1] * 4 + [0] * 4, [0] * 4 + [P - 1] * 4]
    sets += [[rng.choice(edge) for _ in range(8)] for _ in range(400)]
    sets += [[rng.randrange(P) for _ in range(8)] for _ in range(200)]
    for v in sets:
        a, b, x, y = (v[0], v[1]), (v[2], v[3]), (v[4], v[5]), (v[6], v[7])
        words = (ctypes.c_uint32 * 64)()
        for i, c in enumerate(v):
            words[8 * i: 8 * i + 8] = list(_words(c, 8))
        for xi in (0, 1):
            out = _call(lz.hs_gs_fp4_square, 32, words, xi)
            got = tuple(_int(out[8 * i: 8 * i + 8]) for i in range(4))
            assert got == _gs_expected(a, b, x, y, xi), (v, xi)


def test_cyclotomic_square_arbitrary_fp12(lz):
    """The in-place squaring on ANY Fp12 (not only cyclotomic values) equals the oracle's Granger-Scott formula: all-zero
    and all-(p - 1) raw coefficients, alternating extremes, and random values."""
    rng = random.Random(12)
    cases = [[0] * 12, [P - 1] * 12, [P - 1, 0] * 6, [0, P - 1] * 6, [P - 1] * 6 + [0] * 6, [1] * 12]
    cases += [[rng.choice([0, 1, P - 1, P - 2]) for _ in range(12)] for _ in range(100)]
    cases += [[rng.randrange(P) for _ in range(12)] for _ in range(100)]
    for raw in cases:
        words = (ctypes.c_uint32 * 96)()
        for i, c in enumerate(raw):
            words[8 * i: 8 * i + 8] = list(_words(c, 8))
        out = _call(lz.hs_cyclotomic_square, 96, words)
        got = [_int(out[8 * i: 8 * i + 8]) for i in range(12)]
        f = o.fp12_from_list([c * RINV % P for c in raw])
        assert got == [c * R % P for c in o.fp12_to_list(o.cyclotomic_squared(f))], raw

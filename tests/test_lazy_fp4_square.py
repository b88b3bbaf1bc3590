"""CPU tier: the lazily reduced Granger-Scott squaring (pairing.cuh: gs_fp4_square) and the reduction of its 17-limb
accumulators (fp.cuh: fp_redc_acc, lin9_reduce), compiled for the host from the device source (tests/hostsim/lazy_fp4.cu).
Values are passed as RAW Montgomery limbs so that every stated bound can be hit exactly; the host build aborts if a
lin9_reduce input reaches 2^262 or its remainder reaches 2p.  The case lists live in tests/bound_cases.py, shared with
the device build of the same functions (test_gpu_device_bounds.py)."""
import ctypes
import os
import subprocess

import pytest

from tests import bound_cases as bc

HERE = os.path.dirname(os.path.abspath(__file__))
P, RINV = bc.P, bc.RINV


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
    for A in bc.redc_acc_cases():
        V = _int(_call(lz.hs_redc_acc, 9, _words(A, 17)))
        assert V == bc.redc_acc_expected(A), hex(A)
        assert V % P == A * RINV % P


def test_lin9_reduce_quotient_edges(lz):
    """T mod p for every k p - 1, k p, k p + 1 below 2^262 (k up to 338) and the container's extremes: the quotient estimate
    from the top 32 bits may be one short, never more."""
    for T in bc.lin9_cases():
        assert _int(_call(lz.hs_lin9_reduce, 8, _words(T, 9))) == T % P, hex(T)


# ------------------------------------------------------------------------------------------ the squaring
def test_gs_fp4_square_at_bounds(lz):
    """One Fp4 squaring with every input coefficient drawn from the extremes of the raw limb range (0, 1, p - 1, ...),
    both forms (plain and times xi): the accumulators and lin9_reduce inputs reach their stated maxima here."""
    for v in bc.gs_fp4_cases():
        a, b, x, y = (v[0], v[1]), (v[2], v[3]), (v[4], v[5]), (v[6], v[7])
        words = (ctypes.c_uint32 * 64)()
        for i, c in enumerate(v):
            words[8 * i: 8 * i + 8] = list(_words(c, 8))
        for xi in (0, 1):
            out = _call(lz.hs_gs_fp4_square, 32, words, xi)
            got = tuple(_int(out[8 * i: 8 * i + 8]) for i in range(4))
            assert got == bc.gs_expected(a, b, x, y, xi), (v, xi)


def test_cyclotomic_square_arbitrary_fp12(lz):
    """The in-place squaring on ANY Fp12 (not only cyclotomic values) equals the oracle's Granger-Scott formula: all-zero
    and all-(p - 1) raw coefficients, alternating extremes, and random values."""
    for raw in bc.cyclotomic_cases():
        words = (ctypes.c_uint32 * 96)()
        for i, c in enumerate(raw):
            words[8 * i: 8 * i + 8] = list(_words(c, 8))
        out = _call(lz.hs_cyclotomic_square, 96, words)
        got = [_int(out[8 * i: 8 * i + 8]) for i in range(12)]
        assert got == bc.cyclotomic_expected(raw), raw

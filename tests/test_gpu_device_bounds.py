"""GPU tier: the DEVICE versions of the lazy-reduction primitives (the PTX carry chains of fp.cuh), the lazily reduced
Granger-Scott squaring, the in-place Fp12 operations on a shared-memory slot and the two-lane operations of
pairing_lanes.cuh, each with values placed on the bounds the source comments state, against exact Python integers or
the oracle.  The harness is tests/hostsim/device_bounds.cu; test_lazy_fp4_square.py runs the same case lists
(tests/bound_cases.py) through the host versions.  Every input stays inside the contract of the function it feeds."""
import ctypes
import os
import random
import shutil
import subprocess

import numpy as np
import pytest

from oracle import bn254_py as o
from tests import bound_cases as bc
from tests import wire as w

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
P, R, RINV, PINV, TOP = bc.P, bc.R, bc.RINV, bc.PINV, bc.TOP
M512, M544 = (1 << 512) - 1, (1 << 544) - 1

# device_bounds.cu: enum Prim, enum Slot, enum Lanes
(MUL_WIDE, REDC_WIDE, REDC_LOW, MUL, FP2_MUL, WIDE_SUB, WIDE_ADD_PR, LIFT_SUB1, LIFT_SUB2, ACC_ADD, ACC_SUB, ACC_MADD9,
 REDC_ACC, LIN9_ACC, LIN9_REDUCE, U9_SHL0, U9_SHL1, U9_SHL3, LIN3, GS, GS_XI) = range(21)
S_SQR, S_SPARSE, S_CYCLOTOMIC, S_MUL, S_MUL_CONJ = range(5)
L_SQR, L_SPARSE, L_MUL, L_MUL_CONJ, L_CYCLOTOMIC, L_FROB1, L_FROB2, L_FROB3, L_INV = range(9)


@pytest.fixture(scope="module")
def db(tmp_path_factory):
    """The harness, built with the library's code-generation flags."""
    so = str(tmp_path_factory.mktemp("device_bounds") / "libdevice_bounds.so")
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-shared",
                           "-Xcompiler", "-fPIC", "-o", so, os.path.join(HERE, "hostsim", "device_bounds.cu")])
    lib = ctypes.CDLL(so)
    vp, i = ctypes.c_void_p, ctypes.c_int
    lib.db_prim.argtypes = [i, vp, vp, i, vp]
    lib.db_fp12_slot.argtypes = lib.db_lanes.argtypes = [i, vp, vp, vp, i, vp]
    lib.db_prim.restype = lib.db_fp12_slot.restype = lib.db_lanes.restype = i
    return lib


def _launch(fn, op, ins, out_width):
    """fn(op, *inputs, out, n, stream) on torch's current stream; ins are (n, width) uint8 arrays."""
    import torch

    dev = torch.device("cuda", 0)
    d_in = [torch.from_numpy(a).to(dev) for a in ins]
    n = ins[0].shape[0]
    out = torch.zeros((n, out_width), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    err = fn(op, *[ctypes.c_void_p(t.data_ptr()) for t in d_in], ctypes.c_void_p(out.data_ptr()), n,
             ctypes.c_void_p(stream))
    assert err == 0, "launch failed: cudaError %d" % err
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _words(*fields):
    """Little-endian limbs of (value, number of 32-bit words) fields, concatenated."""
    return b"".join(v.to_bytes(4 * n, "little") for v, n in fields)


def prim(db, op, rows):
    """One k_prim launch over rows of (value, words) fields; returns each item's 32 output words as bytes."""
    a = np.frombuffer(b"".join(_words(*r).ljust(256, b"\0") for r in rows), np.uint8).reshape(len(rows), 256).copy()
    return [bytes(r) for r in _launch(db.db_prim, op, [a], 128)]


def get(row, off, n):
    return int.from_bytes(row[4 * off: 4 * (off + n)], "little")


def _alt(nbits, byte):
    return int.from_bytes(bytes([byte]) * (nbits // 8), "little")


def _limb_mix(nwords, pattern):
    """Limb i is all ones where pattern(i) holds, else zero."""
    return sum(0xffffffff << (32 * i) for i in range(nwords) if pattern(i))


# ------------------------------------------------------------------------------------------ products and reductions
def test_fp_mul_wide(db):
    """fp.cuh fp_mul_wide: "T = a * b ... Requires a[7] != 0xffffffff (see wide_row_fold); b is any 256-bit value"; every
    first operand of the library is below 4p.  All 16 limbs must equal a * b, with a up to 4p - 1 and at the contract's
    edge (a[7] = 0xfffffffe, every lower limb all ones), b up to 2^256 - 1 and carry-ripple limb patterns."""
    rng = random.Random(101)
    edge_a = [0, 1, 2, P - 1, P, 2 * P - 1, 3 * P, 4 * P - 1, 0xfffffffe << 224, (0xfffffffe << 224) | ((1 << 224) - 1),
              (0xfffffffe << 224) | _alt(224, 0x55), (1 << 224) - 1, _limb_mix(7, lambda i: i % 2 == 0)]
    edge_b = [0, 1, 2, P - 1, 4 * P - 1, R - 1, R - 2, 1 << 255, (1 << 255) - 1, _alt(256, 0x55), _alt(256, 0xaa),
              _limb_mix(8, lambda i: i % 2 == 0), _limb_mix(8, lambda i: i % 2 == 1), (R - 1) ^ (0xffffffff << 96),
              (R - 1) ^ 0xffffffff, (R - 1) ^ (0xffffffff << 224)]
    pairs = [(a, b) for a in edge_a for b in edge_b]
    pairs += [(rng.randrange(4 * P), rng.choice(edge_b)) for _ in range(500)]
    pairs += [((0xfffffffe << 224) | rng.randrange(1 << 224), rng.randrange(R)) for _ in range(500)]
    pairs += [(rng.randrange(4 * P), rng.randrange(R)) for _ in range(1000)]
    for a, _ in pairs:
        assert a >> 224 != 0xffffffff
    out = prim(db, MUL_WIDE, [((a, 8), (b, 8)) for a, b in pairs])
    for (a, b), r in zip(pairs, out):
        assert get(r, 0, 16) == a * b, (hex(a), hex(b))


def test_fp_redc_wide_and_low(db):
    """fp.cuh fp_redc_wide: "r = T * R^-1 mod p, fully reduced, for T < p * R: W + T_hi with W <= p, T_hi < p", and
    redc_low: "W = (T_lo + M p) / R <= p for the low half T_lo".  T at 0, 1, p R - 1, p^2 +- 1, 4 p^2 (the fp2_sqr
    maximum) and random values; T_lo over the whole 256-bit range."""
    rng = random.Random(102)
    ts = [0, 1, 2, R - 1, R, P * R - 1, P * R - R, (P - 1) * R, P * P - 1, P * P, P * P + 1, 2 * P * P, 4 * P * P - 1,
          4 * P * P, (1 << 509) - 1, _alt(509, 0xff)]
    ts += [rng.randrange(P * R) for _ in range(2000)]
    for T in ts:
        assert T < P * R
    out = prim(db, REDC_WIDE, [((T, 16),) for T in ts])
    for T, r in zip(ts, out):
        assert get(r, 0, 8) == T * RINV % P, hex(T)
    lows = [0, 1, 2, P - 1, P, P + 1, R - P, R - 1, _alt(256, 0x55), _alt(256, 0xaa)] + [rng.randrange(R) for _ in range(1000)]
    out = prim(db, REDC_LOW, [((t, 8),) for t in lows])
    for t, r in zip(lows, out):
        W = get(r, 0, 8)
        assert W == (t + ((-t * PINV) % R) * P) // R, hex(t)
        assert W <= P


def test_fp_mul_at_contract(db):
    """fp.cuh fp_mul: "Requires a < 2p ... and a * b < p * R; b may be ANY 256-bit value as long as the product bound
    holds - so conversions of unreduced inputs put the constant first: fp_mul(R^2, x) is valid for every x < 2^256"."""
    rng = random.Random(103)
    r2 = R * R % P
    pairs = []
    for a in [P, P + 1, 2 * P - 1, (3 * P) // 2] + [rng.randrange(P, 2 * P) for _ in range(300)]:
        b = (P * R - 1) // a  # a * b just below p R
        pairs += [(a, b), (a, b - 1), (a, rng.randrange(b))]
    pairs += [(1, R - 1), (1, R - 2), (2, R - 1), (P - 1, P - 1), (0, R - 1)]
    xs = [0, 1, P - 1, P, P + 1, 2 * P, 4 * P, R - 1, R - 2, _alt(256, 0x55), _alt(256, 0xaa)]
    pairs += [(r2, x) for x in xs + [rng.randrange(R) for _ in range(500)]]
    pairs += [(rng.randrange(P), rng.randrange(P)) for _ in range(500)]
    for a, b in pairs:
        assert a < 2 * P and a * b < P * R and b < R
    out = prim(db, MUL, [((a, 8), (b, 8)) for a, b in pairs])
    for (a, b), r in zip(pairs, out):
        assert get(r, 0, 8) == a * b * RINV % P, (hex(a), hex(b))


def test_fp2_mul_signed_real_part(db):
    """tower.cuh fp2_mul: "c0 = a0 b0 - a1 b1 in (-p^2, p^2): add p*R when negative, then < p*R" - wide_sub, its borrow
    mask and wide_add_pR on raw Montgomery limbs, with a0 b0 - a1 b1 at -1, 0, +1, -(p - 1)^2 and (p - 1)^2."""
    rng = random.Random(104)
    cases = []  # (a0, a1, b0, b1, a0 b0 - a1 b1)
    for x in [1, 2, P - 2] + [rng.randrange(1, P - 1) for _ in range(100)]:
        cases.append((x + 1, x, x - 1, x, -1))
        cases.append((x, x + 1, x, x - 1, 1))
    for x, y in [(P - 1, P - 1), (0, 0), (1, P - 1)] + [(rng.randrange(P), rng.randrange(P)) for _ in range(100)]:
        cases.append((x, x, y, y, 0))
    for z in [0, 1, P - 1] + [rng.randrange(P) for _ in range(20)]:
        cases.append((0, P - 1, z, P - 1, -(P - 1) ** 2))
        cases.append((z, P - 1, 0, P - 1, -(P - 1) ** 2))
        cases.append((P - 1, 0, P - 1, z, (P - 1) ** 2))
        cases.append((P - 1, z, P - 1, 0, (P - 1) ** 2))
    cases += [(rng.randrange(P), rng.randrange(P), rng.randrange(P), rng.randrange(P), None) for _ in range(500)]
    for a0, a1, b0, b1, want in cases:
        assert want is None or a0 * b0 - a1 * b1 == want
    out = prim(db, FP2_MUL, [((a0, 8), (a1, 8), (b0, 8), (b1, 8)) for a0, a1, b0, b1, _ in cases])
    for (a0, a1, b0, b1, _), r in zip(cases, out):
        assert get(r, 0, 8) == (a0 * b0 - a1 * b1) * RINV % P, (a0, a1, b0, b1)
        assert get(r, 8, 8) == (a0 * b1 + a1 * b0) * RINV % P, (a0, a1, b0, b1)


def test_wide_sub_and_add_pR(db):
    """fp.cuh wide_sub: "16-limb a -= b; returns 0xffffffff if the subtraction borrowed (a < b), else 0", and wide_add_pR:
    "a[8..15] += p & mask (adds p * R to the 512-bit value when mask = 0xffffffff)", exact mod 2^512."""
    rng = random.Random(105)
    edge = [0, 1, 2, M512, M512 - 1, R - 1, R, P * R - 1, P * R, _alt(512, 0x55), _alt(512, 0xaa), 1 << 511,
            _limb_mix(16, lambda i: i % 2 == 0), _limb_mix(16, lambda i: i >= 8)] + [rng.randrange(1 << 512) for _ in range(10)]
    pairs = [(a, b) for a in edge for b in edge] + [(rng.randrange(1 << 512), rng.randrange(1 << 512)) for _ in range(300)]
    out = prim(db, WIDE_SUB, [((a, 16), (b, 16)) for a, b in pairs])
    for (a, b), r in zip(pairs, out):
        assert get(r, 0, 16) == (a - b) & M512, (hex(a), hex(b))
        assert get(r, 16, 1) == (0xffffffff if a < b else 0)
    rows = [(a, m) for a in edge for m in (0, 0xffffffff)]
    out = prim(db, WIDE_ADD_PR, [((a, 16), (m, 1)) for a, m in rows])
    for (a, m), r in zip(rows, out):
        assert get(r, 0, 16) == (a + (P * R if m else 0)) & M512, (hex(a), m)


# ------------------------------------------------------------------------------------------ the 17-limb accumulators
def test_accumulator_helpers(db):
    """fp.cuh acc_*: "The limbs are exact mod 2^544, so only the FINAL value has to lie in [0, 2^544)"; acc_lift_sub:
    "A = L p R - T for T < L p R ... A[16] = 0" (L = 1, 2); acc_add, acc_sub and acc_madd<9> at all-ones and zero limbs."""
    rng = random.Random(106)
    for op, L in ((LIFT_SUB1, 1), (LIFT_SUB2, 2)):
        lim = L * P * R
        ts = [0, 1, R - 1, R, lim - 1, lim - R, lim - R + 1, P * R - 1, (1 << 256) - 1 + (1 << 300),
              _alt(500, 0xff)] + [rng.randrange(lim) for _ in range(300)]
        ts = [t for t in ts if t < lim]
        out = prim(db, op, [((t, 16),) for t in ts])
        for t, r in zip(ts, out):
            assert get(r, 0, 17) == lim - t, (L, hex(t))
    acc_edge = [0, 1, M544, M544 - 1, M512, 1 << 512, 1 << 543, _alt(544, 0x55), _alt(544, 0xaa), M544 ^ M512,
                _limb_mix(17, lambda i: i % 2 == 0), _limb_mix(17, lambda i: i % 2 == 1)]
    acc_edge += [rng.randrange(1 << 544) for _ in range(8)]
    t_edge = [0, 1, 2, M512, M512 - 1, 1 << 511, R - 1, P * R - 1, _alt(512, 0x55), _alt(512, 0xaa),
              _limb_mix(16, lambda i: i % 2 == 0)] + [rng.randrange(1 << 512) for _ in range(8)]
    pairs = [(A, T) for A in acc_edge for T in t_edge]
    pairs += [(rng.randrange(1 << 544), rng.randrange(1 << 512)) for _ in range(300)]
    rows = [((A, 17), (T, 16)) for A, T in pairs]
    for op, f in ((ACC_ADD, lambda A, T: A + T), (ACC_SUB, lambda A, T: A - T), (ACC_MADD9, lambda A, T: A + 9 * T)):
        out = prim(db, op, rows)
        for (A, T), r in zip(pairs, out):
            assert get(r, 0, 17) == f(A, T) & M544, (op, hex(A), hex(T))


def test_fp_redc_acc_exact(db):
    """fp.cuh fp_redc_acc: "V = A * R^-1 mod p, not reduced: V = W + A_hi with W <= p (redc_low) and A_hi = floor(A / R)";
    V is (A + M p) / R exactly, for the accumulators of the squaring (up to 45.3 p^2 < 2^513) and the edges below
    2^261 R.  The cases of test_lazy_fp4_square.py::test_redc_acc_exact."""
    cases = bc.redc_acc_cases()
    out = prim(db, REDC_ACC, [((A, 17),) for A in cases])
    for A, r in zip(cases, out):
        V = get(r, 0, 9)
        assert V == bc.redc_acc_expected(A), hex(A)
        assert V % P == A * RINV % P


def test_lin9_acc(db):
    """fp.cuh lin9_acc: "T[0..8] += a[0..7]" for sums below 2^288, with the carry rippling through every limb."""
    rng = random.Random(107)
    top = (1 << 288) - 1
    rows = []
    for a in [0, 1, R - 1, P - 1, P, _alt(256, 0x55)] + [rng.randrange(R) for _ in range(50)]:
        rows += [(top - a, a), (0, a), (R - 1, min(a, 1)), (rng.randrange(top - a + 1), a)]
    rows += [((R - 1) | (rng.randrange(1 << 31) << 256), 1) for _ in range(20)]
    out = prim(db, LIN9_ACC, [((t, 9), (a, 8)) for t, a in rows])
    for (t, a), r in zip(rows, out):
        assert t + a <= top
        assert get(r, 0, 9) == t + a, (hex(t), hex(a))


def test_lin9_reduce_quotient_edges(db):
    """fp.cuh lin9_reduce: "lin9_reduce takes any 9-limb T < 2^262 (338 p ...).  The quotient is estimated from the top 32
    bits ... T - q p in [0, 2p)"; the result must be the canonical residue.  Every k p - 2 .. k p + 2 below 2^262
    (k up to 338) and the container's extremes: the cases of test_lazy_fp4_square.py::test_lin9_reduce_quotient_edges."""
    cases = bc.lin9_cases()
    out = prim(db, LIN9_REDUCE, [((T, 9),) for T in cases])
    for T, r in zip(cases, out):
        assert get(r, 0, 8) == T % P, hex(T)


def test_u9_add_shl(db):
    """fp.cuh u9_add_shl: "r = a + (b << s) (9 limbs, s < 32 a compile-time constant; the caller guarantees no overflow)"
    for the shifts the squaring uses (0, 1, 3), with sums up to 2^288 - 1."""
    rng = random.Random(108)
    top = (1 << 288) - 1
    for op, s in ((U9_SHL0, 0), (U9_SHL1, 1), (U9_SHL3, 3)):
        bmax = (top >> s)
        bs = [0, 1, bmax, bmax - 1, R - 1, _alt(288, 0x55) & bmax, _alt(288, 0xaa) & bmax, 1 << (287 - s)]
        bs += [rng.randrange(bmax + 1) for _ in range(100)]
        rows = []
        for b in bs:
            rows += [(top - (b << s), b), (0, b), (rng.randrange(top - (b << s) + 1), b)]
        out = prim(db, op, [((a, 9), (b, 9)) for a, b in rows])
        for (a, b), r in zip(rows, out):
            assert get(r, 0, 9) == a + (b << s), (s, hex(a), hex(b))


def test_fp_lin3(db):
    """fp.cuh fp_lin3: "3 V + y mod p for a 9-limb V and y < 2^256 (3 V + y < 2^262)", with 3 V + y on every lin9_reduce
    case (k p - 2 .. k p + 2 for k up to 338 and the extremes), once with y small and once with y as large as allowed."""
    rows = []
    for T in bc.lin9_cases():
        lo = T % 3
        hi = min(T, R - 1)
        hi -= (hi - lo) % 3
        for y in {lo, hi}:
            rows.append(((T - y) // 3, y))
    out = prim(db, LIN3, [((V, 9), (y, 8)) for V, y in rows])
    for (V, y), r in zip(rows, out):
        assert 3 * V + y < (1 << 262) and y < R
        assert get(r, 0, 8) == (3 * V + y) % P, (hex(V), hex(y))


# ------------------------------------------------------------------------------------------ the Granger-Scott squaring
def test_gs_fp4_square_at_bounds(db):
    """pairing.cuh gs_fp4_square: "A0 = S_a + 9 S_b - Q_b + p R < 45.3 p^2 ... all below 2^513" and "the reduced inputs
    of lin9_reduce are at most ... < 177 p ...: all below its 338 p", both forms (plain and times xi), with every input
    coefficient from the extremes of the raw limb range: the cases of test_lazy_fp4_square.py."""
    sets = bc.gs_fp4_cases()
    rows = [tuple((c, 8) for c in v) for v in sets]
    for op, xi in ((GS, 0), (GS_XI, 1)):
        out = prim(db, op, rows)
        for v, r in zip(sets, out):
            got = tuple(get(r, 8 * i, 8) for i in range(4))
            assert got == bc.gs_expected((v[0], v[1]), (v[2], v[3]), (v[4], v[5]), (v[6], v[7]), xi), (v, xi)


# ------------------------------------------------------------------------------------------ Fp12 operations
def _raw_fp12(f):
    """An Fp12 value as 384 bytes of raw Montgomery coefficients (the layout of fp12_load_raw)."""
    return b"".join((c * R % P).to_bytes(32, "little") for c in o.fp12_to_list(f))


def _fp12_run(fn, op, a, b):
    A = np.frombuffer(b"".join(a), np.uint8).reshape(len(a), 384).copy()
    B = np.frombuffer(b"".join(b), np.uint8).reshape(len(b), 384).copy()
    return [bytes(r) for r in _launch(fn, op, [A, B], 384)]


def test_cyclotomic_square_raw_coefficients(db):
    """pairing.cuh cyclotomic_square_assign on a shared-memory slot, on ANY twelve raw coefficients: the cases of
    test_lazy_fp4_square.py::test_cyclotomic_square_arbitrary_fp12."""
    cases = bc.cyclotomic_cases()
    a = [b"".join(c.to_bytes(32, "little") for c in raw) for raw in cases]
    out = _fp12_run(db.db_fp12_slot, S_CYCLOTOMIC, a, a)
    for raw, r in zip(cases, out):
        assert [get(r, 8 * i, 8) for i in range(12)] == bc.cyclotomic_expected(raw), raw


@pytest.fixture(scope="module")
def fp12_items():
    """The edge-coefficient pairs of test_gpu_parity.py::test_fp12_edge_coefficients and 300 random pairs."""
    a, b = bc.fp12_edge_pairs()
    rng = random.Random(109)
    a = a + [w.rand_fp12(rng) for _ in range(300)]
    b = b + [w.rand_fp12(rng) for _ in range(300)]
    return a, b, [_raw_fp12(x) for x in a], [_raw_fp12(y) for y in b]


_EXPECT = {
    "sqr": lambda x, y: o.fp12_sqr(x),
    "sparse": lambda x, y: o.fp12_sparse_mul(x, y[0][0], y[0][1], y[0][2]),
    "cyclotomic": lambda x, y: o.cyclotomic_squared(x),
    "mul": lambda x, y: o.fp12_mul(x, y),
    "mul_conj": lambda x, y: o.fp12_mul(x, o.fp12_conj(y)),
    "frob1": lambda x, y: o.fp12_frobenius(x, 1),
    "frob2": lambda x, y: o.fp12_frobenius(x, 2),
    "frob3": lambda x, y: o.fp12_frobenius(x, 3),
    "inv": lambda x, y: o.fp12_inv(x),
}


def _check_fp12(out, items, name):
    a, b = items[0], items[1]
    for k, (x, y, r) in enumerate(zip(a, b, out)):
        assert r == _raw_fp12(_EXPECT[name](x, y)), (name, k)


@pytest.mark.parametrize("name,op", [("sqr", S_SQR), ("sparse", S_SPARSE), ("cyclotomic", S_CYCLOTOMIC), ("mul", S_MUL),
                                     ("mul_conj", S_MUL_CONJ)])
def test_fp12_in_place_on_shared_slot(db, fp12_items, name, op):
    """tower.cuh fp12_sqr_assign, fp12_sparse_mul_assign, fp12_mul_assign (conj_b false and true: "conj_b = true
    multiplies by the conjugate (b.c0, -b.c1) without materialising it") and pairing.cuh cyclotomic_square_assign,
    updating f in a shared-memory slot at SY_ACC_STRIDE as k_miller and k_final_exp do."""
    _check_fp12(_fp12_run(db.db_fp12_slot, op, fp12_items[2], fp12_items[3]), fp12_items, name)


@pytest.mark.parametrize("name,op", [("sqr", L_SQR), ("sparse", L_SPARSE), ("mul", L_MUL), ("mul_conj", L_MUL_CONJ),
                                     ("cyclotomic", L_CYCLOTOMIC), ("frob1", L_FROB1), ("frob2", L_FROB2),
                                     ("frob3", L_FROB3), ("inv", L_INV)])
def test_two_lane_operations(db, fp12_items, name, op):
    """pairing_lanes.cuh lanes_fp12_sqr, lanes_sparse_mul (PairSlot), lanes_fp12_mul (both flags),
    lanes_cyclotomic_square, lanes_frobenius_to (e = 1, 2, 3) and lanes_fp12_inv (FexpHot), two threads per item; the
    item count (500) leaves surplus lane pairs in the last block, which redo the last item."""
    _check_fp12(_fp12_run(db.db_lanes, op, fp12_items[2], fp12_items[3]), fp12_items, name)


# ------------------------------------------------------------------------------------------ final exponentiation
@pytest.mark.parametrize("lanes", ["0", "2"])
def test_final_exp_structured_inputs(monkeypatch, lanes):
    """final_exp_batch through k_final_exp (SYLOW_B200_LANES=0) and k_final_exp_lanes (=2): zero gives zero, one gives
    one, a nonzero element of Fp6 (c1 = 0) gives one (f^(p^6 - 1) = 1), every coefficient at the Montgomery top value
    and random values give the oracle's result.  The ten items are repeated seven times, past one two-lane block."""
    import sylow_b200

    rng = random.Random(110)
    zero = o.fp12_from_list([0] * 12)
    in_fp6 = [o.fp12_from_list([rng.randrange(P) for _ in range(6)] + [0] * 6), o.fp12_from_list([TOP] * 6 + [0] * 6),
              o.fp12_from_list([0, 0, 5] + [0] * 9)]
    top = o.fp12_from_list([TOP] * 12)
    rand = [w.rand_fp12(rng) for _ in range(4)]
    items = [zero, o.FP12_ONE] + in_fp6 + [top] + rand
    expect = [zero, o.FP12_ONE] + [o.FP12_ONE] * len(in_fp6) + [o.final_exponentiation(f) for f in [top] + rand]
    assert [o.final_exponentiation(f) for f in items[:2 + len(in_fp6)]] == expect[:2 + len(in_fp6)]
    F = np.frombuffer(b"".join(w.fp12_b(f) for f in items * 7), np.uint8).reshape(7 * len(items), 384).copy()
    monkeypatch.setenv("SYLOW_B200_LANES", lanes)
    eng = sylow_b200.Engine(0)
    try:
        out = eng.final_exp_batch(F)
    finally:
        eng.close()
    assert [w.b_fp12(bytes(r)) for r in out] == expect * 7

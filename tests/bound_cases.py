"""Case lists at the stated bounds of the lazy-reduction primitives (fp.cuh: fp_redc_acc, lin9_reduce; pairing.cuh:
gs_fp4_square, cyclotomic_square_assign) and of the tower operations, with their expected values.  One list, two
implementations: the host build of the device source (test_lazy_fp4_square.py) and the device build
(test_gpu_device_bounds.py) run the same cases.  Values are RAW Montgomery limbs unless a function says otherwise."""
import random

from oracle import bn254_py as o

P = o.P
R = 1 << 256
RINV = pow(R, -1, P)
PINV = pow(P, -1, R)
# the largest Montgomery limb pattern: -1/R mod p is stored as p - 1
TOP = P - RINV


def redc_acc_cases():
    """17-limb accumulators A for fp_redc_acc: up to the largest the squaring forms (A0 < S_a + 9 S_b + p R, 45.3 p^2
    < 2^513) and the 17-limb edges below 2^261 R."""
    rng = random.Random(17)
    top = 4 * P * P + 9 * 4 * P * P + P * R  # A0's bound: S_a + 9 S_b + p R
    cases = [0, 1, R - 1, R, P * R, P * R - 1, top - 1, top, (1 << 513) - 1, (1 << 512), (1 << 512) - 1,
             (1 << 261) * R - 1]
    cases += [k * P * R + d for k in (1, 2, 9, 27) for d in (-1, 0, 1)]
    cases += [rng.randrange(top) for _ in range(2000)] + [rng.randrange((1 << 261) * R) for _ in range(200)]
    return cases


def redc_acc_expected(A):
    """V = (A + M p) / R with M = -A p^-1 mod R: exact, not reduced."""
    M = (-A * PINV) % R
    return (A + M * P) // R


def lin9_cases():
    """9-limb T for lin9_reduce: every k p - 2 .. k p + 2 below 2^262 (k up to 338) and the container's extremes."""
    rng = random.Random(262)
    cases = [0, 1, P - 1, P, (1 << 256) - 1, 1 << 256, (1 << 262) - 1, (1 << 261), (1 << 262) - P]
    for k in range(1, 340):
        for d in (-2, -1, 0, 1, 2):
            T = k * P + d
            if 0 <= T < (1 << 262):
                cases.append(T)
    cases += [rng.randrange(1 << 262) for _ in range(5000)]
    return cases


def _fp2_raw(a):
    return [a[0] * RINV % P, a[1] * RINV % P]


def _to_raw(a):
    return tuple(c * R % P for c in a)


def gs_fp4_cases():
    """Eight raw coefficients (a, b, x, y) per case for one Fp4 squaring: every coefficient from the extremes of the
    raw limb range (0, 1, p - 1, ...); the accumulators and the lin9_reduce inputs reach their stated maxima here."""
    rng = random.Random(4)
    edge = [0, 1, 2, P - 1, P - 2, (P - 1) // 2, (P + 1) // 2, (1 << 253), (1 << 254) - 1 - (1 << 200)]
    edge = [e for e in edge if e < P]
    sets = [[P - 1] * 8, [0] * 8, [P - 1, 0] * 4, [0, P - 1] * 4, [P - 1] * 4 + [0] * 4, [0] * 4 + [P - 1] * 4]
    sets += [[rng.choice(edge) for _ in range(8)] for _ in range(400)]
    sets += [[rng.randrange(P) for _ in range(8)] for _ in range(200)]
    return sets


def gs_expected(a, b, x, y, xi):
    """x <- 3 A - 2 x, y <- 3 B + 2 y (3 xi B + 2 y) with (A, B) the Fp4 square of (a, b), all on raw Montgomery limbs."""
    a, b, x, y = (tuple(_fp2_raw(v)) for v in (a, b, x, y))
    t0, t1 = o._fp4_square(a, b)
    if xi:
        t1 = o.fp2_residue_mul(t1)
    nx = o.fp2_sub(o.fp2_scale(t0, 3), o.fp2_scale(x, 2))
    ny = o.fp2_add(o.fp2_scale(t1, 3), o.fp2_scale(y, 2))
    return _to_raw(nx) + _to_raw(ny)


def cyclotomic_cases():
    """Twelve raw coefficients per case: all-zero and all-(p - 1), alternating extremes, and random values."""
    rng = random.Random(12)
    cases = [[0] * 12, [P - 1] * 12, [P - 1, 0] * 6, [0, P - 1] * 6, [P - 1] * 6 + [0] * 6, [1] * 12]
    cases += [[rng.choice([0, 1, P - 1, P - 2]) for _ in range(12)] for _ in range(100)]
    cases += [[rng.randrange(P) for _ in range(12)] for _ in range(100)]
    return cases


def cyclotomic_expected(raw):
    """The Granger-Scott formula of the oracle on twelve raw coefficients, as raw coefficients."""
    f = o.fp12_from_list([c * RINV % P for c in raw])
    return [c * R % P for c in o.fp12_to_list(o.cyclotomic_squared(f))]


def fp12_edge_pairs():
    """200 pairs (a, b) of CANONICAL Fp12 values whose coefficients sit at the carry-propagation extremes of the
    lazy-reduction Fp2 arithmetic: {0, 1, 2, p - 1, p - 2, (p - 1)/2, (p + 1)/2, 2^32 - 1, 2^224, R mod p, ...}, the value
    stored as the limb pattern p - 1 (TOP) and 0/TOP mixtures."""
    rng = random.Random(29)
    edge = [0, 1, 2, P - 1, P - 2, (P - 1) // 2, (P + 1) // 2, (1 << 32) - 1, 1 << 224, (1 << 253) + 1,
            R % P, P - (R % P), 0xFFFFFFFF00000000FFFFFFFF00000000FFFFFFFF00000000 % P]
    # the lazy-reduction bounds are on the MONTGOMERY representatives
    edge += [TOP, (P - 2) * RINV % P]
    n = 200
    a = [o.fp12_from_list([rng.choice(edge) for _ in range(12)]) for _ in range(n)]
    b = [o.fp12_from_list([rng.choice(edge) for _ in range(12)]) for _ in range(n)]
    a[0] = o.fp12_from_list([P - 1] * 12)
    b[0] = o.fp12_from_list([P - 1] * 12)
    a[1], b[1] = o.fp12_from_list([TOP] * 12), o.fp12_from_list([TOP] * 12)
    a[2], b[2] = o.fp12_from_list([TOP, 0] * 6), o.fp12_from_list([0, TOP] * 6)
    a[3], b[3] = o.fp12_from_list([TOP] * 6 + [0] * 6), o.fp12_from_list([0] * 6 + [TOP] * 6)
    for i in range(4, 64):
        a[i] = o.fp12_from_list([rng.choice([0, TOP]) for _ in range(12)])
        b[i] = o.fp12_from_list([rng.choice([0, TOP]) for _ in range(12)])
    return a, b

"""Extreme inputs for the pairing, group-law and ladder kernels, built deterministically (no sampling of the edges):

- G1 points whose canonical x is at the top of the wire range (p - 1, p - 2, ...) and points whose x is STORED as an
  extreme Montgomery limb pattern v (x = v R^-1 mod p, so the device holds v); each with y and p - y.  Every curve point
  is in G1 (cofactor 1), so they are inside every entry point's contract.
- Scalars at the edges of every recoding: the GLV halves (glv_decompose + signed_windows4<32>), the four GLS components
  (gls_decompose + signed_windows4<17>, shared by g2_mul and gt_pow), the signed 8-bit digits of the fixed-base ladder
  (scalar_reduce_r + scalar_digit<8>), the bucket MSM's c-bit digits, and the common edges 0, 1, r - 1, r, ...
- Fp12 values: the coefficient patterns of the lazy-reduction tests (tests/bound_cases.py).

The GLV / GLS scalars are built from chosen components, k = sum_j k_j e^j mod r; Babai rounding returns the chosen
components only inside its cell, so every candidate is decomposed by the host build of the device source and kept only
if it reproduces its components (glv_scalars / gls_scalars take the loaded tests/hostsim library)."""
import ctypes

from oracle import bn254_py as o
from tests import bound_cases as bc

P, R = o.P, o.R_ORDER
RM = 1 << 256
RINV = pow(RM, -1, P)
LAMBDA = 0xB3C4D79D41A917585BFC41088D8DAAA78B17EA66B99C90DD  # phi(x, y) = (beta x, y) acts as lambda (curve.cuh)
MU = P % R  # psi acts on the r-torsion of the twist as mu (the GLS base)
EDGE_SCALARS = [0, 1, R - 1, R, R + 1, (1 << 254) - 1, 1 << 255, (1 << 256) - 1]
# stored limb patterns of Montgomery-extreme x coordinates (each stepped down until x^3 + 3 is a square)
MONT_TARGETS = [P - 1, P - 2, (P + 1) // 2, (1 << 253) + 1, (1 << 253) - 1, (1 << 252) + 1, 1 << 224, 3]


# ------------------------------------------------------------------------------------------ G1 points
def _y(x):
    return o.fp_sqrt((x * x * x + 3) % P)


def _pair(x, y):
    return [(x, y, False), (x, P - y, False)]


def g1_wire_extremes(count=4):
    """(x, y) and (x, p - y) for the `count` largest canonical x < p with x^3 + 3 a square: (p - 1)^3 + 3 = 2 is one
    (p = 7 mod 8)."""
    out, x = [], P - 1
    while len(out) < 2 * count:
        y = _y(x)
        if y is not None:
            out += _pair(x, y)
        x -= 1
    return out


def g1_mont_extremes():
    """[(v, point), ...]: for each target limb pattern, the largest v <= target with x = v R^-1 mod p on the curve;
    the device stores x as v.  Both y and p - y."""
    out = []
    for v in MONT_TARGETS:
        while _y(v * RINV % P) is None:
            v -= 1
        x = v * RINV % P
        out += [(v, pt) for pt in _pair(x, _y(x))]
    return out


def g1_extremes():
    """every extreme G1 point, affine (x, y, False)"""
    return g1_wire_extremes() + [pt for _, pt in g1_mont_extremes()]


# ------------------------------------------------------------------------------------------ recodings
def signed_windows4(mag, nw):
    """curve.cuh signed_windows4<NW>: digits in [-8, 8] of a magnitude, least significant first, and each window's
    carry out"""
    digits, carries, carry = [], [], 0
    for w in range(nw):
        d = ((mag >> (4 * w)) & 15) + carry
        carry = int(d > 8)
        digits.append(d - 16 * carry)
        carries.append(carry)
    return digits, carries


def fixed_base_digits(k, c=8):
    """curve.cuh scalar_reduce_r + scalar_digit<C>: (the signed digits of k mod r, each window's carry out,
    the subtractions of r scalar_reduce_r makes)"""
    subs = 0
    while k >= R:
        k -= R
        subs += 1
    nw = (254 + c - 1) // c
    digits, carries, carry = [], [], 0
    for w in range(nw):
        d = ((k >> (c * w)) & ((1 << c) - 1)) + carry
        carry = int(d > (1 << (c - 1)))
        digits.append(d - (carry << c))
        carries.append(carry)
    return digits, carries, subs


def _nibbles(top, fill, n):
    """the n-nibble magnitude with top nibble `top` and every other nibble `fill`"""
    return (top << (4 * (n - 1))) | int(("%x" % fill) * (n - 1), 16)


def _component_patterns(n, seed_bits):
    """magnitudes of n nibbles for one recoded component: every lower nibble 9 (every window carries), every lower
    nibble 8 (digit 8, no carry), all ones below the top nibble (carry chain into the top window), each with every
    top nibble, and the largest values below 2^(4n - 1)"""
    pats = []
    for top in range(8):
        pats += [_nibbles(top, 9, n), _nibbles(top, 8, n), _nibbles(top, 15, n)]
    pats += [(1 << (4 * n - 1)) - 1 - d for d in (0, 1, 7, 8, 9, 1 << 60)]
    pats += [1 << seed_bits, (1 << seed_bits) - 1, 0, 1]
    return pats


GLV_CLASSES = ("every_window_carries", "every_digit_8", "top_digit_from_carry", "top_nibble_max", "mixed_signs",
               "zero_half")


def _classes(mags, negs, nw, limit_top):
    """which recoding edges the decomposed components (magnitudes, signs) reach"""
    got = set()
    tops = []
    for m in mags:
        d, c = signed_windows4(m, nw)
        assert c[-1] == 0 and -8 <= d[-1] <= 8  # the ladders' contract: the top window never carries
        if all(c[:-1]):
            got.add("every_window_carries")
        if all(x == 8 for x in d[:-1]):
            got.add("every_digit_8")
        if c[-2] and m >> (4 * (nw - 1)):
            got.add("top_digit_from_carry")
        tops.append(m >> (4 * (nw - 1)))
        if m == 0:
            got.add("zero_half")
    if max(tops) >= limit_top:
        got.add("top_nibble_max")
    if len({n for m, n in zip(mags, negs) if m}) == 2:
        got.add("mixed_signs")
    return got


def _glv_decompose(hs, k):
    out = ctypes.create_string_buffer(32)
    f = hs.hs_glv_decompose(k.to_bytes(32, "little"), out)
    b = out.raw
    return [int.from_bytes(b[:16], "little"), int.from_bytes(b[16:], "little")], [bool(f & 1), bool(f & 2)]


def _gls_decompose(hs, k):
    out = ctypes.create_string_buffer(48)
    f = hs.hs_gls_decompose(k.to_bytes(32, "little"), out)
    b = out.raw
    return [int.from_bytes(b[12 * j:12 * j + 12], "little") for j in range(4)], [bool(f >> j & 1) for j in range(4)]


# the top nibble a component reaches at most in practice: Babai rounding keeps |k1|, |k2| of the GLV split below
# |a1| + |a2| < 2^127 and the GLS components (a basis of index 3, DESIGN) near 2^65, so "top_nibble_max" is a
# component with that top nibble
GLV_TOP, GLS_TOP = 6, 1
# the GLS classes reached: a component's top window (bits 64..67) is at most 1 with no carry into it from below
GLS_REACHED = tuple(c for c in GLV_CLASSES if c != "top_digit_from_carry")


def _search(decompose, candidates, nw, top):
    """{class: [k, ...]} over the candidate scalars, classified by their actual decomposition"""
    out = {c: [] for c in GLV_CLASSES}
    for k in dict.fromkeys(candidates):
        mags, negs = decompose(k)
        for c in _classes(mags, negs, nw, top):
            out[c].append(k)
    return out


def glv_scalars(hs):
    """{class: [k, ...]}: k = s1 k1 + s2 k2 lambda mod r from chosen halves (Babai rounding returns most of them), and
    a seeded sweep of scalars near the cell's edge, classified by what glv_decompose returns"""
    import random

    pats = _component_patterns(32, 120)
    cand = [(s1 * a + s2 * b * LAMBDA) % R for i, a in enumerate(pats) for b in pats[i % 5::5] + [0]
            for s1, s2 in ((1, 1), (1, -1), (-1, 1), (-1, -1))]
    rng = random.Random(127)
    cand += [rng.randrange(R) for _ in range(400)]
    return _search(lambda k: _glv_decompose(hs, k), cand, 32, GLV_TOP)


def gls_scalars(hs):
    """{class: [k, ...]}: k = sum_j s_j k_j mu^j mod r from chosen components and a seeded sweep, classified by what
    gls_decompose returns (the split reproduces a chosen k0 below about 2^64 with the others zero)"""
    import random

    pats = _component_patterns(17, 60)
    signs = [(1, 1, 1, 1), (1, -1, 1, -1), (-1, 1, -1, 1), (-1, -1, -1, -1)]
    cand = []
    for i, a in enumerate(pats):
        for cs in ([a, 0, 0, 0], [a, pats[(i + 7) % len(pats)], 0, pats[(i + 3) % len(pats)]]):
            for sg in signs:
                cand.append(sum(s * c * pow(MU, j, R) for j, (s, c) in enumerate(zip(sg, cs))) % R)
    rng = random.Random(67)
    cand += [rng.randrange(R) for _ in range(2000)]
    return _search(lambda k: _gls_decompose(hs, k), cand, 17, GLS_TOP)


FIXED_CLASSES = ("digit_128_every_window", "digit_minus127_every_window", "top_window_limit", "reduce_1", "reduce_2",
                 "reduce_3", "reduce_4", "reduce_5")


def fixed_base_scalars():
    """{class: [k, ...]} for the fixed-base ladder's 8-bit signed digits"""
    b80 = int("80" * 31, 16)
    b81 = b80 + 1  # bytes 0x81, 0x80, 0x80, ...: with the carry every window sees 0x81
    out = {
        # byte 0x80 in every window below the top: digit 128, no carry
        "digit_128_every_window": [b80, (0x2F << 248) | b80],
        # byte 0x81: digit -127 and a carry into every next window, the top one included
        "digit_minus127_every_window": [b81, (0x2F << 248) | b81, (0x10 << 248) | b81],
        # the top window (bits 248..253, below r's top byte 0x30) at its largest, with and without a carry into it
        "top_window_limit": [R - 1, (0x2F << 248) | b81, (0x30 << 248) | int("63" + "ff" * 30, 16)],
    }
    base = [1, 0x80, b80 >> 8, b81 >> 16, (1 << 250) + 0x81]
    for j in range(1, 6):
        out["reduce_%d" % j] = [k + j * R for k in base if k + j * R < RM]
    out["reduce_5"].append(RM - 1)
    return out


def fixed_base_class_check(cls, k):
    """True if k reaches the fixed-base edge `cls`"""
    d, c, subs = fixed_base_digits(k)
    if cls == "digit_128_every_window":
        return all(x == 128 for x in d[:-1])
    if cls == "digit_minus127_every_window":
        return all(x == -127 for x in d[1:-1]) and all(c[:-1])
    if cls == "top_window_limit":
        return d[-1] >= 0x30
    return subs == int(cls[-1])


# ------------------------------------------------------------------------------------------ bucket MSM
MSM_WINDOWS = (4, 5, 7, 8, 9, 11, 13, 16)


def msm_digits(k, c):
    """the unsigned c-bit digits of the 256-bit k (sylow_b200.cu msm_digit), least significant first"""
    return [(k >> (c * w)) & ((1 << c) - 1) for w in range((256 + c - 1) // c)]


# ------------------------------------------------------------------------------------------ Fp12
def fp12_extremes():
    """canonical Fp12 values at the lazy-reduction extremes: the pattern pairs of tests/bound_cases.py, flattened"""
    a, b = bc.fp12_edge_pairs()
    return a + b

"""The lazily reduced Fp12 product on the device (tower.cuh: fp12_mul_assign over fp4_mul_redc) against the oracle on
arbitrary Fp12 values: zero, the largest Montgomery limb pattern p - 1 in every position, mixtures of the two, other edge
coefficients and random values; through fp12_op 0 and, for both values of conj_b, on a shared-memory slot."""
import random

import numpy as np
import pytest

from oracle import bn254_py as o
from tests import wire as w
from tests.test_gpu_device_bounds import S_MUL, S_MUL_CONJ, _fp12_run, _raw_fp12, db  # noqa: F401 (db: fixture)

pytestmark = pytest.mark.gpu


def test_fp12_mul_edges_and_random():
    import sylow_b200

    rng = random.Random(1213)
    P = o.P
    top = P - pow(1 << 256, -1, P)  # stored as the limb pattern p - 1
    edge = [0, 1, P - 1, P - 2, top, (P - 2) * pow(1 << 256, -1, P) % P, (P + 1) // 2, 1 << 253]
    pats = [[0] * 12, [top] * 12, [top, 0] * 6, [0, top] * 6, [top] * 6 + [0] * 6, [0] * 6 + [top] * 6]
    pairs = [(x, y) for x in pats for y in pats]
    pairs += [([rng.choice([0, top]) for _ in range(12)], [rng.choice([0, top]) for _ in range(12)]) for _ in range(100)]
    pairs += [([rng.choice(edge) for _ in range(12)], [rng.choice(edge) for _ in range(12)]) for _ in range(100)]
    pairs += [([rng.randrange(P) for _ in range(12)], [rng.randrange(P) for _ in range(12)]) for _ in range(300)]
    a = [o.fp12_from_list(x) for x, _ in pairs]
    b = [o.fp12_from_list(y) for _, y in pairs]
    A = np.frombuffer(b"".join(w.fp12_b(x) for x in a), dtype=np.uint8).reshape(len(a), -1).copy()
    B = np.frombuffer(b"".join(w.fp12_b(y) for y in b), dtype=np.uint8).reshape(len(b), -1).copy()
    eng = sylow_b200.Engine(0)
    try:
        out = eng.fp12_op_batch(0, A, B)
    finally:
        eng.close()
    assert [w.b_fp12(bytes(r)) for r in out] == [o.fp12_mul(x, y) for x, y in zip(a, b)]


def test_fp12_mul_assign_conj_on_device(db):
    """fp12_mul_assign with conj_b = false and true on the device (tests/hostsim/device_bounds.cu, the running value in
    a shared-memory slot as in k_final_exp), on raw limb patterns with every coefficient 0 or p - 1 and on random
    values, against the oracle's a b and a conj(b)."""
    rng = random.Random(1214)
    P, R = o.P, 1 << 256
    rinv = pow(R, -1, P)
    pats = [[0] * 12, [P - 1] * 12, [P - 1, 0] * 6, [0, P - 1] * 6]
    raws = [(x, y) for x in pats for y in pats]
    raws += [([rng.choice([0, P - 1]) for _ in range(12)], [rng.choice([0, P - 1]) for _ in range(12)])
             for _ in range(100)]
    raws += [([rng.randrange(P) for _ in range(12)], [rng.randrange(P) for _ in range(12)]) for _ in range(200)]
    a = [o.fp12_from_list([c * rinv % P for c in x]) for x, _ in raws]
    b = [o.fp12_from_list([c * rinv % P for c in y]) for _, y in raws]
    ra, rb = [_raw_fp12(x) for x in a], [_raw_fp12(y) for y in b]
    for op, conj in ((S_MUL, False), (S_MUL_CONJ, True)):
        out = _fp12_run(db.db_fp12_slot, op, ra, rb)
        want = [_raw_fp12(o.fp12_mul(x, o.fp12_conj(y) if conj else y)) for x, y in zip(a, b)]
        assert [bytes(r) for r in out] == want, conj

"""The lazily reduced Granger-Scott squaring on the device (fp12_op 6, pairing.cuh: cyclotomic_square_assign) against the
oracle's formula on arbitrary Fp12 values: zero, the largest Montgomery limb pattern p - 1 in every position, mixtures of
the two, other edge coefficients and random values."""
import random

import numpy as np
import pytest

from oracle import bn254_py as o
from tests import wire as w

pytestmark = pytest.mark.gpu


def test_cyclotomic_square_edges_and_random():
    import sylow_b200

    rng = random.Random(66)
    P = o.P
    top = P - pow(1 << 256, -1, P)  # stored as the limb pattern p - 1
    edge = [0, 1, P - 1, P - 2, top, (P - 2) * pow(1 << 256, -1, P) % P, (P + 1) // 2, 1 << 253]
    cases = [[0] * 12, [top] * 12, [P - 1] * 12, [top, 0] * 6, [0, top] * 6, [top] * 6 + [0] * 6, [0] * 6 + [top] * 6]
    cases += [[rng.choice([0, top]) for _ in range(12)] for _ in range(100)]
    cases += [[rng.choice(edge) for _ in range(12)] for _ in range(100)]
    cases += [[rng.randrange(P) for _ in range(12)] for _ in range(300)]
    a = [o.fp12_from_list(c) for c in cases]
    A = np.frombuffer(b"".join(w.fp12_b(x) for x in a), dtype=np.uint8).reshape(len(a), -1).copy()
    eng = sylow_b200.Engine(0)
    try:
        out = eng.fp12_op_batch(6, A, A)
    finally:
        eng.close()
    assert [w.b_fp12(bytes(r)) for r in out] == [o.cyclotomic_squared(x) for x in a]

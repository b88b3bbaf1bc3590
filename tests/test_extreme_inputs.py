"""CPU tier: the extreme inputs of tests/extreme_inputs.py are what they claim to be: every G1 point is on the curve
with the intended canonical or stored (Montgomery) x, and every scalar class is reached by the host build's GLV / GLS
decompositions and by the fixed-base and bucket digit recodings."""
from oracle import bn254_py as o
from tests import extreme_inputs as X
from tests.test_hostsim import hs  # noqa: F401 (fixture)

P = o.P


def test_g1_points():
    wire = X.g1_wire_extremes()
    assert wire[0][0] == P - 1 and wire[0][1] ** 2 % P == 2  # (p - 1)^3 + 3 = 2
    assert sorted({p[0] for p in wire}, reverse=True)[0] == P - 1
    mont = X.g1_mont_extremes()
    for v, (x, y, inf) in mont:
        assert x * X.RM % P == v and 0 <= x < P and 0 < y < P and not inf
    assert {v for v, _ in mont} >= {P - 1, P - 2, (P + 1) // 2}  # usable as they are
    for x, y, _ in X.g1_extremes():
        assert o.g1_is_on_curve(x, y) and o.g1_affine_neg((x, y, False)) in X.g1_extremes()


def test_scalar_classes(hs):  # noqa: F811
    glv = X.glv_scalars(hs)
    assert all(glv[c] for c in X.GLV_CLASSES), {c: len(v) for c, v in glv.items()}
    gls = X.gls_scalars(hs)
    assert all(gls[c] for c in X.GLS_REACHED), {c: len(v) for c, v in gls.items()}
    for c, ks in X.fixed_base_scalars().items():
        assert ks and all(X.fixed_base_class_check(c, k) for k in ks), c
        assert all(0 <= k < X.RM for k in ks)
    top = (1 << 256) - 1
    for c in X.MSM_WINDOWS:
        d = X.msm_digits(top, c)
        assert d[:-1] == [(1 << c) - 1] * (len(d) - 1) and d[-1] == (1 << (256 - c * (len(d) - 1))) - 1


def test_fp12_values():
    vals = X.fp12_extremes()
    assert o.fp12_from_list([X.P - X.RINV] * 12) in vals  # every coefficient stored as p - 1
    assert o.fp12_from_list([0] * 12) in vals or o.fp12_from_list([P - X.RINV, 0] * 6) in vals

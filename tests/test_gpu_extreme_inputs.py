"""GPU tier (-m gpu): the Miller, check-product, group-law and ladder kernels on the extreme inputs of
tests/extreme_inputs.py (G1 points with top-of-range wire and Montgomery x coordinates, scalars at the edges of the GLV,
GLS, fixed-base and bucket recodings, extreme Fp12 values), every value compared bit for bit with the C oracle (whole
arrays) or bn254_py (samples), every verdict with a known construction.  Each case names the kernel form it targets and
fails if the launch plan (host build of launch_plan.h, SYLOW_B200_LANES) or the context's launch count says it was not
reached.  Batches are the extreme items tiled, so the first and last item of every launch segment and block is one."""
import random

import numpy as np
import pytest

from oracle import bn254_py as o
from oracle import c_oracle as c
from tests import extreme_inputs as X
from tests import wire as w
from tests.test_hostsim import hs  # noqa: F401 (fixture)
from tests.test_launch_plan import ALWAYS, AUTO, MILLER, NEVER, _launches
from tests.test_gpu_verdict_seams import _plan, seams  # noqa: F401 (fixture)

pytestmark = pytest.mark.gpu
R = o.R_ORDER
EXT = X.g1_extremes()
TABLE_COST = 6045  # miller_product_tables' cost of one pair against a table for glue_pairs
ERR_DECODE = -6
MSM_ITEM = 256  # SY_MSM_ITEM: points per work item of a bucket sum
MSM_BUCKET_LAUNCHES = 10


@pytest.fixture(scope="module")
def eng():
    import sylow_b200

    e = sylow_b200.Engine(0)
    yield e
    e.close()


def arr(bs):
    return np.frombuffer(b"".join(bs), dtype=np.uint8).reshape(len(bs), -1).copy()


def _scal(ks):
    return arr([w.fp_b(k % (1 << 256)) for k in ks])


def _tile(a, n):
    return np.resize(a, (n,) + a.shape[1:]).copy()


G1X = arr([w.g1_b(p) for p in EXT])
NEG = {i: EXT.index(o.g1_affine_neg(p)) for i, p in enumerate(EXT)}  # every extreme point's negation is one too


@pytest.fixture(scope="module")
def g2pool():
    """random G2 subgroup points (the C oracle's multiples of the generator) and the generator"""
    rs = np.random.RandomState(77)
    k = rs.randint(0, 256, size=(16, 32), dtype=np.uint8)
    k[:, 31] &= 0x1F
    gen = np.tile(np.frombuffer(w.g2_b(o.G2_GEN), np.uint8), (16, 1))
    q, inf = c.g2_mul_batch(gen, k)
    assert not inf.any()
    return q


@pytest.fixture(scope="module")
def scalars(hs):  # noqa: F811
    """every scalar class, a few scalars each: {name: [k, ...]}"""
    out = {"edge": X.EDGE_SCALARS}
    for name, classes in (("glv", X.glv_scalars(hs)), ("gls", X.gls_scalars(hs))):
        for cls, ks in classes.items():
            if ks:
                out["%s_%s" % (name, cls)] = ks[:3] + ks[-1:]
    for cls, ks in X.fixed_base_scalars().items():
        out["fixed_" + cls] = ks
    return out


def _all(scalars):
    return [k for ks in scalars.values() for k in ks]


def _scal_r(ks):
    """the scalars reduced mod r for the C oracle, which reads a scalar as an Fp value (mod p); k P = (k mod r) P"""
    return _scal([k % R for k in ks])


# ------------------------------------------------------------------------------------------ Miller loops
@pytest.mark.parametrize("mode, form", [(NEVER, "k_miller"), (ALWAYS, "k_miller_lanes")])
def test_miller_loop_batch_forms(eng, seams, g2pool, monkeypatch, mode, form):  # noqa: F811
    """miller_loop_batch and pairing_batch on every extreme G1 point against random G2 points, on k_miller (one thread
    per pair) and k_miller_lanes (two lanes), several blocks, against the C oracle's Miller loops and pairings."""
    n = 5 * len(EXT) + 3
    g1, g2 = _tile(G1X, n), _tile(g2pool, n)
    plan = _launches(seams.lib, MILLER, n, mode, seams.sms)
    assert [s[4] for s in plan] == [mode == ALWAYS] * len(plan), (form, plan)
    monkeypatch.setenv("SYLOW_B200_LANES", str(mode))
    before = eng.launch_count
    f = eng.miller_loop_batch(g1, g2)
    assert eng.launch_count - before == len(plan), form
    ref = c.miller_loop_batch(g1, g2)
    assert (f == ref).all(), (form, np.flatnonzero((f != ref).any(1))[:8].tolist())
    assert w.b_fp12(bytes(f[1])) == o.miller_loop(o.g2_precompute(w.b_g2(bytes(g2[1]))), EXT[1])
    gt = eng.pairing_batch(g1, g2)
    assert (gt == c.pairing_batch(g1, g2)).all(), form


def test_miller_product_extremes(eng, seams, g2pool):  # noqa: F811
    """miller_product (launch_miller, then product_reduce) over extreme G1 points against random G2 points: equal to
    o.glued_miller_loop on a small batch and to the product of the C oracle's Miller values on several blocks"""
    n = 9
    ps = [EXT[i] for i in range(n)]
    qs = [w.b_g2(bytes(r)) for r in g2pool[:n]]
    got = eng.miller_product(G1X[:n], g2pool[:n])
    assert w.b_fp12(bytes(got)) == o.glued_miller_loop([o.g2_precompute(q) for q in qs], ps)
    n = 7 * len(EXT) + 5
    g1, g2 = _tile(G1X, n), _tile(g2pool, n)
    plan = _launches(seams.lib, MILLER, n, AUTO, seams.sms)
    before = eng.launch_count
    got = eng.miller_product(g1, g2)
    assert eng.launch_count - before == len(plan) + _product_passes(n)[0] + 1, plan
    want = o.FP12_ONE
    for f in c.miller_loop_batch(g1, g2):
        want = o.fp12_mul(want, w.b_fp12(bytes(f)))
    assert w.b_fp12(bytes(got)) == want


def _pow12(f, e):
    r = o.FP12_ONE
    for bit in bin(e)[2:]:
        r = o.fp12_sqr(r)
        if bit == "1":
            r = o.fp12_mul(r, f)
    return r


PRODUCT_T_CAP = 148 * 256  # product_reduce: k_fp12_product_strided runs min(n / 4, this) threads per pass


def _product_passes(n):
    """the k_fp12_product_strided launches of product_reduce over n values, and whether one ran at the thread cap"""
    passes, capped = 0, False
    while n > 1:
        t = max(1, n // 4)
        capped |= t > PRODUCT_T_CAP
        n = min(t, PRODUCT_T_CAP)
        passes += 1
    return passes, capped


def _glue_sizes(seams):  # noqa: F811
    """{glue: n} the smallest n from n = 64 on at which glue_pairs(n, TABLE_COST) picks 1, 2 and 4 pairs per thread
    with one leftover pair (n % glue = 1 for glue > 1)"""
    out, n = {}, 64
    while len(out) < 3:
        g = seams.lib.lp_glue(seams.sms, n, TABLE_COST)
        if g not in out and (g == 1 or n % g == 1):
            out[g] = n
        n += 1
        assert n < 1 << 22
    return out


def test_miller_tables_forms(eng, seams, g2pool):  # noqa: F811
    """g2_precompute(_dev) tables, miller_loop_precomputed_batch (k_miller_tables<1>) and miller_product_precomputed_dev
    at the sizes where glue_pairs runs k_miller_tables<1>, <2> and <4> (with a leftover pair), extreme G1 points against
    resident tables chosen by index: the product equals the product of the C oracle's Miller values."""
    import torch

    dev = torch.device("cuda", 0)
    nq = 5
    tables = eng.g2_precompute(g2pool[:nq])
    d_tab = torch.empty(nq * tables.shape[1], dtype=torch.uint8, device=dev)
    eng.g2_precompute_dev(torch.from_numpy(g2pool[:nq]).to(dev), d_tab)
    m = 3 * len(EXT)
    g1 = _tile(G1X, m)
    tq = np.arange(m) % nq
    f1 = eng.miller_loop_precomputed_batch(tables[tq], g1)
    mill = c.miller_loop_batch(np.concatenate([G1X] * nq), np.repeat(g2pool[:nq], len(EXT), axis=0))
    val = {(i, j): mill[j * len(EXT) + i] for i in range(len(EXT)) for j in range(nq)}
    assert all((f1[t] == val[t % len(EXT), tq[t]]).all() for t in range(m)), "k_miller_tables<1>"
    for glue, n in sorted(_glue_sizes(seams).items()):
        pi, qi = np.arange(n) % len(EXT), (np.arange(n) // 7) % nq
        idx = torch.from_numpy(qi.astype(np.int32)).to(dev)
        d_g1 = torch.from_numpy(G1X[pi]).to(dev)
        d_out = torch.empty(384, dtype=torch.uint8, device=dev)
        before = eng.launch_count
        eng.miller_product_precomputed_dev(d_tab, d_g1, d_out, d_table_idx=idx)
        launches = eng.launch_count - before
        got = w.b_fp12(bytes(d_out.cpu().numpy()))
        counts = {}
        for a, b in zip(pi.tolist(), qi.tolist()):
            counts[a, b] = counts.get((a, b), 0) + 1
        want = o.FP12_ONE
        for (a, b), e in counts.items():
            want = o.fp12_mul(want, _pow12(w.b_fp12(bytes(val[a, b])), e))
        # k_miller_tables<glue> over n // glue items, a k_miller_tables<1> launch for the leftover pair, product_reduce's
        # passes over the item and leftover values and its conversion to canonical form
        left = n % glue
        assert launches == 1 + (left > 0) + _product_passes(n // glue + left)[0] + 1, (glue, n, launches)
        print("n = %d: k_miller_tables<%d> + %d leftover, %d launches" % (n, glue, n % glue if glue > 1 else 0,
                                                                        launches))
        assert got == want, (glue, n)
        if glue == 1:
            host = eng.miller_product_precomputed(tables[qi], G1X[pi])
            assert w.b_fp12(bytes(host)) == want


# ------------------------------------------------------------------------------------------ checks with verdicts
def _extreme_checks(g2pool, k, n_checks):
    """n_checks checks of k pairs: pairs (P, Q), (-P, Q) per two, P extreme; check c fails when c % 3 == 1 (the last
    pair's Q replaced by another point) and, for k = 2, has pair 0's G1 flagged infinite when c % 7 == 3 (fails:
    e(-P, Q) is left) or both pairs' G2 flagged when c % 7 == 5 (holds: both skipped)"""
    n = k * n_checks
    cc = np.arange(n_checks)
    pi = (np.arange(n) // 2 * 5 + cc.repeat(k)) % len(EXT)
    pi[1::2] = [NEG[i] for i in pi[0::2]]
    qi = (np.arange(n) // 2) % (len(g2pool) - 1)
    bad = cc % 3 == 1
    last = cc * k + k - 1
    qi[last[bad]] = len(g2pool) - 1
    g1_inf, g2_inf = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    expect = ~bad
    if k == 2:
        br, sk = (cc % 7 == 3) & ~bad, (cc % 7 == 5)
        g1_inf[cc[br] * k] = 1
        expect = expect & ~br
        g2_inf[cc[sk] * k] = g2_inf[cc[sk] * k + 1] = 1
        expect = expect | sk
    return G1X[pi], g1_inf, g2pool[qi], g2_inf, expect


@pytest.mark.parametrize("k, base, off", [(2, "L", 0), (2, "L", 1), (2, "W", -1), (2, "W", 0), (4, "L", -1),
                                          (4, "L", 0)])
def test_pairing_check_seams_extreme(eng, seams, g2pool, k, base, off):  # noqa: F811
    """pairing_check_batch_dev on both sides of the two-lane / fused k_check_products seam L and of the glued-2 seam W,
    and k_glued<4, 0> from L 4-pair checks, on extreme G1 points: [(P, Q), (-P, Q)] holds, another Q fails, flagged
    pairs are skipped."""
    import torch

    n_checks = getattr(seams, base) + off
    launches, _, form = _plan(seams, k, n_checks, AUTO)
    print("k = %d, %d checks: %s" % (k, n_checks, form))
    g1, g1_inf, g2, g2_inf, expect = _extreme_checks(g2pool, k, n_checks)
    dev = torch.device("cuda", 0)
    d = [torch.from_numpy(x).to(dev) for x in (g1, g2, g1_inf, g2_inf)]
    d_ok = torch.zeros(n_checks, dtype=torch.uint8, device=dev)
    before = eng.launch_count
    eng.pairing_check_batch_dev(d[0], d[1], k, d_ok, d_g1_inf=d[2], d_g2_inf=d[3])
    assert eng.launch_count - before == launches, form
    got = d_ok.cpu().numpy().astype(bool)
    assert (got == expect).all(), (form, np.flatnonzero(got != expect)[:16].tolist())
    m = 40 * k
    assert eng.pairing_check_batch(g1[:m], g2[:m], k, g1_inf[:m], g2_inf[:m]).tolist() == expect[:40].tolist()


def test_pairing_check_ragged_extreme(eng, g2pool):
    """pairing_check_ragged_batch over checks of 0 .. 6 pairs of extreme points: cancelling pairs (P, Q), (-P, Q), an
    odd pair flagged infinite; every third check has one Q replaced and fails.  (The values only: the ragged plan's
    launch forms are covered by test_gpu_ragged_check.py.)"""
    g1, g1_inf, g2, g2_inf, offs, expect = [], [], [], [], [0], []
    rng = random.Random(5)
    for cidx in range(300):
        s = cidx % 7
        fail = cidx % 3 == 1 and s > 0
        for j in range(s // 2):
            i = rng.randrange(len(EXT))
            q = rng.randrange(len(g2pool) - 1)
            g1 += [G1X[i], G1X[NEG[i]]]
            g2 += [g2pool[q], g2pool[len(g2pool) - 1 if fail and j == 0 else q]]
            g1_inf += [0, 0]
            g2_inf += [0, 0]
        if s % 2:
            g1.append(G1X[rng.randrange(len(EXT))])
            g2.append(g2pool[0])
            g1_inf.append(0)
            g2_inf.append(0 if fail and s == 1 else 1)
        offs.append(len(g1))
        expect.append(not fail)
    ok = eng.pairing_check_ragged_batch(np.array(g1), np.array(g2), np.array(offs, np.uint64),
                                        np.array(g1_inf, np.uint8), np.array(g2_inf, np.uint8))
    assert ok.tolist() == expect


def _g1_be(p):
    return p[0].to_bytes(32, "big") + p[1].to_bytes(32, "big")


def _g2_be(q):
    return b"".join(x.to_bytes(32, "big") for x in (q[0][1], q[0][0], q[1][1], q[1][0]))


def test_eip197_wire_extremes(eng, g2pool):
    """eip197_pairing_check_batch on the wire-extreme points: (P, Q), (-P, Q) holds, another Q fails, x = p is
    ERR_DECODE."""
    qs = [w.b_g2(bytes(r)) for r in g2pool[:2]]
    rows, ok_want, st_want = [], [], []
    for p in X.g1_wire_extremes():
        rows.append(_g1_be(p) + _g2_be(qs[0]) + _g1_be(o.g1_affine_neg(p)) + _g2_be(qs[0]))
        rows.append(_g1_be(p) + _g2_be(qs[0]) + _g1_be(o.g1_affine_neg(p)) + _g2_be(qs[1]))
        rows.append(o.P.to_bytes(32, "big") + p[1].to_bytes(32, "big") + rows[-1][64:])
        ok_want += [True, False, False]
        st_want += [0, 0, ERR_DECODE]
    ok, st = eng.eip197_pairing_check_batch(arr(rows), 2)
    assert ok.tolist() == ok_want and st.tolist() == st_want


# ------------------------------------------------------------------------------------------ G1 group law and ladders
def test_g1_mul_extreme_points_and_scalars(eng, scalars):
    """g1_mul_batch (GLV) on every extreme point times every scalar class, and eip196_mul_batch on the same, against
    the C oracle's double-and-add."""
    ks = _all(scalars)
    pi = np.repeat(np.arange(len(EXT)), len(ks))
    K = _scal(ks * len(EXT))
    pts = G1X[pi]
    out, inf = eng.g1_mul_batch(pts, K)
    ref, rinf = c.g1_mul_batch(pts, _scal_r(ks * len(EXT)))
    bad = np.flatnonzero((out != ref).any(1) | (inf != rinf))
    assert not len(bad), [(EXT[pi[i]][:2], hex(int.from_bytes(bytes(K[i]), "little"))) for i in bad[:4]]
    sel = np.arange(0, len(pi), 97)
    be = arr([_g1_be(EXT[pi[i]]) + int.from_bytes(bytes(K[i]), "little").to_bytes(32, "big") for i in sel])
    e_out, st = eng.eip196_mul_batch(be)
    assert (st == 0).all()
    want = [bytes(64) if rinf[i] else _g1_be(w.b_g1(bytes(ref[i]))) for i in sel]
    assert [bytes(r) for r in e_out] == want


def _aff(p):
    return o.proj_to_affine(o.FpOps, p)


def _add(a, b):
    return _aff(o.proj_add(o.FpOps, o.affine_to_proj(o.FpOps, a), o.affine_to_proj(o.FpOps, b)))


def test_g1_add_extremes(eng):
    """g1_add_batch and eip196_add_batch: P + P, P - P, P + Q and P - Q over the extreme points"""
    n = len(EXT)
    a = np.concatenate([G1X] * 3)
    b = np.concatenate([G1X, G1X[[(i + 5) % n for i in range(n)]], G1X[[NEG[i] for i in range(n)]]])
    pa = [w.b_g1(bytes(r)) for r in a]
    pb = [w.b_g1(bytes(r)) for r in b]
    for sub in (False, True):
        out, inf = eng.g1_add_batch(a, b, subtract=sub)
        want = [_add(x, o.g1_affine_neg(y) if sub else y) for x, y in zip(pa, pb)]
        assert [w.b_g1(bytes(r), i) for r, i in zip(out, inf)] == want, sub
    e_out, st = eng.eip196_add_batch(arr([_g1_be(x) + _g1_be(y) for x, y in zip(pa, pb)]))
    assert (st == 0).all()
    assert [bytes(r) for r in e_out] == [bytes(64) if s[2] else _g1_be(s) for s in (_add(x, y) for x, y in zip(pa, pb))]


def _sum_ref(pairs):
    """sum of k P over (point index, k) pairs, by the oracle, grouped by point"""
    by = {}
    for i, k in pairs:
        by[i] = (by.get(i, 0) + k) % R
    acc = o.proj_zero(o.FpOps)
    for i, k in by.items():
        acc = o.proj_add(o.FpOps, acc, o.proj_mul(o.FpOps, o.affine_to_proj(o.FpOps, EXT[i]), k))
    return _aff(acc)


def test_g1_sum_and_msm_extremes(eng, scalars):
    """g1_sum, g1_msm and g1_msm_bucket at several window sizes over extreme points with the scalar classes, 2^256 - 1
    everywhere (digit 2^c - 1 in every window, the partial top window too), and 255, 256, 257 equal scalars (one bucket
    of one and two SY_MSM_ITEM work items)."""
    ks = _all(scalars)
    n = len(ks)
    pi = np.arange(n) % len(EXT)
    P, K = G1X[pi], _scal(ks)
    s, sinf = eng.g1_sum(P)
    assert w.b_g1(bytes(s), sinf) == _sum_ref([(i, 1) for i in pi.tolist()])
    ref = _sum_ref(list(zip(pi.tolist(), ks)))
    assert w.b_g1(bytes(eng.g1_msm(P, K)[0]), 0) == ref
    for cbits in X.MSM_WINDOWS:
        before = eng.launch_count
        out, inf = eng.g1_msm_bucket(P, K, window_bits=cbits)
        # count, offsets, scatter, conversion, item sums, bucket sums, chunk reduction, window sums, Horner, affine
        assert eng.launch_count - before == MSM_BUCKET_LAUNCHES, cbits
        assert w.b_g1(bytes(out), inf) == ref, cbits
    top = (1 << 256) - 1
    for m in (255, 256, 257, 2 * 256 + 1):
        # every window's bucket 2^c - 1 (2^(256 mod c) - 1 in a partial top window) holds all m points: one work item of
        # SY_MSM_ITEM = 256 points for 255 and 256, two for 257, three for 513
        assert -(-m // MSM_ITEM) == {255: 1, 256: 1, 257: 2, 513: 3}[m]
        assert all(set(X.msm_digits(top, cb)[:-1]) == {(1 << cb) - 1} for cb in (5, 8, 11, 16))
        pm = np.arange(m) % len(EXT)
        want = _sum_ref([(i, top) for i in pm.tolist()])
        for cbits in (5, 8, 11, 16):
            out, inf = eng.g1_msm_bucket(G1X[pm], _scal([top] * m), window_bits=cbits)
            assert w.b_g1(bytes(out), inf) == want, (m, cbits)
        # one point repeated: every digit's bucket holds all m copies
        same = np.zeros(m, np.int64)
        want = _sum_ref([(0, top)] * m)
        for cbits in (4, 13):
            out, inf = eng.g1_msm_bucket(G1X[same], _scal([top] * m), window_bits=cbits)
            assert w.b_g1(bytes(out), inf) == want, (m, cbits, "same point")


def test_threshold_aggregate_extreme_shares(eng):
    """threshold_aggregate_batch with extreme points as the partial signatures (t = 3 and t = 40)"""
    rng = random.Random(9)
    for n_sets, t in ((6, 3), (2, 40)):
        ids = [rng.sample(range(1, 1000), t) for _ in range(n_sets)]
        idx = [[(s * 7 + j) % len(EXT) for j in range(t)] for s in range(n_sets)]
        S = np.stack([G1X[row] for row in idx])
        out, inf = eng.threshold_aggregate_batch(np.array(ids, np.uint64), S)
        for s in range(n_sets):
            assert w.b_g1(bytes(out[s]), inf[s]) == o.threshold_aggregate(ids[s], [EXT[i] for i in idx[s]])


def test_g1_validate_and_codecs_extremes(eng):
    """g1_validate_batch accepts every extreme point and rejects x = p; the big-endian codecs round-trip them"""
    st = eng.g1_validate_batch(G1X)
    assert (st == 0).all()
    over = arr([w.fp_b(o.P) + w.fp_b(p[1]) for p in X.g1_wire_extremes()])
    assert (eng.g1_validate_batch(over) == ERR_DECODE).all()
    enc = eng.g1_to_be_bytes_batch(G1X)
    assert [bytes(r) for r in enc] == [_g1_be(p) for p in EXT]
    out, inf, st = eng.g1_from_be_bytes_batch(enc)
    assert (st == 0).all() and not inf.any() and (out == G1X).all()
    out, inf, st = eng.g1_from_be_bytes_batch(enc, eip_mode=True)
    assert (st == 0).all() and (out == G1X).all()


# ------------------------------------------------------------------------------------------ other ladders
def test_g2_mul_gls_and_gt_pow_edges(eng, scalars, g2pool):
    """g2_mul_batch (GLS) and gt_mul_batch (gt_pow, the same split) with every scalar class: against the C oracle's
    G2 double-and-add and against the C oracle's pairing e(k P, Q) = e(P, Q)^k on extreme P"""
    ks = _all(scalars)
    n = len(ks)
    Q, K = _tile(g2pool, n), _scal(ks)
    out, inf = eng.g2_mul_batch(Q, K)
    ref, rinf = c.g2_mul_batch(Q, _scal_r(ks))
    assert (out == ref).all() and (inf == rinf).all()
    g1 = _tile(G1X, n)
    gt = eng.pairing_batch(g1, Q)
    got = eng.gt_mul_batch(gt, K)
    kp, kp_inf = c.g1_mul_batch(g1, _scal_r(ks))
    want = c.pairing_batch(kp, Q, g1_inf=kp_inf)
    bad = np.flatnonzero((got != want).any(1))
    assert not len(bad), [hex(ks[i]) for i in bad[:4]]
    for i in (0, n // 2, n - 1):
        assert w.b_fp12(bytes(got[i])) == o.gt_mul(w.b_fp12(bytes(gt[i])), ks[i] % R)


def test_generator_mul_fixed_base_edges(eng, scalars):
    """g1/g2_mul_generator_batch (scalar_reduce_r + scalar_digit<8>) with every scalar class against the C oracle"""
    ks = _all(scalars)
    K = _scal(ks)
    for g, gen, mul in (("g1", w.g1_b(o.G1_GEN), c.g1_mul_batch), ("g2", w.g2_b(o.G2_GEN), c.g2_mul_batch)):
        out, inf = getattr(eng, g + "_mul_generator_batch")(K)
        ref, rinf = mul(np.tile(np.frombuffer(gen, np.uint8), (len(ks), 1)), _scal_r(ks))
        bad = np.flatnonzero((out != ref).any(1) | (inf != rinf))
        assert not len(bad), (g, [hex(ks[i]) for i in bad[:4]])


# ------------------------------------------------------------------------------------------ extreme Fp12 partials
def test_fp12_product_extremes(eng):
    """fp12_product (k_fp12_product_strided, T = n / 4 threads per pass, at most 148 * 256) over extreme values at
    lengths around 4 T and around the cap"""
    vals = X.fp12_extremes()
    V = arr([w.fp12_b(v) for v in vals])
    cap = 4 * PRODUCT_T_CAP
    capped = []
    for n in (1, 3, 4, 5, 7, 8, 9, 255, 257, cap - 1, cap, cap + 1, cap + 3, cap + 4, cap + 5):
        idx = np.arange(n) % len(vals)
        want = o.FP12_ONE
        cnt = np.bincount(idx, minlength=len(vals))
        for i in np.flatnonzero(cnt):
            want = o.fp12_mul(want, _pow12(vals[i], int(cnt[i])))
        before = eng.launch_count
        got = eng.fp12_product(V[idx])
        passes, at_cap = _product_passes(n)
        # the conversion to Montgomery form, the strided passes, the conversion back
        assert eng.launch_count - before == 1 + passes + 1, n
        capped.append(at_cap)
        assert w.b_fp12(bytes(got)) == want, n
    assert capped[-3:] == [False, True, True], "the thread cap is reached from n = 4 (148 * 256 + 1) values on"


def test_verify_batch_finish_extremes(eng):
    """verify_batch_finish on partials a and a^-1 for extreme a: the product is 1, so True; one coefficient of a^-1
    changed: the verdict of the C oracle's final exponentiation of the product (False unless the product falls into a
    subfield the final exponentiation sends to 1), and False for at least one of them"""
    vals = [v for v in X.fp12_extremes()[:40] if v != o.fp12_from_list([0] * 12)][:20]
    one = w.fp12_b(o.FP12_ONE)
    bads, prods = [], []
    for i, v in enumerate(vals):
        inv = o.fp12_inv(v)
        assert eng.verify_batch_finish(arr([w.fp12_b(v), w.fp12_b(inv)])) is True
        bad = o.fp12_to_list(inv)
        bad[i % 12] = (bad[i % 12] + 1) % o.P
        bads.append(o.fp12_from_list(bad))
        prods.append(w.fp12_b(o.fp12_mul(v, bads[-1])))
    want = [bytes(r) == one for r in c.final_exp_batch(arr(prods))]
    got = [eng.verify_batch_finish(arr([w.fp12_b(v), w.fp12_b(b)])) for v, b in zip(vals, bads)]
    assert got == want and not all(want)


# ------------------------------------------------------------------------------------------ G2 off the subgroup
def test_g2_extreme_coordinates_off_subgroup(eng):
    """twist points with x = (p - 1 - i, p - 1 - j) are almost never in G2: g2_validate_batch gives ERR_NOT_IN_SUBGROUP
    (-4), the big-endian encoder writes them and the decoder
    gives the same status (no pairing value is asserted on them: outside the contract)"""
    pts = []
    for i in range(40):
        x = (o.P - 1 - i, o.P - 1 - (i * 7) % 11)
        y = o.fp2_sqrt(o.fp2_add(o.fp2_mul(o.fp2_sqr(x), x), o.FP2_TWIST_CURVE_CONSTANT))
        if y is not None:
            pts += [(x, y), (x, o.fp2_neg(y))]
    assert len(pts) >= 4
    raw = arr([w.g2_b((x, y)) for x, y in pts])
    assert (eng.g2_validate_batch(raw) == -4).all()
    enc = eng.g2_to_be_bytes_batch(raw)
    assert [bytes(r) for r in enc] == [_g2_be(q) for q in pts]
    out, inf, st = eng.g2_from_be_bytes_batch(enc)
    assert (st == -4).all() and not inf.any()


# ------------------------------------------------------------------------------------------ Groth16 public inputs
def test_groth16_fold_fixed_base_edges(eng):
    """groth16_verify_each and groth16_verify_batch with public inputs from the fixed-base digit classes (inputs < r:
    the fold gen_scalar_mul_add walks the IC tables from a non-zero accumulator) and r - 1, 0, 1, against the verdicts
    of tests/groth16_ref.py: valid proofs hold, a proof with one input changed by one fails, an input r fails."""
    from tests import groth16_ref as g

    ins = [k for ks in X.fixed_base_scalars().values() for k in ks if k < R] + [R - 1, 0, 1, R - 2]
    l = 3
    td = g.Trapdoor(l, 71)
    vk_pts = td.vk()
    vk = np.frombuffer(g.vk_bytes(vk_pts), np.uint8).copy()
    xs = [[ins[(3 * i + j) % len(ins)] for j in range(l)] for i in range(len(ins))]
    proofs = []
    for row in xs:
        a, b, cc = td.proof_scalars(row)
        proofs.append((g.g1_mul(a), g.g2_mul(b), g.g1_mul(cc)))
    expect = [True] * len(xs)
    # a proof for other inputs: the input changed by one after proving; an input equal to r
    xs[1] = [xs[1][0], (xs[1][1] + 1) % R, xs[1][2]]
    xs[-1] = [R, xs[-1][1], xs[-1][2]]
    expect[1] = expect[-1] = False
    P = arr([g.proof_bytes(p) for p in proofs])
    X_ = arr([b"".join(x.to_bytes(32, "little") for x in row) for row in xs])
    got = eng.groth16_verify_each(vk, P, X_, l)
    assert got.tolist() == expect
    for i in (0, 1, len(xs) - 1):
        assert g.groth16_verify(vk_pts, proofs[i], xs[i]) is expect[i], i
    ok = [i for i, e in enumerate(expect) if e]
    assert eng.groth16_verify_batch(vk, P[ok], X_[ok], l, bytes(range(32))) is True
    assert eng.groth16_verify_batch(vk, P, X_, l, bytes(range(32))) is False

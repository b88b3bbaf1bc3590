"""GPU tier (-m gpu): the boolean verdicts of the pairing checks and BLS verification on both sides of every switch
between launch forms.  Each entry point picks its kernels by batch size, pairs per check and SM count (launch_plan.h);
the seams are derived at run time from this GPU's SM count through the host build of the launch policy
(tests/hostsim/launch_plan.cu), and every case asserts, through the context's launch count, that it reached the form it
is meant to test.  Inputs are multiples of the generators with scalars chosen so that each check's product is known:
pairs (a_j G1, b_j G2) with sum_j a_j b_j = 0 mod r cancel; invalid checks, infinite pairs that break a check and
infinite pairs that leave it cancelling are planted at the first and last item of every launch segment and block.
Verdicts are compared with that construction and, on a sample, with the oracle's glued_pairing."""
import random
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import bn254_py as o
from tests import wire as w
from tests.test_launch_plan import AUTO, MILLER, NEVER, _check, _launches, load_launch_plan

pytestmark = pytest.mark.gpu
R = o.R_ORDER
POOL = 64  # distinct G2 points b_i G2 the checks draw from
PAIR_COST = 8444  # verify_partial_core's cost of one fused pair for glue_pairs
SEED = bytes(range(7, 39))  # weight seed of the weighted verification cases


@pytest.fixture(scope="module")
def eng():
    import sylow_b200

    e = sylow_b200.Engine(0)
    yield e
    e.close()


def _first(pred, hi):
    """smallest n in [1, hi] with pred(n), for pred false below some n and true from there on"""
    lo = 1
    assert pred(hi)
    while lo < hi:
        mid = (lo + hi) // 2
        if pred(mid):
            hi = mid
        else:
            lo = mid + 1
    return lo


@pytest.fixture(scope="module")
def seams(tmp_path_factory):
    """The launch-form seams on this GPU: L (largest batch of one two-lane wave: check products on two lanes up to L
    checks, fused k_check_products above), W (2-pair checks glued into one loop from W checks on), and the batch
    sizes at which verify_partial_core glues 2 and 4 pairs per thread with n % glue = 1, 2, 3 leftover pairs."""
    import torch

    lib = load_launch_plan(tmp_path_factory.mktemp("launch_plan"))
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    lanes = lambda n: _check(lib, n, AUTO, sms)[4]
    glued = lambda k, n: bool(lib.lp_check_glued(sms, k, n))
    L = _first(lambda n: not lanes(n), 1 << 30) - 1
    W = _first(lambda n: glued(2, n), 1 << 30)
    assert lanes(L) and not lanes(L + 1) and not glued(2, W - 1) and glued(2, W)
    assert not glued(4, L - 1) and glued(4, L), "4-pair checks are glued from one two-lane wave of checks on"
    first = {}  # glue_pairs is not monotone in n (a whole number of waves of single pairs beats glued ones)
    n = 0
    while 4 not in first:
        n += 1
        first.setdefault(lib.lp_glue(sms, n, PAIR_COST), n)
        assert n < 64 * W
    verify = {}
    for glue, r in ((2, 1), (4, 1), (4, 2), (4, 3)):
        n = first[glue]
        while lib.lp_glue(sms, n, PAIR_COST) != glue or n % glue != r:
            n += 1
        assert lib.lp_glue(sms, n + glue - r, PAIR_COST) == glue
        verify[glue, r] = n
    if sms == 148:  # a B200: the seams the launch policy documents
        assert (L, W, first[2], first[4]) == (18944, 37888, 37889, 113665)
        assert verify == {(2, 1): 37889, (4, 1): 113665, (4, 2): 113666, (4, 3): 113667}
    return SimpleNamespace(lib=lib, sms=sms, L=L, W=W, verify=verify)


def _le(xs):
    """integers in [0, 2^256) as (n, 32) little-endian rows"""
    return np.frombuffer(b"".join(x.to_bytes(32, "little") for x in xs), np.uint8).reshape(-1, 32).copy()


def _scal(xs):
    return _le([x % R for x in xs])


@pytest.fixture(scope="module")
def pool(eng):
    """(b, b^-1 mod r, the points b G2) for POOL random scalars b"""
    rng = random.Random(300)
    b = [rng.randrange(1, R) for _ in range(POOL)]
    q, q_inf = eng.g2_mul_generator_batch(_scal(b))
    assert not q_inf.any()
    return b, [pow(x, -1, R) for x in b], q


def _edges(segments):
    """the first and last item of every launch segment and, where there are several blocks, the last item of its first
    block and the first of its second"""
    out = set()
    for first, count, blocks, threads, lanes in segments:
        per = threads // 2 if lanes else threads
        out |= {first, first + count - 1}
        if blocks > 1:
            out |= {first + per - 1, first + per}
    return out


def _plant(rng, k, n_checks, bad_pairs, bad_checks):
    """(bad pairs, breaks, cancels): the given pairs, one pair of each given check and a few random checks invalid;
    a few other checks broken or left cancelling by an infinite pair (breaks only with k >= 2: a 1-pair check holds only
    when its pair is infinite)"""
    bad = set(bad_pairs) | {c * k + rng.randrange(k) for c in bad_checks}
    free = sorted(set(range(n_checks)) - {p // k for p in bad})
    rng.shuffle(free)
    m = min(8, len(free) // 4)
    bad |= {c * k + rng.randrange(k) for c in free[:m]}
    return bad, (free[m:2 * m] if k > 1 else []), free[2 * m:3 * m]


def _checks(eng, pool, k, n_checks, bad, breaks=(), cancels=(), fixed=None, g2_flags=True, seed=0):
    """n_checks checks of k pairs (a_p G1, b_p G2), pair p = c k + j, with sum_j a_p b_p = 0 mod r, except:
    bad: pairs whose a_p is one more (their check fails); breaks: checks whose pair 0 is flagged infinite (its factor
    is missing, the check fails); cancels: checks whose pair 0 is flagged infinite and left out of the sum (the check
    holds).  The flags alternate between G1 and G2 unless g2_flags is false.  fixed: the pool index of every check's
    last G2 point.  Returns (g1, g1_inf, g2, g2_inf, expected verdicts); a 0 scalar gives an infinite G1 point."""
    rng = random.Random(seed)
    b, binv, q = pool
    n = k * n_checks
    idx = np.array([rng.randrange(POOL) for _ in range(n)])
    if fixed is not None:
        idx[k - 1::k] = fixed
    a = [rng.getrandbits(253) | 1 for _ in range(n)]
    g1_flag, g2_flag = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    for i, c in enumerate(sorted(set(breaks) | set(cancels))):
        (g2_flag if g2_flags and i % 2 else g1_flag)[c * k] = 1
    dropped = set(cancels)
    for c in range(n_checks):
        p = c * k
        if k == 1 and c in dropped:
            continue  # the check's only pair is flagged: any scalar
        s = sum(a[p + j] * b[idx[p + j]] for j in range(k - 1) if not (j == 0 and c in dropped))
        a[p + k - 1] = -s * binv[idx[p + k - 1]] % R
    for p in bad:
        a[p] += 1
    g1, g1_inf = eng.g1_mul_generator_batch(_scal(a))
    expect = np.ones(n_checks, bool)
    expect[sorted({p // k for p in bad})] = False
    expect[list(breaks)] = False
    assert not (set(cancels) & {p // k for p in bad})
    return g1, g1_inf | g1_flag, q[idx], g2_flag, expect


def _oracle_agrees(g1, g1_inf, g2, g2_inf, k, expect, checks):
    """glued_pairing of each sampled check's finite pairs == 1 (an infinite pair contributes 1) against expect"""
    for c in checks:
        pairs = [(w.b_g1(bytes(g1[p])), w.b_g2(bytes(g2[p]))) for p in range(c * k, c * k + k)
                 if not (g1_inf[p] or g2_inf[p])]
        got = o.glued_pairing([x for x, _ in pairs], [y for _, y in pairs]) == o.FP12_ONE
        assert got == bool(expect[c]), (k, c)


def _sample(rng, expect, bad, breaks, cancels, k):
    picks = sorted({p // k for p in bad})[:3] + list(breaks[:2]) + list(cancels[:2])
    valid = [c for c in np.flatnonzero(expect) if c not in cancels]
    return sorted(set(picks + rng.sample(valid, min(2, len(valid)))))


def _plan(s, k, n_checks, mode):
    """(kernel launches, Miller launch segments or None for one glued loop, description) of pairing_check_batch:
    the Miller values (one glued loop per check, or launch_miller's segments over the pairs), then launch_check_products
    (two lanes: k_group_products when a check has several values, k_final_exp_lanes, k_gt_is_one; else one fused
    k_check_products)"""
    if s.lib.lp_check_glued(s.sms, k, n_checks):
        segs, miller, k_prod, desc = None, 1, 1, "one glued loop per check"
    else:
        segs = _launches(s.lib, MILLER, k * n_checks, mode, s.sms)
        miller, k_prod = len(segs), k
        desc = "launch_miller %s" % ["two lanes" if g[4] else "%d threads" % g[3] for g in segs]
    if _check(s.lib, n_checks, mode, s.sms)[4]:
        return miller + 2 + (k_prod > 1), segs, desc + " + two-lane check products, %d values per check" % k_prod
    return miller + 1, segs, desc + " + fused k_check_products, %d values per check" % k_prod


# ------------------------------------------------------------------------------------------ (a) pairing_check_batch
@pytest.mark.parametrize("k, base, off", [
    (2, "L", 0), (2, "L", 1), (2, "W", -1), (2, "W", 0),
    (4, "L", -1), (4, "L", 0), (4, "L", 1),
    (1, "L", 0), (1, "L", 1), (3, "L", 0), (3, "L", 1), (5, "L", 0), (5, "L", 1),
])
def test_pairing_check_seams(eng, seams, pool, k, base, off):
    """pairing_check_batch_dev under the default policy on both sides of the two-lane seam L and the glued seam W:
    two-lane products with and without k_group_products, fused k_check_products multiplying k Miller values, one glued
    loop per check with two-lane or fused products."""
    import torch

    n_checks = getattr(seams, base) + off
    launches, segs, form = _plan(seams, k, n_checks, AUTO)
    print("k = %d, %d checks: %s" % (k, n_checks, form))
    rng = random.Random(1000 * k + off)
    checks = _edges([_check(seams.lib, n_checks, AUTO, seams.sms)]) | {0, n_checks - 1}
    bad, breaks, cancels = _plant(rng, k, n_checks, _edges(segs) if segs else (), checks)
    g1, g1_inf, g2, g2_inf, expect = _checks(eng, pool, k, n_checks, bad, breaks, cancels, seed=k * 7 + off)
    dev = torch.device("cuda", 0)
    d = [torch.from_numpy(x).to(dev) for x in (g1, g2, g1_inf, g2_inf)]
    d_ok = torch.zeros(n_checks, dtype=torch.uint8, device=dev)
    before = eng.launch_count
    eng.pairing_check_batch_dev(d[0], d[1], k, d_ok, d_g1_inf=d[2], d_g2_inf=d[3])
    assert eng.launch_count - before == launches, form
    got = d_ok.cpu().numpy().astype(bool)
    assert (got == expect).all(), (form, np.flatnonzero(got != expect)[:16].tolist())
    # the host-buffer entry point on a prefix (a small batch: the separate Miller values on two lanes)
    m = 32 * k
    assert eng.pairing_check_batch(g1[:m], g2[:m], k, g1_inf[:m], g2_inf[:m]).tolist() == expect[:32].tolist()
    _oracle_agrees(g1, g1_inf, g2, g2_inf, k, expect, _sample(rng, expect, bad, breaks, cancels, k))


# ------------------------------------------------------------------------------------------ (b) fused products, small
@pytest.mark.parametrize("k", [1, 2, 3, 5])
def test_pairing_check_fused_products_small_batches(eng, seams, pool, monkeypatch, k):
    """SYLOW_B200_LANES=0 sends small batches through the fused k_check_products (k Miller values multiplied in the
    kernel); its verdicts equal the two-lane form's (=1) and the construction."""
    for n_checks in (5, 33, 150):
        rng = random.Random(2000 * k + n_checks)
        segs = _launches(seams.lib, MILLER, k * n_checks, NEVER, seams.sms)
        bad, breaks, cancels = _plant(rng, k, n_checks, _edges(segs), {0, n_checks - 1})
        g1, g1_inf, g2, g2_inf, expect = _checks(eng, pool, k, n_checks, bad, breaks, cancels, seed=n_checks + k)
        got = {}
        for mode in (NEVER, AUTO):
            monkeypatch.setenv("SYLOW_B200_LANES", str(mode))
            launches, _, form = _plan(seams, k, n_checks, mode)
            assert ("fused" in form) == (mode == NEVER), form
            before = eng.launch_count
            got[mode] = eng.pairing_check_batch(g1, g2, k, g1_inf, g2_inf)
            assert eng.launch_count - before == launches, form
        assert got[NEVER].tolist() == got[AUTO].tolist() == expect.tolist(), (k, n_checks)
        _oracle_agrees(g1, g1_inf, g2, g2_inf, k, expect, _sample(rng, expect, bad, breaks, cancels, k)[:4])


# ------------------------------------------------------------------------------------------ BLS verification
@pytest.fixture(scope="module")
def signed(eng, seams):
    """Key pairs, distinct 32-byte messages, their signatures and message hashes, enough for every seam below."""
    n = max(max(v + g - r for (g, r), v in seams.verify.items()), seams.L + 2)
    rs = np.random.RandomState(400)
    sks = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
    sks[:, 31] &= 0x1F  # < 2^253 < r
    sks[:, 0] |= 1
    msgs = np.zeros((n, 32), np.uint8)
    msgs[:, :8] = np.arange(n, dtype=np.uint64).view(np.uint8).reshape(n, 8)
    msgs[:, 8:] = rs.randint(0, 256, size=(n, 24), dtype=np.uint8)
    offs = np.arange(n + 1, dtype=np.uint64) * 32
    sigs = eng.sign_batch(sks, (msgs.reshape(-1), offs))
    pks, pks_inf = eng.g2_mul_generator_batch(sks)
    hm, hm_inf = eng.hash_to_g1_batch((msgs.reshape(-1), offs))
    assert not pks_inf.any() and not hm_inf.any()
    return SimpleNamespace(msgs=msgs, offs=offs, sigs=sigs, pks=pks, hm=hm)


def _packed(msgs):
    return msgs.reshape(-1), np.arange(msgs.shape[0] + 1, dtype=np.uint64) * 32


def _ints(k):
    w64 = k.view("<u8").reshape(-1, 4)
    return [int(a) | (int(b) << 64) | (int(c) << 128) | (int(d) << 192) for a, b, c, d in w64]


def _partial_reference(eng, S, n, pks_inf, sigs_inf, seed, first_index):
    """miller_product over the explicit pairs (-r_i H(m_i), pk_i) for i < n and (sum_i r_i sig_i, G2gen): the partial
    of verify_batch_partial, bit for bit (Fp12 multiplication is exact and commutative); r_i = 1 unweighted"""
    if seed is None:
        hm, hm_inf = S.hm[:n], np.zeros(n, np.uint8)
        s, s_inf = eng.g1_sum(S.sigs[:n], sigs_inf)
    else:
        r = np.zeros((n, 32), np.uint8)
        r[:, :8] = eng.batch_weights(seed, first_index, n).view(np.uint8).reshape(n, 8)
        hm, hm_inf = eng.g1_mul_batch(S.hm[:n], r)
        s, s_inf = eng.g1_msm(S.sigs[:n], r, sigs_inf)
    neg = hm.copy()
    neg[:, 32:] = _le([(o.P - y) % o.P for y in _ints(np.ascontiguousarray(hm[:, 32:]))])  # y -> p - y
    g1 = np.concatenate([neg, s.reshape(1, 64)])
    g2 = np.concatenate([S.pks[:n], np.frombuffer(w.g2_b(o.G2_GEN), np.uint8).reshape(1, 128)])
    g1_inf = np.concatenate([hm_inf, [s_inf]]).astype(np.uint8)
    g2_inf = np.concatenate([pks_inf, [0]]).astype(np.uint8)
    return eng.miller_product(g1, g2, g1_inf=g1_inf, g2_inf=g2_inf)


@pytest.mark.parametrize("glue, r", [(2, 1), (4, 1), (4, 2), (4, 3)])
def test_verify_partial_glue_seams(eng, seams, signed, glue, r):
    """verify_partial_core just past the batch sizes where it starts gluing 2 and 4 signatures per thread, with 1, 2
    and 3 leftover signatures after the glued ones (k_glued<glue, 0> over the first n - r, launch_miller over the rest
    at offset n - r): the partial bit-identical to a reference built through other entry points, and verify_batch's
    verdict on keys, messages and infinity flags changed among the glued and among the leftover signatures."""
    S = signed
    n = seams.verify[glue, r]
    done = n - r
    eng.verify_batch_partial(S.pks[:3], _packed(S.msgs[:3]), S.sigs[:3])  # the generator's table: first call only
    # n = done + r against done + glue (no leftover, same glue, and the same hashing, summing and reduction launches):
    # the difference is the leftover launch_miller
    counts = []
    for m in (done + glue, n):
        before = eng.launch_count
        eng.verify_batch_partial(S.pks[:m], _packed(S.msgs[:m]), S.sigs[:m])
        counts.append(eng.launch_count - before)
    leftover = _launches(seams.lib, MILLER, r, AUTO, seams.sms)
    print("n = %d: k_glued<%d, 0> over %d items + leftover launch_miller %s" % (n, glue, done // glue, leftover))
    assert counts[1] - counts[0] == len(leftover), counts
    P, M, G = S.pks[:n], S.msgs[:n], S.sigs[:n]
    # the partial, with flags on glued and leftover items (a key alone, a signature alone, both)
    pks_inf, sigs_inf = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    pks_inf[[1, n - 1]] = 1
    sigs_inf[[2, n - 1]] = 1
    for seed, first_index in ((None, 0), (SEED, 1234567)):
        part = eng.verify_batch_partial(P, _packed(M), G, pks_inf=pks_inf, sigs_inf=sigs_inf, weight_seed=seed,
                                        first_index=first_index)
        ref = _partial_reference(eng, S, n, pks_inf, sigs_inf, seed, first_index)
        assert (part == ref).all(), ("weighted" if seed else "unweighted", n)
    # verdicts
    assert eng.verify_batch(P, _packed(M), G) is True
    assert eng.verify_batch(P, _packed(M), G, weight_seed=SEED) is True
    # another signer's key or message at the first and last glued and leftover items
    for i in (0, n - 1):
        P2 = P.copy()
        P2[i] = P[i - 1]
        assert eng.verify_batch(P2, _packed(M), G) is False, ("key", i)
    for i in (done - 1, done):
        M2 = M.copy()
        M2[i] = M[i - 1]
        assert eng.verify_batch(P, _packed(M2), G) is False, ("message", i)
    both = np.zeros(n, np.uint8)
    both[done] = 1
    assert eng.verify_batch(P, _packed(M), G, pks_inf=both, sigs_inf=both) is True
    assert eng.verify_batch(P, _packed(M), G, pks_inf=both) is False
    assert eng.verify_batch(P, _packed(M), G, pks_inf=both, sigs_inf=both, weight_seed=SEED) is True
    assert eng.verify_batch(P, _packed(M), G, pks_inf=both, weight_seed=SEED) is False


def test_verify_each_check_seam(eng, seams, signed):
    """verify_each at one two-lane wave of signatures (two-lane check products) and one more (fused
    k_check_products): bad signatures at the first and last item and the block edges, the four infinity flag
    combinations (only both infinite, or neither, verifies)."""
    S = signed
    L = seams.L
    eng.verify_each(S.pks[:3], _packed(S.msgs[:3]), S.sigs[:3])  # the generator's table: first call only
    counts = {}
    for n in (L, L + 1):
        rng = random.Random(n)
        seg = _check(seams.lib, n, AUTO, seams.sms)
        bad = sorted(_edges([seg]) | set(rng.sample(range(n), 8)))
        free = [i for i in rng.sample(range(n), 40) if i not in bad and i + 1 not in bad][:3]
        sigs = S.sigs[:n].copy()
        sigs[bad] = S.sigs[[i + 1 for i in bad]]  # another signer's valid signature
        pks_inf, sigs_inf = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
        pks_inf[free[0]] = sigs_inf[free[1]] = 1
        pks_inf[free[2]] = sigs_inf[free[2]] = 1
        expect = np.ones(n, bool)
        expect[bad + free[:2]] = False
        before = eng.launch_count
        ok = eng.verify_each(S.pks[:n], _packed(S.msgs[:n]), sigs, pks_inf=pks_inf, sigs_inf=sigs_inf)
        counts[n] = eng.launch_count - before, 2 if seg[4] else 1
        print("n = %d: %s check products" % (n, "two-lane" if seg[4] else "fused"))
        assert (ok == expect).all(), (n, np.flatnonzero(ok != expect)[:16].tolist())
    # the same hashing and glued Miller launches at both sizes: the difference is the check products' form
    assert counts[L][1] == 2 and counts[L + 1][1] == 1
    assert counts[L + 1][0] - counts[L][0] == counts[L + 1][1] - counts[L][1], counts


# ------------------------------------------------------------------------------------------ (e) fixed G2 tables
@pytest.mark.parametrize("k_var", [0, 1])
@pytest.mark.parametrize("off", [0, 1])
def test_pairing_check_fixed_seam(eng, seams, pool, k_var, off):
    """pairing_check_fixed_batch with shapes (0, 1) and (1, 1) at L and L + 1 checks: one glued loop per check against
    the fixed table, then two-lane or fused check products."""
    n_checks = seams.L + off
    k, fixed = k_var + 1, 5
    seg = _check(seams.lib, n_checks, AUTO, seams.sms)
    rng = random.Random(3000 + 10 * k_var + off)
    bad, breaks, cancels = _plant(rng, k, n_checks, (), _edges([seg]))
    g1, g1_inf, g2, g2_inf, expect = _checks(eng, pool, k, n_checks, bad, breaks, cancels, fixed=fixed,
                                             g2_flags=k_var > 0, seed=4000 + k_var + off)
    table = eng.g2_precompute(pool[2][fixed:fixed + 1])
    var = (np.arange(k * n_checks) % k) < k_var
    before = eng.launch_count
    ok = eng.pairing_check_fixed_batch(g1, g2[var] if k_var else None, table, k_var, 1, g1_inf=g1_inf,
                                       g2_var_inf=g2_inf[var] if k_var else None)
    # the table's conversion to Montgomery form, the glued loop, the check products
    assert eng.launch_count - before == 2 + (2 if seg[4] else 1), seg
    assert (ok == expect).all(), (k_var, n_checks, np.flatnonzero(ok != expect)[:16].tolist())
    m = 32 * k
    assert eng.pairing_check_batch(g1[:m], g2[:m], k, g1_inf[:m], g2_inf[:m]).tolist() == expect[:32].tolist()
    _oracle_agrees(g1, g1_inf, g2, g2_inf, k, expect, _sample(rng, expect, bad, breaks, cancels, k))


# ------------------------------------------------------------------------------------------ (f) no pairs per check
@pytest.mark.parametrize("size", ["1", "5", "L+1"])
def test_pairing_check_zero_pairs_per_check(seams, size):
    """pairs_per_check = 0 through the C ABI (the wrappers reject it): every check is the empty product, the identity,
    so every verdict is 1, on a fresh context (no scratch buffers yet) and with no kernel launched."""
    import torch

    import sylow_b200

    n = seams.L + 1 if size == "L+1" else int(size)
    for form in ("host", "dev", "multi"):
        e = sylow_b200.Engine([0, 0] if form == "multi" else 0)
        try:
            before = e.launch_count
            if form == "dev":
                d_ok = torch.zeros(n, dtype=torch.uint8, device="cuda:0")
                e._call("sylow_b200_pairing_check_batch_dev", None, None, None, None, 0, n, d_ok, e._stream())
                ok = d_ok.cpu().numpy()
            else:
                # non-null points on the two-slot context, so that the checks are sliced over both slots
                pts = np.zeros((1, 128), np.uint8) if form == "multi" else None
                ok = np.zeros(n, np.uint8)
                e._call("sylow_b200_pairing_check_batch", pts, None, pts, None, 0, n, ok)
            assert e.launch_count == before, form
            assert (ok == 1).all(), (form, n)
        finally:
            e.close()

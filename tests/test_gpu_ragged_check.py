"""GPU tier (-m gpu): pairing checks with a pair count per check (sylow_b200_pairing_check_ragged_batch{,_dev}) and the
EIP-197 body over inputs of any length.  Inputs are built as in test_gpu_verdict_seams.py: multiples of the generators
with scalars chosen so that each check's product is known, failures, breaking and cancelling infinite pairs planted at
chosen pairs.  Here checks have their own lengths (offsets), failures also sit at the class and block edges of the
gathered order that the host build of the plan (tests/hostsim/ragged_plan.cu) gives, and pairs of adjacent checks are
built so that each check fails while their union cancels, which only a boundary that holds rejects.  Every case
asserts the plan's launch count through the context's counter."""
import random

import numpy as np
import pytest

from oracle import bn254_py as o
from tests import wire as w
from tests.test_gpu_verdict_seams import POOL, R, _checks, _plant, _scal, eng, pool, seams  # noqa: F401
from tests.test_launch_plan import AUTO, FEXP, MILLER, _launches
from tests.test_ragged_plan import build, load_ragged_plan

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def rp(tmp_path_factory):
    return load_ragged_plan(tmp_path_factory.mktemp("ragged_plan"))


def _offsets(ks, o0=0):
    return (o0 + np.concatenate([[0], np.cumsum(ks)])).astype(np.uint64)


def _ragged(eng, pool, ks, bad=(), breaks=(), cancels=(), straddles=(), seed=0, o0=0):
    """checks of ks[c] pairs (a_p G1, b_p G2) from pair o0 on (o0 leading pairs that no check holds), every check's
    sum_j a_p b_p = 0 mod r, except: bad pairs (a_p one more: the check fails); breaks: checks whose pair 0 is flagged
    infinite (fails); cancels: checks whose pair 0 is flagged infinite and left out of the sum (holds); straddles: c
    such that check c's last pair and check c + 1's first share their G2 point and their scalars move by +1 and -1, so
    that both checks fail while their union cancels.  Returns (g1, g1_inf, g2, g2_inf, offsets, expected verdicts)."""
    rng = random.Random(seed)
    b, binv, q = pool
    offs = _offsets(ks, o0).astype(np.int64)
    n = int(offs[-1])
    idx = np.array([rng.randrange(POOL) for _ in range(n)])
    for c in straddles:
        idx[offs[c + 1]] = idx[offs[c + 1] - 1]
    a = [rng.getrandbits(253) | 1 for _ in range(n)]
    g1_flag, g2_flag = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    for i, c in enumerate(sorted(set(breaks) | set(cancels))):
        assert ks[c] >= (2 if c in breaks else 1)
        (g2_flag if i % 2 else g1_flag)[offs[c]] = 1
    for c, k in enumerate(ks):
        p0 = int(offs[c])
        if k == 0 or (k == 1 and c in cancels):
            continue
        s = sum(a[p0 + j] * b[idx[p0 + j]] for j in range(k - 1) if not (j == 0 and c in cancels))
        a[p0 + k - 1] = -s * binv[idx[p0 + k - 1]] % R
    check_of = lambda p: int(np.searchsorted(offs[1:], p, side="right"))
    expect = np.ones(len(ks), bool)
    for c in straddles:
        assert ks[c] >= 1 and ks[c + 1] >= 1
        a[offs[c + 1] - 1] += 1
        a[offs[c + 1]] -= 1
        expect[[c, c + 1]] = False
    for p in bad:
        a[p] += 1
        expect[check_of(p)] = False
    expect[list(breaks)] = False
    assert not ({check_of(p) for p in bad} & (set(cancels) | set(straddles)))
    g1, g1_inf = eng.g1_mul_generator_batch(_scal(a))
    return g1, g1_inf | g1_flag, q[idx], g2_flag, offs.astype(np.uint64), expect


def _oracle_agrees(g1, g1_inf, g2, g2_inf, offs, expect, checks):
    """glued_pairing of each sampled check's finite pairs == 1 against expect (test_gpu_verdict_seams' check, on offsets)"""
    for c in checks:
        pairs = [(w.b_g1(bytes(g1[p])), w.b_g2(bytes(g2[p]))) for p in range(int(offs[c]), int(offs[c + 1]))
                 if not (g1_inf[p] or g2_inf[p])]
        got = o.glued_pairing([x for x, _ in pairs], [y for _, y in pairs]) == o.FP12_ONE
        assert got == bool(expect[c]), c


def _launch_count(rp, s, offs, glue=0):
    """the kernels pairing_check_ragged_batch launches for these offsets: the gather, the glued loops of the 4- and
    2-pair items, launch_miller over the single ones, one product launch per level, launch_final_exp, k_gt_is_one"""
    p = build(rp, offs, glue, s.sms)
    if not p["n_pairs"]:
        return 0, p
    n4, n2, n1 = p["items"]
    miller = len(_launches(s.lib, MILLER, n1, AUTO, s.sms)) if n1 else 0
    return 1 + (n4 > 0) + (n2 > 0) + miller + len(p["levels"]) + len(_launches(s.lib, FEXP, offs.size - 1, AUTO,
                                                                                 s.sms)) + 1, p


def _run(eng, rp, s, g1, g1_inf, g2, g2_inf, offs, glue=0):
    """the verdicts of the _dev form (asserting its launch count) and of the host form, which must agree"""
    import torch

    dev = torch.device("cuda", 0)
    d = [torch.from_numpy(x).to(dev) for x in (g1, g2, g1_inf, g2_inf)]
    d_ok = torch.zeros(offs.size - 1, dtype=torch.uint8, device=dev)
    launches, plan = _launch_count(rp, s, offs, glue)
    before = eng.launch_count
    eng.pairing_check_ragged_batch_dev(d[0], d[1], offs, d_ok, d_g1_inf=d[2], d_g2_inf=d[3])
    assert eng.launch_count - before == launches, (plan["glue"], plan["items"], len(plan["levels"]))
    got = d_ok.cpu().numpy().astype(bool)
    host = eng.pairing_check_ragged_batch(g1, g2, offs, g1_inf, g2_inf)
    assert host.tolist() == got.tolist()
    return got, plan


def _gathered_edges(plan, offs):
    """source pairs at the class edges of the gathered order and at the block edges of the glued and Miller launches"""
    n4, n2, n1 = plan["items"]
    g = plan["gather"]
    pos = {0, 4 * n4 - 1, 4 * n4, 4 * n4 + 2 * n2 - 1, 4 * n4 + 2 * n2, plan["n_pairs"] - 1}
    pos |= {4 * 127, 4 * 128, 4 * n4 + 2 * 127, 4 * n4 + 2 * 128, 4 * n4 + 2 * n2 + 127, 4 * n4 + 2 * n2 + 128}
    return {int(g[p]) + int(offs[0]) for p in pos if 0 <= p < plan["n_pairs"]}


# ------------------------------------------------------------------------------------------ uniform offsets
@pytest.mark.parametrize("k, base, off", [
    (1, "L", 0), (1, "L", 1), (2, "W", -1), (2, "W", 0), (3, "L", 0), (3, "L", 1),
    (4, "L", -1), (4, "L", 0), (5, "L", 0), (8, "L", 1),
])
def test_uniform_offsets_equal_pairing_check_batch(eng, seams, pool, rp, k, base, off):
    """k pairs in every check, on both sides of the two-lane seam L and the glued seam W: the ragged verdicts equal
    pairing_check_batch_dev's on the same inputs, and the construction."""
    import torch

    n_checks = getattr(seams, base) + off
    rng = random.Random(5000 + 10 * k + off)
    bad, breaks, cancels = _plant(rng, k, n_checks, (), {0, n_checks - 1, n_checks // 2})
    g1, g1_inf, g2, g2_inf, expect = _checks(eng, pool, k, n_checks, bad, breaks, cancels, seed=6000 + k + off)
    offs = _offsets([k] * n_checks)
    got, plan = _run(eng, rp, seams, g1, g1_inf, g2, g2_inf, offs)
    print("k = %d, %d checks: G = %d, items %s" % (k, n_checks, plan["glue"], plan["items"]))
    dev = torch.device("cuda", 0)
    d = [torch.from_numpy(x).to(dev) for x in (g1, g2, g1_inf, g2_inf)]
    d_ok = torch.zeros(n_checks, dtype=torch.uint8, device=dev)
    eng.pairing_check_batch_dev(d[0], d[1], k, d_ok, d_g1_inf=d[2], d_g2_inf=d[3])
    uniform = d_ok.cpu().numpy().astype(bool)
    assert (got == uniform).all() and (got == expect).all(), np.flatnonzero(got != expect)[:16].tolist()


# ------------------------------------------------------------------------------------------ mixes
@pytest.mark.parametrize("n_checks, glue", [(40, 0), (700, 0), (12000, 0), (12000, 1), (12000, 2)])
def test_mixes(eng, seams, pool, rp, monkeypatch, n_checks, glue):
    """k from 0 to 12 per check: failures at the first and last pair of checks and at the class and block edges of the
    gathered order, breaking and cancelling infinite pairs, adjacent checks that fail alone but cancel together; a
    sample against the oracle.  glue > 0: G fixed by SYLOW_B200_RAGGED_GLUE, with the same verdicts."""
    if glue:
        monkeypatch.setenv("SYLOW_B200_RAGGED_GLUE", str(glue))
    rng = random.Random(7000 + n_checks + glue)
    ks = [rng.choice([0, 1, 2, 2, 3, 4, 4, 5, 6, 7, 8, 9, 12]) for _ in range(n_checks)]
    offs = _offsets(ks, 3)
    plan = build(rp, offs, glue, seams.sms)
    busy = [c for c in range(n_checks) if ks[c] >= 2]
    used = set()
    straddles = [c for c in busy if c + 1 < n_checks and ks[c + 1] >= 1][:: max(1, len(busy) // 12)][:12]
    used |= set(straddles) | {c + 1 for c in straddles}
    free = [c for c in busy if c not in used]
    rng.shuffle(free)
    breaks, cancels = free[:6], free[6:12]
    used |= set(breaks) | set(cancels)
    edge = {p for p in _gathered_edges(plan, offs)}
    ends = {int(offs[c]) for c in free[12:20]} | {int(offs[c + 1]) - 1 for c in free[20:28]}
    check_of = lambda p: int(np.searchsorted(offs[1:].astype(np.int64), p, side="right"))
    bad = {p for p in edge | ends if check_of(p) not in used}
    g1, g1_inf, g2, g2_inf, offs, expect = _ragged(eng, pool, ks, bad, breaks, cancels, straddles, seed=n_checks, o0=3)
    got, plan = _run(eng, rp, seams, g1, g1_inf, g2, g2_inf, offs, glue)
    print("%d checks, G = %d, items %s, %d levels" % (n_checks, plan["glue"], plan["items"], len(plan["levels"])))
    assert (got == expect).all(), np.flatnonzero(got != expect)[:16].tolist()
    assert not got[straddles].any() and not got[[c + 1 for c in straddles]].any()
    if n_checks <= 700 and not glue:
        sample = straddles[:1] + [straddles[0] + 1] + breaks[:1] + cancels[:1]
        sample += [c for c in range(n_checks) if expect[c] and 1 <= ks[c] <= 4][:2]
        _oracle_agrees(g1, g1_inf, g2, g2_inf, offs, expect, sample)


# ------------------------------------------------------------------------------------------ long checks
@pytest.mark.parametrize("items", ["S", "S+1", "S*S+1"])
def test_long_checks_at_chunk_seams(eng, seams, pool, rp, monkeypatch, items):
    """checks of S, S + 1 and S^2 + 1 single-pair items (G fixed at 1), valid and invalid, among short ones"""
    monkeypatch.setenv("SYLOW_B200_RAGGED_GLUE", "1")
    S = int(rp.rp_chunk())
    m = eval(items, {"S": S})
    ks = [3, m, 2, m, 0, 1]
    offs = _offsets(ks)
    bad = {int(offs[3]) + m - 1}  # the last pair of the second long check
    g1, g1_inf, g2, g2_inf, offs, expect = _ragged(eng, pool, ks, bad, seed=m)
    got, plan = _run(eng, rp, seams, g1, g1_inf, g2, g2_inf, offs, 1)
    assert len(plan["levels"]) == {"S": 1, "S+1": 2, "S*S+1": 3}[items]
    assert got.tolist() == expect.tolist() == [True, True, True, False, True, True]


def test_checks_of_more_than_2_16_pairs(eng, seams, pool, rp):
    """one valid and one invalid check of 70 001 pairs each between short checks"""
    m = 70001
    ks = [2, m, 4, m, 1]
    offs = _offsets(ks)
    bad = {int(offs[3]) + m // 2}
    g1, g1_inf, g2, g2_inf, offs, expect = _ragged(eng, pool, ks, bad, breaks=[2], seed=11)
    got, plan = _run(eng, rp, seams, g1, g1_inf, g2, g2_inf, offs)
    print("G = %d, items %s, %d levels" % (plan["glue"], plan["items"], len(plan["levels"])))
    assert got.tolist() == expect.tolist() == [True, True, False, False, True]


def test_dev_on_a_torch_stream(eng, seams, pool, rp):
    import torch

    ks = [0, 3, 5, 2, 8, 1, 4, 12, 0, 6] * 20
    g1, g1_inf, g2, g2_inf, offs, expect = _ragged(eng, pool, ks, {5, 101, 400}, breaks=[4], cancels=[7], seed=13)
    dev = torch.device("cuda", 0)
    st = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(st):
        d = [torch.from_numpy(x).to(dev) for x in (g1, g2, g1_inf, g2_inf)]
        d_ok = torch.zeros(len(ks), dtype=torch.uint8, device=dev)
        eng.pairing_check_ragged_batch_dev(d[0], d[1], offs, d_ok, d_g1_inf=d[2], d_g2_inf=d[3])
        got = d_ok.cpu().numpy().astype(bool)
    st.synchronize()
    assert got.tolist() == expect.tolist()


def test_two_slot_context_cuts_inside_long_checks(eng, pool):
    """Engine([0, 0]) cuts the batch inside a run of long checks; its verdicts equal one slot's and the construction"""
    import sylow_b200

    ks = [1] * 5 + [5000] * 7 + [3] * 11
    offs = _offsets(ks)
    bad = {int(offs[6]), int(offs[12]) - 1, int(offs[20])}
    g1, g1_inf, g2, g2_inf, offs, expect = _ragged(eng, pool, ks, bad, breaks=[7], cancels=[10], straddles=[8],
                                                   seed=17)
    one = eng.pairing_check_ragged_batch(g1, g2, offs, g1_inf, g2_inf)
    e2 = sylow_b200.Engine([0, 0])
    try:
        two = e2.pairing_check_ragged_batch(g1, g2, offs, g1_inf, g2_inf)
        c2, s2 = e2.eip197_pairing_check_ragged_batch(_eip_inputs(eng, g1, g1_inf, g2, g2_inf, offs))
    finally:
        e2.close()
    assert one.tolist() == two.tolist() == expect.tolist() == c2.tolist()
    assert not s2.any()


# ------------------------------------------------------------------------------------------ EIP-197
def _eip_inputs(eng, g1, g1_inf, g2, g2_inf, offs):
    """each check's pairs as EIP-197 calldata (infinity all-zero)"""
    b1 = eng.g1_to_be_bytes_batch(g1, g1_inf, scrubbed=True)
    b2 = eng.g2_to_be_bytes_batch(g2, g2_inf, scrubbed=True)
    rows = np.concatenate([b1, b2], axis=1)
    return [rows[int(offs[c]):int(offs[c + 1])].tobytes() for c in range(offs.size - 1)]


def test_eip197_ragged_equals_uniform_per_length(eng, pool):
    rng = random.Random(19)
    ks = [rng.choice([1, 2, 3, 4]) for _ in range(400)]
    bad = set(rng.sample(range(int(sum(ks))), 25))
    g1, g1_inf, g2, g2_inf, offs, expect = _ragged(eng, pool, ks, bad, seed=19)
    inputs = _eip_inputs(eng, g1, g1_inf, g2, g2_inf, offs)
    ok, st = eng.eip197_pairing_check_ragged_batch(inputs)
    assert ok.tolist() == expect.tolist() and not st.any()
    for k in (1, 2, 3, 4):
        sel = [c for c in range(len(ks)) if ks[c] == k]
        uok, ust = eng.eip197_pairing_check_batch(np.frombuffer(b"".join(inputs[c] for c in sel), np.uint8)
                                                  .reshape(len(sel), 192 * k), k)
        assert uok.tolist() == ok[sel].tolist() and ust.tolist() == st[sel].tolist(), k


def test_eip197_ragged_vectors_and_malformed(eng, kats):
    """the reference's pinned ecPairing vector, empty inputs, malformed lengths between valid inputs, and decode,
    curve and subgroup failures at the first and last pair of an input"""
    from tests.test_gpu_parity import _g2_be
    from tests.test_hostsim import _twist_points_outside_subgroup

    good = bytes.fromhex(kats["eip197_pair"]["input"])
    assert bytes.fromhex(kats["eip197_pair"]["expected"])[-1] == 1
    rng = random.Random(23)
    q = _twist_points_outside_subgroup(rng, 1)[0]
    four = good + good  # 4 pairs: two cancelling halves

    def at(base, pair, lo, hi, value):
        b = bytearray(base)
        b[192 * pair + lo:192 * pair + hi] = value
        return bytes(b)

    over = (o.P + 5).to_bytes(32, "big")
    cases = [
        (good, True, 0), (b"", True, 0), (b"\x00", False, -1), (good, True, 0), (bytes(191), False, -1),
        (four, True, 0), (bytes(193), False, -1), (bytes(384), True, 0),
        (at(four, 0, 0, 32, over), False, -6), (at(four, 3, 0, 32, over), False, -6),   # decode: x >= p
        (at(four, 0, 63, 64, bytes([four[63] ^ 1])), False, -3),                        # G1 off the curve
        (at(four, 3, 63, 64, bytes([four[192 * 3 + 63] ^ 1])), False, -3),
        (at(four, 0, 64, 192, _g2_be(q)), False, -4), (at(four, 3, 64, 192, _g2_be(q)), False, -4),  # subgroup
        (at(four, 3, 0, 32, over)[:-1], False, -1), (good, True, 0),
    ]
    # the first failing pair wins (G1 before G2 within a pair): pair 0's G2 over pair 1's G1
    both = at(at(four, 0, 64, 192, _g2_be(q)), 1, 0, 32, over)
    cases.append((both, False, -4))
    ok, st = eng.eip197_pairing_check_ragged_batch([c[0] for c in cases])
    assert ok.tolist() == [c[1] for c in cases]
    assert st.tolist() == [c[2] for c in cases]


# ------------------------------------------------------------------------------------------ empty batches
@pytest.mark.parametrize("n", [1, 5, 300])
def test_all_empty_batches_launch_nothing(n):
    import torch

    import sylow_b200

    offs = np.full(n + 1, 9, np.uint64)
    for form in ("host", "dev", "multi", "eip197", "eip197 multi"):
        e = sylow_b200.Engine([0, 0] if "multi" in form else 0)
        try:
            before = e.launch_count
            if form == "dev":
                d_ok = torch.zeros(n, dtype=torch.uint8, device="cuda:0")
                e._call("sylow_b200_pairing_check_ragged_batch_dev", None, None, None, None, offs, n, d_ok,
                        e._stream())
                ok = d_ok.cpu().numpy()
            elif form.startswith("eip197"):
                ok, st = e.eip197_pairing_check_ragged_batch([b""] * n)
                assert not st.any()
            else:
                ok = np.zeros(n, np.uint8)
                e._call("sylow_b200_pairing_check_ragged_batch", None, None, None, None, offs, n, ok)
            assert e.launch_count == before, form
            assert (np.asarray(ok) == 1).all(), form
        finally:
            e.close()

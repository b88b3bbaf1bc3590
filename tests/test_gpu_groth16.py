"""GPU tier (-m gpu): Groth16 verification (sylow_b200_groth16_*) against trapdoor-made keys and proofs
(tests/groth16_ref.py).  verify_each is compared with pairing_check_fixed_batch(.., 1, 3) on records [A, -alpha, -L, -C]
assembled here, and on a sample with the oracle's verifier; verify_batch with the AND of verify_each.  Large batches come
from the library's generator multiplications (tested against the oracle in test_gpu_generator_mul.py); the scalars are
known, so every expected verdict is too."""
import ctypes
import random

import numpy as np
import pytest

from oracle import bn254_py as o
from tests import groth16_ref as g
from tests import wire as w
from tests.test_launch_plan import AUTO, _check, load_launch_plan

pytestmark = pytest.mark.gpu
R = o.R_ORDER
SEED = bytes(range(40, 72))
# launch-shape switches on a B200 (148 SMs; asserted against launch_plan.h in test_switch_sizes)
LANES_WAVE = 18944      # launch_check_products: checks on two lanes up to one two-lane wave, fused k_check_products above
AFF_MIN_BATCH = 32768   # point_batch: batched affine conversion of -L from SY_AFF_MIN_BATCH proofs on
GLUE2, GLUE4 = 37889, 113665  # fused_product_values: 2 / 4 pairs per thread from these batch sizes on


@pytest.fixture(scope="module")
def eng():
    import sylow_b200

    e = sylow_b200.Engine(0)
    yield e
    e.close()


def _le(xs):
    return np.frombuffer(b"".join(int(x).to_bytes(32, "little") for x in xs), np.uint8).reshape(-1, 32).copy()


class Batch:
    """n proofs of random inputs under one trapdoor key; tamper with .proofs / .x / .inf, then read the verdicts"""

    def __init__(self, eng, l, n, seed):
        self.eng, self.l, self.n = eng, l, n
        self.td = g.Trapdoor(l, seed)
        self.vk_pts = self.td.vk()
        self.vk = np.frombuffer(g.vk_bytes(self.vk_pts), np.uint8).copy()
        rng = random.Random(seed + 1)
        self.xs = [[rng.randrange(R) for _ in range(l)] for _ in range(n)]
        inv = pow(self.td.de, -1, R)
        self.a, self.b, self.c = [], [], []
        for xs in self.xs:
            a, b = rng.randrange(1, R), rng.randrange(1, R)
            self.a.append(a)
            self.b.append(b)
            self.c.append((a * b - self.td.al * self.td.be - self.td.l_scalar(xs) * self.td.ga) * inv % R)
        self.build()
        self.inf = np.zeros((n, 3), np.uint8)

    def build(self):
        A = self.eng.g1_mul_generator_batch(_le(self.a))[0]
        B = self.eng.g2_mul_generator_batch(_le(self.b))[0]
        C = self.eng.g1_mul_generator_batch(_le(self.c))[0]
        self.proofs = np.concatenate([A, B, C], axis=1)
        self.set_x(self.xs)

    def set_x(self, xs):
        self.xs = xs
        self.x = _le([v for row in xs for v in row]).reshape(self.n, 32 * self.l) if self.l else None

    def each(self, eng=None):
        return (eng or self.eng).groth16_verify_each(self.vk, self.proofs, self.x, self.l, proofs_inf=self.inf)

    def batch(self, eng=None, seed=SEED):
        return (eng or self.eng).groth16_verify_batch(self.vk, self.proofs, self.x, self.l, seed, proofs_inf=self.inf)

    def fixed_check(self):
        """pairing_check_fixed_batch(.., 1, 3) on [A, -alpha, -L, -C] assembled on the host, and the input ranges"""
        n = self.n
        neg_l = self.eng.g1_mul_generator_batch(_le([-self.td.l_scalar(xs) % R for xs in self.xs]))[0]
        neg_a = np.frombuffer(w.g1_b(o.g1_affine_neg(self.vk_pts[0])), np.uint8)
        cy = [int.from_bytes(bytes(r[224:256]), "little") for r in self.proofs]
        neg_c = self.proofs[:, 192:256].copy()
        neg_c[:, 32:] = _le([(-y) % o.P if not f else y for y, f in zip(cy, self.inf[:, 2])])
        g1 = np.concatenate([self.proofs[:, :64], np.tile(neg_a, (n, 1)), neg_l, neg_c], axis=1).reshape(4 * n, 64)
        g1_inf = np.zeros((n, 4), np.uint8)
        g1_inf[:, 0] = self.inf[:, 0] | self.inf[:, 1]  # a flagged B drops the pair through its G1 side here
        g1_inf[:, 3] = self.inf[:, 2]
        co = self.eng.g2_precompute(np.frombuffer(self.vk.tobytes()[64:448], np.uint8).reshape(3, 128))
        ok = self.eng.pairing_check_fixed_batch(g1, self.proofs[:, 64:192], co, 1, 3, g1_inf=g1_inf.reshape(-1))
        in_range = np.array([all(v < R for v in xs) for xs in self.xs], bool)
        return ok & in_range

    def proof_pts(self, j):
        p = bytes(self.proofs[j])
        return (w.b_g1(p[:64], self.inf[j, 0]), w.b_g2(p[64:192], self.inf[j, 1]), w.b_g1(p[192:], self.inf[j, 2]))


def _tamper(bt, j, kind):
    """one tampered case at proof j; the proofs it invalidates (swapped inputs invalidate both proofs)"""
    k = (j + 1) % bt.n
    if kind == "c_plus_1":
        bt.c[j] = (bt.c[j] + 1) % R
    elif kind == "swap_inputs":
        xs = [list(r) for r in bt.xs]
        xs[j], xs[k] = xs[k], xs[j]
        bt.xs = xs
        return {j, k}
    elif kind == "x_plus_r":
        xs = [list(r) for r in bt.xs]
        xs[j][0] += R
        bt.xs = xs
    elif kind == "b_of_other":
        bt.b[j] = bt.b[k]
    elif kind == "a_inf":
        pass
    else:
        raise ValueError(kind)
    return {j}


KINDS = ["c_plus_1", "swap_inputs", "x_plus_r", "b_of_other", "a_inf"]


def _apply(bt, plan):
    """plan: {proof: kind}; rebuilds the points and flags and returns the proofs that no longer verify"""
    bad = set()
    for j, kind in sorted(plan.items()):
        if kind in ("swap_inputs", "x_plus_r") and bt.l == 0:
            kind = "c_plus_1"
        bad |= _tamper(bt, j, kind)
    bt.build()
    for j, kind in plan.items():
        if kind == "a_inf":
            bt.inf[j, 0] = 1
    return bad


def test_switch_sizes(tmp_path_factory):
    """The sizes named above are the switches of launch_plan.h / sylow_b200.cu on this GPU."""
    import torch

    lib = load_launch_plan(tmp_path_factory.mktemp("launch_plan"))
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if sms != 148:
        pytest.skip("the named sizes are those of a 148-SM B200")
    assert _check(lib, LANES_WAVE, AUTO, sms)[4] and not _check(lib, LANES_WAVE + 1, AUTO, sms)[4]
    assert lib.lp_glue(sms, GLUE2 - 1, 8444) == 1 and lib.lp_glue(sms, GLUE2, 8444) == 2
    assert lib.lp_glue(sms, GLUE4 - 1, 8444) != 4 and lib.lp_glue(sms, GLUE4, 8444) == 4


@pytest.mark.parametrize("l", [0, 1, 3, 16])
def test_verify_each_tampered(eng, l):
    bt = Batch(eng, l, 40, seed=100 + l)
    bad = _apply(bt, {2 + 3 * i: k for i, k in enumerate(KINDS)})
    got = bt.each()
    assert got.tolist() == bt.fixed_check().tolist()
    assert set(np.flatnonzero(~got).tolist()) == bad


def test_verify_each_against_the_oracle(eng):
    bt = Batch(eng, 3, 6, seed=7)
    _apply(bt, {1: "c_plus_1", 2: "x_plus_r", 4: "a_inf"})
    got = bt.each()
    for j in (0, 1, 2, 4):
        assert got[j] == g.groth16_verify(bt.vk_pts, bt.proof_pts(j), bt.xs[j]), j
    assert got.tolist() == [True, False, False, True, False, True]


@pytest.mark.parametrize("n", [LANES_WAVE, LANES_WAVE + 1, AFF_MIN_BATCH - 1, AFF_MIN_BATCH],
                         ids=["two_lane_checks", "fused_checks", "per_thread_affine", "batched_affine"])
def test_verify_each_switch_sizes(eng, n):
    bt = Batch(eng, 1, n, seed=n)
    bad = _apply(bt, {0: "c_plus_1", n // 2: "x_plus_r", n - 1: "b_of_other", 255: "a_inf", 256: "swap_inputs"})
    got = bt.each()
    assert got.tolist() == bt.fixed_check().tolist()
    assert set(np.flatnonzero(~got).tolist()) == bad


@pytest.mark.parametrize("n", [GLUE2 - 1, GLUE2, GLUE4 - 1, GLUE4],
                         ids=["glue1", "glue2", "glue2_below_glue4", "glue4"])
def test_verify_batch_switch_sizes(eng, n):
    bt = Batch(eng, 1, n, seed=n)
    assert bt.batch() is True
    for j in (0, n // 2, n - 1):
        b2 = Batch.__new__(Batch)
        b2.__dict__.update(bt.__dict__)
        b2.c = list(bt.c)
        b2.inf = bt.inf.copy()
        _apply(b2, {j: "c_plus_1"})
        assert b2.batch() is False, j


@pytest.mark.parametrize("l", [0, 1, 3, 16])
def test_verify_batch(eng, l):
    bt = Batch(eng, l, 33, seed=200 + l)
    assert bt.batch() is True
    assert bt.each().all()
    for j in (0, 16, 32):
        for kind in KINDS:
            b2 = Batch(eng, l, 33, seed=200 + l)
            _apply(b2, {j: kind})
            assert b2.batch() is False, (j, kind)


def test_verify_batch_input_out_of_range(eng):
    bt = Batch(eng, 2, 20, seed=5)
    xs = [list(r) for r in bt.xs]
    xs[7][1] += R  # the same residue: the proof itself is right, the input is not canonical
    bt.set_x(xs)
    assert bt.batch() is False
    assert bt.each().tolist() == [j != 7 for j in range(20)]
    xs[7][1] = (1 << 256) - 1
    bt.set_x(xs)
    assert bt.batch() is False


def test_verify_batch_cancelling_errors(eng):
    """C_1 + D and C_2 - D: the unweighted product would hold, the weighted one does not"""
    bt = Batch(eng, 1, 8, seed=9)
    d = random.Random(3).randrange(1, R)
    bt.c[1] = (bt.c[1] + d) % R
    bt.c[2] = (bt.c[2] - d) % R
    bt.build()
    assert bt.each().tolist() == [True, False, False] + [True] * 5
    assert bt.batch() is False


def test_verify_batch_is_and_of_verify_each(eng):
    rng = random.Random(17)
    for trial in range(6):
        bt = Batch(eng, 2, 48, seed=300 + trial)
        plan = {j: rng.choice(KINDS) for j in range(48) if rng.random() < (0.0 if trial == 0 else 0.05)}
        _apply(bt, plan)
        each = bt.each()
        assert each.tolist() == bt.fixed_check().tolist()
        assert bt.batch() == bool(each.all()), plan


def test_verify_batch_empty_and_seed(eng):
    bt = Batch(eng, 1, 4, seed=11)
    assert eng.groth16_verify_batch(bt.vk, np.zeros((0, 256), np.uint8), np.zeros((0, 32), np.uint8), 1, SEED) is True
    ok = ctypes.c_int(0)
    with pytest.raises(Exception) as e:
        eng._call("sylow_b200_groth16_verify_batch", bt.vk, 1, bt.proofs, None, bt.x, 4, None, ctypes.byref(ok))
    assert e.value.status == -1  # SYLOW_B200_ERR_ARG
    assert bt.batch(seed=bytes(32)) is True  # any seed verifies a valid batch


def test_multi_device_context(eng):
    import sylow_b200

    multi = sylow_b200.Engine([0, 0])
    try:
        bt = Batch(eng, 3, 21, seed=21)
        assert bt.batch(multi) is True and bt.batch() is True
        _apply(bt, {20: "c_plus_1", 3: "a_inf"})  # 20: in the last slice
        assert bt.each(multi).tolist() == bt.each().tolist()
        assert bt.batch(multi) is False
        bt2 = Batch(eng, 3, 21, seed=21)
        _apply(bt2, {20: "x_plus_r"})
        assert bt2.batch(multi) is False and bt2.batch() is False
    finally:
        multi.close()


@pytest.mark.parametrize("l", [0, 4])
def test_dev_path_matches_host_path(eng, l):
    import torch
    import sylow_b200

    bt = Batch(eng, l, 50, seed=400 + l)
    _apply(bt, {3: "c_plus_1", 4: "a_inf", 49: "b_of_other"})
    host = bt.each()
    d_vk = torch.empty(sylow_b200.groth16_vk_dev_bytes(l), dtype=torch.uint8, device="cuda")
    eng.groth16_prepare_vk(bt.vk, l, d_vk)
    d_p = torch.from_numpy(bt.proofs).cuda()
    d_x = torch.from_numpy(bt.x).cuda() if l else None
    d_inf = torch.from_numpy(bt.inf.reshape(-1).copy()).cuda()
    d_ok = torch.empty(bt.n, dtype=torch.uint8, device="cuda")
    eng.groth16_verify_each_dev(d_vk, l, d_p, d_x, d_ok, d_proofs_inf=d_inf)
    torch.cuda.synchronize()
    assert d_ok.cpu().numpy().tolist() == host.astype(np.uint8).tolist()
    # the batch verdict from two device partials over global indices, combined by verify_batch_finish
    parts = []
    for lo, hi in ((0, 20), (20, 50)):
        d_f = torch.empty(384, dtype=torch.uint8, device="cuda")
        eng.groth16_verify_batch_partial_dev(d_vk, l, d_p[lo:hi], d_x[lo:hi] if l else None, d_f, SEED, first_index=lo,
                                             d_proofs_inf=d_inf[3 * lo:3 * hi])
        torch.cuda.synchronize()
        parts.append(d_f.cpu().numpy())
    assert eng.verify_batch_finish(np.stack(parts)) is False
    bt_ok = Batch(eng, l, 50, seed=400 + l)
    d_p = torch.from_numpy(bt_ok.proofs).cuda()
    d_x = torch.from_numpy(bt_ok.x).cuda() if l else None
    parts = []
    for lo, hi in ((0, 20), (20, 50)):
        d_f = torch.empty(384, dtype=torch.uint8, device="cuda")
        eng.groth16_verify_batch_partial_dev(d_vk, l, d_p[lo:hi], d_x[lo:hi] if l else None, d_f, SEED, first_index=lo)
        torch.cuda.synchronize()
        parts.append(d_f.cpu().numpy())
    assert eng.verify_batch_finish(np.stack(parts)) is True and bt_ok.batch() is True
    # an input >= r makes the device partial the Fp12 zero
    if l:
        bad_x = bt_ok.x.copy()
        bad_x[5, :32] = np.frombuffer((R + 1).to_bytes(32, "little"), np.uint8)
        d_f = torch.empty(384, dtype=torch.uint8, device="cuda")
        eng.groth16_verify_batch_partial_dev(d_vk, l, d_p, torch.from_numpy(bad_x).cuda(), d_f, SEED)
        torch.cuda.synchronize()
        assert not d_f.cpu().numpy().any()


def test_prepare_vk_rejects_invalid_keys(eng):
    import torch
    import sylow_b200
    from tests.test_hostsim import _twist_points_outside_subgroup

    bt = Batch(eng, 2, 4, seed=31)
    d_vk = torch.empty(sylow_b200.groth16_vk_dev_bytes(2), dtype=torch.uint8, device="cuda")
    eng.groth16_prepare_vk(bt.vk, 2, d_vk)
    bad_alpha = bt.vk.copy()
    bad_alpha[:64] = np.frombuffer(w.g1_b((1, 3, False)), np.uint8)  # 3^2 != 1 + 3
    bad_beta = bt.vk.copy()
    bad_beta[64:192] = np.frombuffer(w.g2_b(_twist_points_outside_subgroup(random.Random(1), 1)[0]), np.uint8)
    bad_ic = bt.vk.copy()
    bad_ic[448 + 64 + 32:448 + 128] = np.frombuffer(w.fp_b(o.P), np.uint8)  # IC_1.y = p: not canonical
    for vk, status in ((bad_alpha, -3), (bad_beta, -4), (bad_ic, -6)):
        with pytest.raises(sylow_b200.SylowB200Error) as e:
            eng.groth16_prepare_vk(vk, 2, d_vk)
        assert e.value.status == status
        with pytest.raises(sylow_b200.SylowB200Error) as e:
            eng.groth16_verify_each(vk, bt.proofs, bt.x, 2)
        assert e.value.status == status

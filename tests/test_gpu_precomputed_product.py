"""GPU tier (-m gpu): Miller loops and glued Miller products over one precomputed G2 table per pair (k_miller_tables,
include/sylow_b200.h: sylow_b200_miller_loop_precomputed_batch, _miller_product_precomputed, _g2_precompute_dev,
_miller_product_precomputed_dev).  Bit-exact against the oracle and against the fused Miller loop on the same points."""
import random

import numpy as np
import pytest

from oracle import bn254_py as o
from tests import wire as w

pytestmark = pytest.mark.gpu

TABLE = 87 * 192


@pytest.fixture(scope="module")
def eng():
    import sylow_b200

    e = sylow_b200.Engine(0)
    yield e
    e.close()


def arr(bs):
    return np.frombuffer(b"".join(bs), dtype=np.uint8).reshape(len(bs), -1).copy()


def _scalars(rng, n):
    s = np.frombuffer(rng.randbytes(32 * n), dtype=np.uint8).reshape(n, 32).copy()
    s[:, 31] &= 0x0F  # below p
    return s


@pytest.fixture(scope="module")
def pairs(eng):
    """1031 random pairs (G1, G2 wire form), the G2 generator at index 3, and their canonical tables."""
    rng = random.Random(970)
    n = 1031
    g1, _ = eng.g1_mul_batch(np.tile(np.frombuffer(w.g1_b(o.G1_GEN), np.uint8), (n, 1)), _scalars(rng, n))
    g2, _ = eng.g2_mul_batch(np.tile(np.frombuffer(w.g2_b(o.G2_GEN), np.uint8), (n, 1)), _scalars(rng, n))
    g2[3] = np.frombuffer(w.g2_b(o.G2_GEN), np.uint8)
    return g1, g2, eng.g2_precompute(g2)


def _one():
    return np.frombuffer(w.fp12_b(o.FP12_ONE), np.uint8)


def test_per_item_batch(eng, pairs):
    """One table per pair, 150 ragged pairs with the generator among them and some infinite G1 points: the reference's
    G2PreComputed::miller_loop on a sample, and byte-equal to the fused miller_loop_batch on every pair."""
    g1, g2, coeffs = pairs
    n = 150
    inf = np.zeros(n, np.uint8)
    inf[[0, 7, 77, 149]] = 1
    got = eng.miller_loop_precomputed_batch(coeffs[:n], g1[:n], inf)
    assert (got == eng.miller_loop_batch(g1[:n], g2[:n], g1_inf=inf)).all()
    for i in (0, 1, 3, 76, 148, 149):
        exp = o.FP12_ONE if inf[i] else o.miller_loop(o.g2_precompute(w.b_g2(bytes(g2[i]))), w.b_g1(bytes(g1[i])))
        assert w.b_fp12(bytes(got[i])) == exp, i


@pytest.mark.parametrize("n", [0, 1, 2, 3, 4, 5, 7, 17, 150, 1031])
def test_host_product(eng, pairs, n):
    """glued_miller_loop(&[G2PreComputed], &[G1Affine]) for every n % 4; infinite G1 pairs are skipped."""
    g1, g2, coeffs = pairs
    inf = np.zeros(n, np.uint8)
    inf[[k for k in (2, 9, 100, 1000) if k < n]] = 1
    got = eng.miller_product_precomputed(coeffs[:n], g1[:n], inf)
    assert (got == eng.miller_product(g1[:n], g2[:n], g1_inf=inf)).all()
    if n <= 17:
        keep = [k for k in range(n) if not inf[k]]
        exp = o.glued_miller_loop([o.g2_precompute(w.b_g2(bytes(g2[k]))) for k in keep],
                                  [w.b_g1(bytes(g1[k])) for k in keep])
        assert w.b_fp12(bytes(got)) == exp
    if n == 0:
        assert (got == _one()).all()


def _device_pairs(eng, rng, n):
    import torch

    dev = torch.device("cuda", 0)
    d_g1 = torch.empty((n, 64), dtype=torch.uint8, device=dev)
    d_g2 = torch.empty((n, 128), dtype=torch.uint8, device=dev)
    gen1 = torch.from_numpy(np.frombuffer(w.g1_b(o.G1_GEN), np.uint8).copy()).to(dev).expand(n, 64).contiguous()
    gen2 = torch.from_numpy(np.frombuffer(w.g2_b(o.G2_GEN), np.uint8).copy()).to(dev).expand(n, 128).contiguous()
    eng.g1_mul_batch_dev(gen1, torch.from_numpy(_scalars(rng, n)).to(dev), d_g1)
    eng.g2_mul_batch_dev(gen2, torch.from_numpy(_scalars(rng, n)).to(dev), d_g2)
    return d_g1, d_g2


def test_resident_tables_both_sides_of_the_glue_switch(eng):
    """Resident tables at 2^13 pairs (one pair per thread) and 2^18 pairs (4.4 GB of tables, four pairs per thread),
    with 50 001 pairs (two per thread) and 2^18 - 1, 2^18 - 2 pairs for the leftover launch: bit-identical to the fused
    miller_product_dev on the same points."""
    import torch

    rng = random.Random(2018)
    for n_all, sizes in ((1 << 13, [1 << 13]), (1 << 18, [50001, (1 << 18) - 2, (1 << 18) - 1, 1 << 18])):
        d_g1, d_g2 = _device_pairs(eng, rng, n_all)
        d_inf = torch.zeros(n_all, dtype=torch.uint8, device="cuda:0")
        d_inf[torch.randint(0, n_all, (64,), generator=torch.Generator().manual_seed(n_all))] = 1
        d_tables = torch.empty(n_all * TABLE, dtype=torch.uint8, device="cuda:0")
        eng.g2_precompute_dev(d_g2, d_tables)
        for n in sizes:
            d_got = torch.empty(384, dtype=torch.uint8, device="cuda:0")
            d_ref = torch.empty(384, dtype=torch.uint8, device="cuda:0")
            eng.miller_product_precomputed_dev(d_tables, d_g1[:n], d_got, d_g1_inf=d_inf[:n])
            eng.miller_product_dev(d_g1[:n], d_g2[:n], d_ref, d_g1_inf=d_inf[:n])
            torch.cuda.synchronize()
            assert torch.equal(d_got, d_ref), n
        del d_tables
        torch.cuda.empty_cache()


def test_device_tables_indices_and_guard(eng, pairs):
    """g2_precompute_dev equals tables_to_device(g2_precompute(..)); an index array (permutation with repeats) gives the
    host product of the gathered tables; an index past the last table makes the product zero, and its final
    exponentiation zero (never the identity); no index with more pairs than tables is an argument error."""
    import torch

    from sylow_b200 import _lib

    g1, g2, coeffs = pairs
    dev = torch.device("cuda", 0)
    k = 37
    d_tab = torch.empty(k * TABLE, dtype=torch.uint8, device=dev)
    eng.g2_precompute_dev(torch.from_numpy(g2[:k].copy()).to(dev), d_tab)
    d_ref = torch.empty(k * TABLE, dtype=torch.uint8, device=dev)
    eng.tables_to_device(coeffs[:k], d_ref)
    torch.cuda.synchronize()
    assert torch.equal(d_tab, d_ref)

    rng = random.Random(37)
    d_out = torch.empty(384, dtype=torch.uint8, device=dev)
    # no index: pair i uses table i
    n = 29
    eng.miller_product_precomputed_dev(d_tab, torch.from_numpy(g1[:n].copy()).to(dev), d_out)
    assert (d_out.cpu().numpy() == eng.miller_product_precomputed(coeffs[:n], g1[:n])).all()
    # a permutation with repeats, over more pairs than tables
    for n in (5, 150):
        idx = np.array([rng.randrange(k) for _ in range(n)], dtype=np.int32)
        idx[: min(n, 4)] = [3, 3, 0, k - 1][: min(n, 4)]
        d_g1 = torch.from_numpy(g1[:n].copy()).to(dev)
        eng.miller_product_precomputed_dev(d_tab, d_g1, d_out, d_table_idx=torch.from_numpy(idx).to(dev))
        assert (d_out.cpu().numpy() == eng.miller_product_precomputed(coeffs[idx], g1[:n])).all(), n
    # the index guard: k, a large index and 0xffffffff (int32 -1) each make the product zero
    zero = np.zeros(384, np.uint8)
    for bad in (k, 1 << 30, -1):
        idx = np.arange(9, dtype=np.int32)
        idx[4] = bad
        eng.miller_product_precomputed_dev(d_tab, torch.from_numpy(g1[:9].copy()).to(dev), d_out,
                                           d_table_idx=torch.from_numpy(idx).to(dev))
        got = d_out.cpu().numpy()
        assert (got == zero).all(), bad
        assert (eng.final_exp_batch(got.reshape(1, 384)) == zero).all()
    # no index and more pairs than tables
    with pytest.raises(_lib.SylowB200Error) as ei:
        eng.miller_product_precomputed_dev(d_tab, torch.from_numpy(g1[: k + 1].copy()).to(dev), d_out)
    assert ei.value.status == _lib.ERR_ARG
    # n = 0 gives 1
    eng.miller_product_precomputed_dev(d_tab, torch.empty((0, 64), dtype=torch.uint8, device=dev), d_out)
    assert (d_out.cpu().numpy() == _one()).all()


def test_multi_device_context_matches_single(eng, pairs):
    """Engine([0, 0, 0]) slices the host entry points over three device slots: bit-identical to Engine(0)."""
    import sylow_b200

    g1, g2, coeffs = pairs
    multi = sylow_b200.Engine([0, 0, 0])
    try:
        for n in (1, 2, 150):
            inf = np.zeros(n, np.uint8)
            inf[n // 2] = 1
            assert (multi.miller_loop_precomputed_batch(coeffs[:n], g1[:n], inf)
                    == eng.miller_loop_precomputed_batch(coeffs[:n], g1[:n], inf)).all(), n
            assert (multi.miller_product_precomputed(coeffs[:n], g1[:n], inf)
                    == eng.miller_product_precomputed(coeffs[:n], g1[:n], inf)).all(), n
    finally:
        multi.close()


def test_sylow_glued_miller_loop_takes_precomputed(eng):
    """sylow.glued_miller_loop accepts G2PreComputed values (the reference's signature) with the same result as the
    G2Affine form, infinite points on either side included."""
    from sylow_b200 import sylow as s

    qs = [s.G2Affine.generator()] + [s.G2Affine.rand() for _ in range(4)] + [s.G2Affine.zero()]
    ps = [s.G1Affine.rand() for _ in range(4)] + [s.G1Affine.zero(), s.G1Affine.generator()]
    pcs = [q.precompute() for q in qs]
    assert s.glued_miller_loop(pcs, ps) == s.glued_miller_loop(qs, ps)
    assert s.glued_miller_loop(pcs[:3], ps) == s.glued_miller_loop(qs[:3], ps)  # zip truncation
    assert s.glued_miller_loop([], ps) == s.glued_miller_loop([], [])
    with pytest.raises(TypeError):
        s.glued_miller_loop([pcs[0], qs[1]], ps[:2])

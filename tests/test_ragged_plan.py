"""CPU tier: the launch plan of the ragged pairing checks (sylow_b200/csrc/ragged_plan.h), compiled for the host
(tests/hostsim/ragged_plan.cu).  Every plan is checked against the invariants the kernels rely on: every pair gathered
exactly once; items of 1, 2 or 4 consecutive pairs of one check, 4-pair items first, then 2-pair, then single ones; the
chunk products of each check covering exactly its items' values, each value read once and only after it is written;
no thread multiplying more than kRaggedChunk values; check c's product in final slot c; G equal to glue_pairs.  The
device cuts fall on check boundaries and balance the pairs to within one check."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from tests.test_launch_plan import load_launch_plan

HERE = os.path.dirname(os.path.abspath(__file__))
SMS = 148
PAIR_COST = 8444
FINAL = 0x80000000


def load_ragged_plan(directory):
    """tests/hostsim/ragged_plan.cu compiled into `directory` and loaded (also used by test_gpu_ragged_check.py)"""
    so = os.path.join(str(directory), "libragged_plan.so")
    subprocess.check_call(["nvcc", "-x", "cu", "-O2", "-std=c++17", "-DSYLOW_HOSTSIM", "-shared", "-Xcompiler", "-fPIC",
                           "-w", "-o", so, os.path.join(HERE, "hostsim", "ragged_plan.cu")])
    lib = ctypes.CDLL(so)
    lib.rp_build.restype = ctypes.c_void_p
    lib.rp_build.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int, ctypes.c_void_p,
                             ctypes.c_uint64]
    lib.rp_words.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    lib.rp_free.argtypes = [ctypes.c_void_p]
    lib.rp_cuts.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p]
    lib.rp_offsets_ok.argtypes = [ctypes.c_void_p, ctypes.c_uint64]
    lib.rp_chunk.restype = ctypes.c_uint64
    return lib


@pytest.fixture(scope="module")
def rp(tmp_path_factory):
    return load_ragged_plan(tmp_path_factory.mktemp("ragged_plan"))


@pytest.fixture(scope="module")
def lp(tmp_path_factory):
    return load_launch_plan(tmp_path_factory.mktemp("launch_plan"))


def build(rp, offsets, glue=0, sms=SMS):
    """the plan as a dict: glue, n_pairs, items (n4, n2, n1), n_values, gather, levels [(chunk, dst, idx)]"""
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    head = np.zeros(8 + 2 * 16, dtype=np.uint64)
    h = rp.rp_build(sms, offsets.ctypes.data, offsets.size - 1, glue, head.ctypes.data, head.size)
    try:
        n_levels, n_words = int(head[6]), int(head[7])
        assert n_levels <= 16
        words = np.zeros(n_words, dtype=np.uint32)
        rp.rp_words(h, words.ctypes.data)
    finally:
        rp.rp_free(h)
    levels = []
    for l in range(n_levels):
        nc, at = int(head[8 + 2 * l]), int(head[9 + 2 * l])
        chunk = words[at:at + nc + 1].astype(np.int64)
        dst = words[at + nc + 1:at + 2 * nc + 1].astype(np.int64)
        idx = words[at + 2 * nc + 1:at + 2 * nc + 1 + int(chunk[-1])].astype(np.int64)
        levels.append((chunk, dst, idx))
    n_pairs = int(head[1])
    return dict(glue=int(head[0]), n_pairs=n_pairs, items=tuple(int(x) for x in head[2:5]), n_values=int(head[5]),
                gather=words[:n_pairs].astype(np.int64), levels=levels,
                n_words=n_words, used=n_pairs + sum(len(c) + len(d) + len(i) for c, d, i in levels))


def check_plan(rp, offsets, glue=0, sms=SMS, lp=None):
    """builds the plan of `offsets` and asserts every invariant; returns it"""
    offsets = np.asarray(offsets, dtype=np.uint64)
    S = int(rp.rp_chunk())
    p = build(rp, offsets, glue, sms)
    rel = (offsets - offsets[0]).astype(np.int64)
    n_checks = rel.size - 1
    ks = np.diff(rel)
    N = int(rel[-1])
    assert p["n_pairs"] == N and p["used"] == p["n_words"]
    G = p["glue"]
    if glue:
        assert G == glue
    elif lp is not None and N:
        assert G == lp.lp_glue(sms, N, PAIR_COST)
    # every pair gathered exactly once
    g = p["gather"]
    assert np.array_equal(np.sort(g), np.arange(N))
    check_of = lambda x: np.searchsorted(rel[1:], x, side="right")
    # items: 4-pair, then 2-pair, then single, each of consecutive pairs of one check
    n4, n2, n1 = p["items"]
    assert 4 * n4 + 2 * n2 + n1 == N
    val_check, val_pairs = [], []
    at = 0
    for width, count in ((4, n4), (2, n2), (1, n1)):
        it = g[at:at + width * count].reshape(count, width)
        at += width * count
        assert (np.diff(it, axis=1) == 1).all(), width
        c0 = check_of(it[:, 0])
        assert (check_of(it[:, -1]) == c0).all(), width
        val_check.append(c0)
        val_pairs.append(np.full(count, width, np.int64))
        # k / G items of G pairs, and the remainder as at most one 2-pair and one 1-pair item, per check
        per = np.bincount(c0, minlength=n_checks)
        q4 = ks // 4 if G == 4 else np.zeros_like(ks)
        rem = ks - 4 * q4
        q2 = rem // 2 if G >= 2 else np.zeros_like(ks)
        assert np.array_equal(per, {4: q4, 2: q2, 1: rem - 2 * q2}[width]), width
    assert G in ((1, 2, 4) if N else (0,))
    n_items = n4 + n2 + n1
    # values: check and pair count of every value index, items first, chunk products appended
    vc = np.full(p["n_values"], -1, np.int64)
    vp = np.zeros(p["n_values"], np.int64)
    vc[:n_items] = np.concatenate(val_check)
    vp[:n_items] = np.concatenate(val_pairs)
    defined = n_items
    read = np.zeros(p["n_values"], np.int64)
    final_pairs = np.full(n_checks, -1, np.int64)
    for chunk, dst, idx in p["levels"]:
        nc = dst.size
        sizes = np.diff(chunk)
        assert chunk[0] == 0 and (sizes >= 0).all() and sizes.max(initial=0) <= S
        assert (idx < defined).all(), "a value read before it is written"
        np.add.at(read, idx, 1)
        owner = np.repeat(np.arange(nc), sizes)
        first = vc[idx[chunk[:-1][sizes > 0]]]
        ccheck = np.full(nc, -1, np.int64)
        ccheck[sizes > 0] = first
        assert (vc[idx] == ccheck[owner]).all(), "a chunk mixes checks"
        pairs = np.bincount(owner, weights=vp[idx], minlength=nc).astype(np.int64)
        fin = (dst & FINAL) != 0
        slot = dst & ~FINAL
        assert ((sizes > 0) | fin).all(), "an empty chunk is only a final one"
        assert (ccheck[fin & (sizes > 0)] == slot[fin & (sizes > 0)]).all(), "final slot is not the check's"
        assert (final_pairs[slot[fin]] == -1).all(), "a final slot written twice"
        final_pairs[slot[fin]] = pairs[fin]
        mid = ~fin
        assert np.array_equal(slot[mid], np.arange(defined, defined + mid.sum())), "products appended in order"
        vc[slot[mid]] = ccheck[mid]
        vp[slot[mid]] = pairs[mid]
        defined += int(mid.sum())
    assert defined == p["n_values"]
    assert (read == 1).all(), "every value multiplied into exactly one product"
    assert np.array_equal(final_pairs, ks), "check c's final slot covers exactly its pairs"
    return p


def check_cuts(rp, offsets, D):
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    n = offsets.size - 1
    cut = np.zeros(D + 1, dtype=np.uint64)
    rp.rp_cuts(offsets.ctypes.data, n, D, cut.ctypes.data)
    cut = cut.astype(np.int64)
    rel = (offsets - offsets[0]).astype(np.int64)
    N = int(rel[-1])
    assert cut[0] == 0 and cut[-1] == n and (np.diff(cut) >= 0).all()
    ks = np.diff(rel)
    kmax = int(ks.max(initial=0))
    for g in range(1, D):
        c = cut[g]
        assert c == n or rel[c] * D >= g * N  # the first check at or past the target
        assert c == 0 or rel[c - 1] * D < g * N
    for g in range(D):
        pairs = int(rel[cut[g + 1]] - rel[cut[g]])
        assert abs(pairs * D - N) <= 2 * kmax * D, (g, pairs, N, D)  # within one check at each end of the slice
    return cut


def test_no_checks_and_empty_checks(rp):
    p = check_plan(rp, [5])
    assert p["levels"] == [] and p["items"] == (0, 0, 0)
    for n in (1, 3, 1000):
        p = check_plan(rp, [7] * (n + 1))
        assert p["items"] == (0, 0, 0) and len(p["levels"]) == 1  # one empty chunk (the product 1) per check
        assert (np.diff(p["levels"][0][0]) == 0).all()
    for D in (1, 2, 8):
        check_cuts(rp, [3] * 6, D)


@pytest.mark.parametrize("glue", [1, 2, 4])
@pytest.mark.parametrize("k", range(1, 10))
def test_one_check(rp, glue, k):
    p = check_plan(rp, [11, 11 + k], glue)
    n4, n2, n1 = p["items"]
    assert (n4, n2, n1) == {4: (k // 4, k % 4 // 2, k % 2), 2: (0, k // 2, k % 2), 1: (0, 0, k)}[glue]


def test_many_single_pair_checks(rp, lp):
    n = 1 << 20
    p = check_plan(rp, np.arange(n + 1), lp=lp)
    assert p["glue"] == 4 and p["items"] == (0, 0, n) and len(p["levels"]) == 1


def test_one_long_check(rp, lp):
    n = 1 << 20
    p = check_plan(rp, [0, n], lp=lp)
    assert p["glue"] == 4 and p["items"] == (n // 4, 0, 0)
    # 2^18 values -> 2^13 -> 2^8 -> 8 -> the final slot
    assert [c[1].size for c in p["levels"]] == [1 << 13, 1 << 8, 8, 1]


@pytest.mark.parametrize("items, levels", [("S", 1), ("S+1", 2), ("S*S+1", 3)])
def test_chunk_seams(rp, items, levels):
    S = int(rp.rp_chunk())
    m = eval(items, {"S": S})
    p = check_plan(rp, [0, 3, 3 + m, 3 + m + 5], glue=1)
    assert len(p["levels"]) == levels
    assert max(int(np.diff(c).max()) for c, _, _ in p["levels"]) == S


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("sms", [148, 132, 7])
def test_random_mixes(rp, lp, seed, sms):
    rng = random.Random(seed * 1000 + sms)
    n = rng.choice([1, 5, 100, 3000])
    ks = [0 if rng.random() < 0.2 else rng.choice([1, 2, 3, 4, 5, 6, 8, 12, rng.randrange(1, 200)]) for _ in range(n)]
    if seed == 5:
        ks[rng.randrange(n)] = 40000  # one check of more than S^2 values among short ones
    offsets = np.concatenate([[rng.randrange(1000)], np.cumsum(ks)]).astype(np.uint64)
    offsets[1:] += offsets[0]
    for glue in (0, 1, 2, 4):
        check_plan(rp, offsets, glue, sms, lp)
    for D in (1, 2, 3, 8):
        check_cuts(rp, offsets, D)


def test_cuts_in_a_run_of_long_checks(rp):
    ks = [1] * 5 + [5000] * 7 + [3] * 11
    offsets = np.concatenate([[0], np.cumsum(ks)])
    cut = check_cuts(rp, offsets, 2)
    assert 5 < cut[1] < 12  # inside the long run
    check_cuts(rp, offsets, 4)


def test_offsets_ok(rp):
    ok = lambda o: bool(rp.rp_offsets_ok(np.ascontiguousarray(o, np.uint64).ctypes.data, len(o) - 1))
    assert ok([0]) and ok([3, 3, 5, 9]) and not ok([0, 5, 4]) and not ok([2, 1])

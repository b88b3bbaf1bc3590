"""CPU tier: the launch policy of the batch kernels (sylow_b200/csrc/launch_plan.h), with the block shapes of
csrc/kernels_pairing.cuh, compiled for the host (tests/hostsim/launch_plan.cu).  Pins the launches that launch_miller,
launch_final_exp and launch_check_products make on 148 SMs (a B200) in the three SYLOW_B200_LANES modes, and
glue_pairs' pairs per thread."""
import ctypes
import os
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
SMS = 148
MILLER, FEXP = 0, 1
NEVER, AUTO, ALWAYS = 0, 1, 2  # SYLOW_B200_LANES


@pytest.fixture(scope="module")
def lp(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("launch_plan") / "liblaunch_plan.so")
    subprocess.check_call(["nvcc", "-x", "cu", "-O2", "-std=c++17", "-DSYLOW_HOSTSIM", "-shared", "-Xcompiler", "-fPIC",
                           "-w", "-o", so, os.path.join(HERE, "hostsim", "launch_plan.cu")])
    lib = ctypes.CDLL(so)
    lib.lp_batch.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_uint64, ctypes.c_int, ctypes.c_void_p]
    lib.lp_check.argtypes = [ctypes.c_int, ctypes.c_uint64, ctypes.c_int, ctypes.c_void_p]
    lib.lp_glue.argtypes = [ctypes.c_int, ctypes.c_uint64, ctypes.c_uint64]
    return lib


def _launches(lp, kernel, n, mode, sms=SMS):
    """[(first, count, blocks, threads, two lanes), ...] in launch order"""
    out = (ctypes.c_uint64 * 10)()
    k = lp.lp_batch(kernel, sms, n, mode, out)
    return [tuple(out[5 * i:5 * i + 4]) + (bool(out[5 * i + 4]),) for i in range(k)]


def _check(lp, n_checks, mode, sms=SMS):
    out = (ctypes.c_uint64 * 5)()
    lp.lp_check(sms, n_checks, mode, out)
    return tuple(out[:4]) + (bool(out[4]),)


@pytest.mark.parametrize("kernel, n, mode, launches", [
    # 2^20: whole waves of k_miller; k_final_exp's remainder (< 0.6 wave, too large for two lanes) at low occupancy
    (MILLER, 1 << 20, AUTO, [(0, 1048576, 8192, 128, False)]),
    (FEXP, 1 << 20, AUTO, [(0, 1022976, 2664, 384, False), (1022976, 25600, 134, 192, False)]),
    # 2^17 (a 2^20 batch over 8 GPUs): the remainder after the whole waves on two lanes, 64 pairs per block
    (MILLER, 1 << 17, AUTO, [(0, 113664, 888, 128, False), (113664, 17408, 272, 128, True)]),
    (FEXP, 1 << 17, AUTO, [(0, 113664, 296, 384, False), (113664, 17408, 272, 128, True)]),
    # a small batch: two lanes only, one warp (16 pairs) per block
    (MILLER, 5, AUTO, [(0, 5, 1, 32, True)]),
    (FEXP, 5, AUTO, [(0, 5, 1, 32, True)]),
    # one two-lane wave exactly, and one item more (one-thread kernels at low occupancy)
    (MILLER, 148 * 128, AUTO, [(0, 18944, 296, 128, True)]),
    (MILLER, 148 * 128 + 1, AUTO, [(0, 18945, 198, 96, False)]),
    (FEXP, 148 * 128 + 1, AUTO, [(0, 18945, 119, 160, False)]),
    # SYLOW_B200_LANES=0: the remainders as low-occupancy one-thread launches instead
    (MILLER, 1 << 17, NEVER, [(0, 113664, 888, 128, False), (113664, 17408, 272, 64, False)]),
    (FEXP, 1 << 17, NEVER, [(0, 113664, 296, 384, False), (113664, 17408, 136, 128, False)]),
    (MILLER, 5, NEVER, [(0, 5, 1, 32, False)]),
    # SYLOW_B200_LANES=2: everything on two lanes
    (MILLER, 1 << 20, ALWAYS, [(0, 1048576, 16384, 128, True)]),
    (FEXP, 1 << 17, ALWAYS, [(0, 131072, 2048, 128, True)]),
])
def test_batch_launches(lp, kernel, n, mode, launches):
    assert _launches(lp, kernel, n, mode) == launches


@pytest.mark.parametrize("n_checks, mode, launch", [
    (5, AUTO, (0, 5, 1, 32, True)),
    (5, NEVER, (0, 5, 1, 32, False)),
    (148 * 128, AUTO, (0, 18944, 296, 128, True)),
    (148 * 128, NEVER, (0, 18944, 148, 128, False)),
    # more than one two-lane wave: the fused one-thread kernel whatever the mode (2 does not force two lanes here)
    (148 * 128 + 1, ALWAYS, (0, 18945, 119, 160, False)),
    (1 << 20, AUTO, (0, 1048576, 2731, 384, False)),
    (1 << 20, ALWAYS, (0, 1048576, 2731, 384, False)),
])
def test_check_products_launch(lp, n_checks, mode, launch):
    assert _check(lp, n_checks, mode) == launch


@pytest.mark.parametrize("n, glue", [(1 << 13, 1), (1 << 16, 2), (1 << 20, 4)])
@pytest.mark.parametrize("pair_cost", [8444, 6045])  # a fused pair, a pair against a precomputed table
def test_glue_pairs(lp, n, glue, pair_cost):
    assert lp.lp_glue(SMS, n, pair_cost) == glue


@pytest.mark.parametrize("sms", [1, 7, 132, 148])
def test_launches_cover_the_batch(lp, sms):
    """Every plan launches [0, n) once, in order, with no block that has nothing to do."""
    sizes = sorted({n for w in (sms * 128, sms * 256, sms * 384) for m in range(0, 9 * w, w) for n in (m - 1, m + 1,
                                                                                                     m + w * 6 // 10)
                    if n >= 1} | set(range(1, 300)))
    for n in sizes:
        for kernel in (MILLER, FEXP):
            for mode in (NEVER, AUTO, ALWAYS):
                plan = _launches(lp, kernel, n, mode, sms)
                assert 1 <= len(plan) <= 2
                end = 0
                for first, count, blocks, threads, lanes in plan:
                    per_block = threads // 2 if lanes else threads
                    assert first == end and count > 0 and threads % 32 == 0, (n, kernel, mode, plan)
                    assert (blocks - 1) * per_block < count <= blocks * per_block, (n, kernel, mode, plan)
                    end += count
                assert end == n, (n, kernel, mode, plan)

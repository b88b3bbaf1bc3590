#!/usr/bin/env python3
"""Ragged pairing checks: one pairing_check_ragged_batch_dev call against the uniform pairing_check_batch_dev.

All points are resident on the device (G1: random multiples of the generator; G2: a pool of 64 generator multiples), so
the verdicts are mostly false; the two paths must agree on them.  Times are CUDA events around each call, after warm-up
calls of every shape, with the paths alternating call by call; the ragged call's time includes building its launch plan
on the host.  Configurations:
  uniform k = 2 and k = 4 at 2^16 and 2^18 checks: ragged with offsets c k against pairing_check_batch_dev
  mix: k drawn from {2, 3, 4, 6} (uniformly, seed 1) at 2^14 and 2^16 checks: one ragged call against one
       pairing_check_batch_dev per length (inputs grouped by length beforehand, untimed), and the ragged call with
       SYLOW_B200_RAGGED_GLUE=1 (one pair per Miller loop, no gluing)
Prints the device name and power limit first and one JSON line per configuration.

    python tools/ragged_check_time.py [--warmup 2] [--reps 5] [--out /tmp/ragged.log]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
import sylow_b200  # noqa: E402


def power_limit() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def timed(fn) -> float:
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def scalars(rng, n):
    s = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    s[:, 31] &= 0x1F  # < 2^253 < r
    s[:, 0] |= 1
    return s


def points(eng, n, rng, dev):
    g1, _ = eng.g1_mul_generator_batch(scalars(rng, n))
    pool, _ = eng.g2_mul_generator_batch(scalars(rng, 64))
    g2 = pool[rng.integers(0, 64, size=n)]
    return torch.from_numpy(g1).to(dev), torch.from_numpy(g2).to(dev)


def run(eng, paths, warmup, reps):
    """{name: [ms per rep]} with the paths alternating; each path returns its verdicts on the device"""
    for _ in range(warmup):
        for fn in paths.values():
            fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in paths}
    for _ in range(reps):
        for k, fn in paths.items():
            ms[k].append(round(timed(fn), 3))
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    props = torch.cuda.get_device_properties(0)
    lines = ["device: %s, %d SMs; power.limit, clocks.max.sm: %s" % (props.name, props.multi_processor_count,
                                                                     power_limit())]
    print(lines[0], flush=True)
    eng = sylow_b200.Engine(0)
    rng = np.random.default_rng(1)

    def ragged(g1, g2, offs, ok, glue=None):
        def fn():
            if glue:
                os.environ["SYLOW_B200_RAGGED_GLUE"] = str(glue)
            try:
                eng.pairing_check_ragged_batch_dev(g1, g2, offs, ok)
            finally:
                os.environ.pop("SYLOW_B200_RAGGED_GLUE", None)
        return fn

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        lines.append(line)

    for k in (2, 4):
        for log2 in (16, 18):
            n = 1 << log2
            g1, g2 = points(eng, n * k, rng, dev)
            offs = np.arange(n + 1, dtype=np.uint64) * k
            ok_r = torch.zeros(n, dtype=torch.uint8, device=dev)
            ok_u = torch.zeros(n, dtype=torch.uint8, device=dev)
            ms = run(eng, {"ragged": ragged(g1, g2, offs, ok_r),
                           "uniform": lambda: eng.pairing_check_batch_dev(g1, g2, k, ok_u)}, a.warmup, a.reps)
            med = {p: statistics.median(v) for p, v in ms.items()}
            emit({"config": "uniform", "k": k, "n_checks": n, "ragged_ms": med["ragged"], "uniform_ms": med["uniform"],
                  "ragged_over_uniform": round(med["ragged"] / med["uniform"], 3), "all_ms": ms,
                  "verdicts_equal": bool(torch.equal(ok_r, ok_u))})
            del g1, g2
    for log2 in (14, 16):
        n = 1 << log2
        ks = rng.choice([2, 3, 4, 6], size=n)
        offs = np.concatenate([[0], np.cumsum(ks)]).astype(np.uint64)
        g1, g2 = points(eng, int(offs[-1]), rng, dev)
        ok_r = torch.zeros(n, dtype=torch.uint8, device=dev)
        ok_1 = torch.zeros(n, dtype=torch.uint8, device=dev)
        groups = {}
        for k in (2, 3, 4, 6):
            sel = np.flatnonzero(ks == k)
            pairs = torch.from_numpy((offs[sel][:, None].astype(np.int64) + np.arange(k)).reshape(-1)).to(dev)
            groups[k] = (sel, g1[pairs].contiguous(), g2[pairs].contiguous(),
                         torch.zeros(sel.size, dtype=torch.uint8, device=dev))

        def per_length():
            for k, (_, a1, a2, ok) in groups.items():
                eng.pairing_check_batch_dev(a1, a2, k, ok)
        ms = run(eng, {"ragged": ragged(g1, g2, offs, ok_r), "per_length": per_length,
                       "ragged_glue1": ragged(g1, g2, offs, ok_1, glue=1)}, a.warmup, a.reps)
        med = {p: statistics.median(v) for p, v in ms.items()}
        u = np.zeros(n, np.uint8)
        for k, (sel, _, _, ok) in groups.items():
            u[sel] = ok.cpu().numpy()
        emit({"config": "mix {2,3,4,6}", "n_checks": n, "n_pairs": int(offs[-1]), "ragged_ms": med["ragged"],
              "per_length_ms": med["per_length"], "ragged_glue1_ms": med["ragged_glue1"],
              "per_length_over_ragged": round(med["per_length"] / med["ragged"], 3),
              "glue1_over_ragged": round(med["ragged_glue1"] / med["ragged"], 3), "all_ms": ms,
              "verdicts_equal": bool((ok_r.cpu().numpy() == u).all() and torch.equal(ok_r, ok_1))})
        del g1, g2, groups
    eng.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

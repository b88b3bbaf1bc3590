#!/usr/bin/env python3
"""Groth16 verification throughput: per-proof verdicts, the weighted batch verdict, and the bare (1,3) check.

For 2^14 and 2^18 valid trapdoor-made proofs at l = 1, 4 and 16 public inputs, all resident on the device, times with
CUDA events (warm-ups first, then the paths alternating call by call):
  each     groth16_verify_each_dev (public-input folding + records + glued (1,3) loop + final exponentiations)
  floor    pairing_check_fixed_batch_dev on [A, -alpha, -L, -C] records assembled beforehand: what verify_each costs
           without folding the public inputs
  batch    groth16_verify_batch_partial_dev, then the partial to the host and verify_batch_finish (host clock around
           the whole, after a device synchronise)
Key preparation (groth16_prepare_vk: validation, three G2 tables, l fixed-base tables) is timed once per l after one
warm-up.  Every verdict must be true.  Prints the device name and power limit first and one JSON line per size.

    python tools/groth16_time.py [--warmup 3] [--reps 5] [--out /tmp/groth16.log]
"""
import argparse
import json
import random
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
import sylow_b200  # noqa: E402
from oracle import bn254_py as o  # noqa: E402
from tests import groth16_ref as g  # noqa: E402
from tests import wire as w  # noqa: E402

R = o.R_ORDER
SEED = bytes(range(32))


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


def wall(fn) -> float:
    torch.cuda.synchronize()
    t = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3


def le(xs) -> np.ndarray:
    return np.frombuffer(b"".join(int(x).to_bytes(32, "little") for x in xs), np.uint8).reshape(-1, 32).copy()


def make(eng, td, n, l, rng):
    """n valid proofs (A || B || C), their inputs (n, 32 l) and the records [A, -alpha, -L, -C] + B of the floor"""
    xs = [[rng.getrandbits(252) for _ in range(l)] for _ in range(n)]
    inv = pow(td.de, -1, R)
    a = [rng.randrange(1, R) for _ in range(n)]
    b = [rng.randrange(1, R) for _ in range(n)]
    ls = [td.l_scalar(x) for x in xs]
    c = [(ai * bi - td.al * td.be - li * td.ga) * inv % R for ai, bi, li in zip(a, b, ls)]
    A = eng.g1_mul_generator_batch(le(a))[0]
    B = eng.g2_mul_generator_batch(le(b))[0]
    C = eng.g1_mul_generator_batch(le(c))[0]
    neg_l = eng.g1_mul_generator_batch(le([-v % R for v in ls]))[0]
    neg_c = eng.g1_mul_generator_batch(le([-v % R for v in c]))[0]
    neg_a = np.tile(np.frombuffer(w.g1_b(g.g1_mul(-td.al)), np.uint8), (n, 1))
    records = np.concatenate([A, neg_a, neg_l, neg_c], axis=1).reshape(4 * n, 64)
    x = le([v for row in xs for v in row]).reshape(n, 32 * l)
    return np.concatenate([A, B, C], axis=1), x, records, B


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=3, help="untimed calls of each path per size (at least 3)")
    ap.add_argument("--reps", type=int, default=5, help="timed calls of each path per size, alternating (at least 5)")
    ap.add_argument("--log2", default="14,18", help="batch sizes as powers of two")
    ap.add_argument("--inputs", default="1,4,16", help="numbers of public inputs")
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if args.warmup < 3 or args.reps < 5:
        sys.exit("--warmup must be at least 3 and --reps at least 5")
    if not torch.cuda.is_available():
        sys.exit("groth16_time.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    props = torch.cuda.get_device_properties(0)
    lines = ["device: %s, %d SMs; power.limit, clocks.max.sm: %s" % (props.name, props.multi_processor_count,
                                                                    power_limit())]
    print(lines[-1], flush=True)
    eng = sylow_b200.Engine(0)
    rng = random.Random(2026)
    for l in [int(v) for v in args.inputs.split(",")]:
        td = g.Trapdoor(l, 1000 + l)
        vk_pts = td.vk()
        vk = np.frombuffer(g.vk_bytes(vk_pts), np.uint8).copy()
        d_vk = torch.empty(sylow_b200.groth16_vk_dev_bytes(l), dtype=torch.uint8, device=dev)
        eng.groth16_prepare_vk(vk, l, d_vk)
        prep_ms = wall(lambda: eng.groth16_prepare_vk(vk, l, d_vk))
        d_tables = torch.empty(3 * sylow_b200.api.TABLE, dtype=torch.uint8, device=dev)
        eng.tables_to_device(eng.g2_precompute(vk[64:448].reshape(3, 128)), d_tables)
        for lg in [int(v) for v in args.log2.split(",")]:
            n = 1 << lg
            proofs, x, records, B = make(eng, td, n, l, rng)
            d_p, d_x = torch.from_numpy(proofs).to(dev), torch.from_numpy(x).to(dev)
            d_rec, d_b = torch.from_numpy(records).to(dev), torch.from_numpy(B).to(dev)
            ok = {p: torch.zeros(n, dtype=torch.uint8, device=dev) for p in ("each", "floor")}
            d_f = torch.empty(384, dtype=torch.uint8, device=dev)
            verdict = {}

            def batch():
                eng.groth16_verify_batch_partial_dev(d_vk, l, d_p, d_x, d_f, SEED)
                verdict["batch"] = eng.verify_batch_finish(d_f.cpu().numpy().reshape(1, 384))

            run = {"each": lambda: eng.groth16_verify_each_dev(d_vk, l, d_p, d_x, ok["each"]),
                   "floor": lambda: eng.pairing_check_fixed_batch_dev(d_rec, d_b, d_tables, 1, 3, ok["floor"]),
                   "batch_partial": lambda: eng.groth16_verify_batch_partial_dev(d_vk, l, d_p, d_x, d_f, SEED)}
            for _ in range(args.warmup):
                for f in run.values():
                    f()
                batch()
            torch.cuda.synchronize()
            ms = {p: [] for p in list(run) + ["batch"]}
            for _ in range(args.reps):
                for p, f in run.items():
                    ms[p].append(timed(f))
                ms["batch"].append(wall(batch))
            same = bool(ok["each"].all()) and bool(ok["floor"].all()) and verdict["batch"] is True
            med = {p: statistics.median(v) for p, v in ms.items()}
            rec = {"n": n, "n_public": l, "each_ms": round(med["each"], 3), "floor_ms": round(med["floor"], 3),
                   "batch_ms": round(med["batch"], 3), "batch_partial_ms": round(med["batch_partial"], 3),
                   "each_per_s": round(n / med["each"] * 1e3), "batch_per_s": round(n / med["batch"] * 1e3),
                   "each_over_floor": round(med["each"] / med["floor"], 3),
                   "batch_speedup_over_each": round(med["each"] / med["batch"], 2), "prepare_vk_ms": round(prep_ms, 2),
                   "all_ms": {p: [round(v, 3) for v in vs] for p, vs in ms.items()}, "verdicts_true": same}
            lines.append(json.dumps(rec))
            print(lines[-1], flush=True)
            if not same:
                sys.exit("a verdict on valid proofs is false at n=%d l=%d" % (n, l))
            del d_p, d_x, d_rec, d_b, ok
    eng.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

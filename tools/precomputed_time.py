#!/usr/bin/env python3
"""Miller products over resident per-pair G2 tables against the fused Miller product, on device-resident inputs.

Builds 2^20 random pairs on the GPU (g1_mul_batch_dev / g2_mul_batch_dev) and their tables (g2_precompute_dev, 17.5 GB),
then times with CUDA events, alternating call by call:
  fused    miller_product_dev (k_miller, lines computed in the loop)
  tables   miller_product_precomputed_dev, no index (pair i uses table i)
  perm     miller_product_precomputed_dev with a random permutation index (and the G1 points gathered the same way)
at 2^13 pairs (137 MB of tables: about the 126 MB of L2), one full wave of one-pair threads (SMs x 256, where both the
fused and the table path run one pair per thread), 2^17 and 2^20 (17.5 GB: streamed from HBM).  The three products must
be bit-identical at every size.  Prints the device name and power limit first and one JSON line per size.

    python tools/precomputed_time.py [--reps 10] [--out /tmp/precomputed_time.log]
"""
import argparse
import json
import subprocess
import sys

import torch

sys.path.insert(0, ".")
import sylow_b200  # noqa: E402

TABLE = 87 * 192


def power_limit() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def glue(n: int, sms: int, pair_cost: int) -> int:
    """Pairs per thread the library picks (glue_pairs in sylow_b200/csrc/launch_plan.h), for the report."""
    wave, save = sms * 256, 63 * 36
    best, g_best = None, 1
    for g, c in ((1, pair_cost), (2, 2 * pair_cost - save), (4, 4 * pair_cost - 3 * save)):
        t = -(-(n // g) // wave) * c
        if n >= g and (best is None or t < best):
            best, g_best = t, g
    return g_best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10, help="timed calls per variant and size (after one warm-up call)")
    ap.add_argument("--log2-max", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("precomputed_time.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    props = torch.cuda.get_device_properties(0)
    lines = ["device: %s, %d SMs; power.limit, clocks.max.sm: %s" % (props.name, props.multi_processor_count,
                                                                    power_limit())]
    print(lines[-1], flush=True)
    eng = sylow_b200.Engine(0)
    gen = torch.Generator(device=dev).manual_seed(2020)
    n_all = 1 << args.log2_max

    def scalars(n):
        s = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device=dev, generator=gen)
        s[:, 31] &= 0x0F
        return s

    d_g1 = torch.empty((n_all, 64), dtype=torch.uint8, device=dev)
    d_g2 = torch.empty((n_all, 128), dtype=torch.uint8, device=dev)
    g1gen = torch.zeros(64, dtype=torch.uint8)
    g1gen[0], g1gen[32] = 1, 2
    g2gen = torch.frombuffer(bytearray(b"".join(int(c).to_bytes(32, "little") for c in (
        10857046999023057135944570762232829481370756359578518086990519993285655852781,
        11559732032986387107991004021392285783925812861821192530917403151452391805634,
        8495653923123431417604973247489272438418190587263600148770280649306958101930,
        4082367875863433681332203403145435568316851327593401208105741076214120093531))), dtype=torch.uint8)
    eng.g1_mul_batch_dev(g1gen.to(dev).expand(n_all, 64).contiguous(), scalars(n_all), d_g1)
    eng.g2_mul_batch_dev(g2gen.to(dev).expand(n_all, 128).contiguous(), scalars(n_all), d_g2)
    d_tables = torch.empty(n_all * TABLE, dtype=torch.uint8, device=dev)

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def timed(fn):
        ev[0].record()
        fn()
        ev[1].record()
        ev[1].synchronize()
        return ev[0].elapsed_time(ev[1])

    eng.g2_precompute_dev(d_g2, d_tables)  # warm-up
    t_pre = sorted(timed(lambda: eng.g2_precompute_dev(d_g2, d_tables)) for _ in range(3))
    rec = {"what": "g2_precompute_dev", "n": n_all, "ms": t_pre, "us_per_table": t_pre[1] * 1e3 / n_all}
    lines.append(json.dumps(rec))
    print(lines[-1], flush=True)

    sms = props.multi_processor_count
    for n in sorted({1 << 13, sms * 256, 1 << 17, n_all}):
        if n > n_all:
            continue
        perm = torch.randperm(n, device=dev, generator=gen).to(torch.int32)
        g1p = d_g1[:n][perm.long()].contiguous()
        out = {k: torch.empty(384, dtype=torch.uint8, device=dev) for k in ("fused", "tables", "perm")}
        calls = {
            "fused": lambda: eng.miller_product_dev(d_g1[:n], d_g2[:n], out["fused"]),
            "tables": lambda: eng.miller_product_precomputed_dev(d_tables, d_g1[:n], out["tables"]),
            "perm": lambda: eng.miller_product_precomputed_dev(d_tables, g1p, out["perm"], d_table_idx=perm),
        }
        for fn in calls.values():
            fn()
        ms = {k: [] for k in calls}
        for _ in range(args.reps):
            for k, fn in calls.items():
                ms[k].append(timed(fn))
        torch.cuda.synchronize()
        same = torch.equal(out["fused"], out["tables"]) and torch.equal(out["fused"], out["perm"])
        med = {k: sorted(v)[len(v) // 2] for k, v in ms.items()}
        rec = {"n": n, "glue_tables": glue(n, sms, 6045), "tables_MB": n * TABLE / 1e6,
               "median_ms": med, "min_ms": {k: min(v) for k, v in ms.items()},
               "fused_over_tables": med["fused"] / med["tables"], "fused_over_perm": med["fused"] / med["perm"],
               "bit_identical": same}
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)
        if not same:
            sys.exit("the three products differ at n = %d" % n)
    eng.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

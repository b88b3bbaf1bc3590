#!/usr/bin/env python3
"""Fixed-base multiplication by the generator against the variable-base ladder on the repeated generator.

For G1 and G2 at 2^10, 2^16, 2^20 and 2^22 random 256-bit scalars on the device, times with CUDA events, alternating
call by call:
  ladder     g1_mul_batch_dev / g2_mul_batch_dev with the generator repeated n times (GLV / 4-dimensional GLS ladder)
  generator  g1_mul_generator_batch_dev / g2_mul_generator_batch_dev (fixed-base table, no doublings)
Both write affine points and infinity flags, which must be byte-identical at every size.  The first generator call
builds the context's table and is not timed (warm-ups).  Prints the device name and power limit first and one JSON
line per group and size.

    python tools/generator_mul_time.py [--warmup 3] [--reps 7] [--out /tmp/generator_mul.log]
"""
import argparse
import json
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
import sylow_b200  # noqa: E402
from oracle import bn254_py as o  # noqa: E402
from tests import wire as w  # noqa: E402


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=3, help="untimed calls of each path per size (at least 3)")
    ap.add_argument("--reps", type=int, default=7, help="timed calls of each path per size, alternating (at least 5)")
    ap.add_argument("--log2", default="10,16,20,22", help="batch sizes as powers of two")
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if args.warmup < 3 or args.reps < 5:
        sys.exit("--warmup must be at least 3 and --reps at least 5")
    if not torch.cuda.is_available():
        sys.exit("generator_mul_time.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    props = torch.cuda.get_device_properties(0)
    lines = ["device: %s, %d SMs; power.limit, clocks.max.sm: %s" % (props.name, props.multi_processor_count,
                                                                    power_limit())]
    print(lines[-1], flush=True)
    eng = sylow_b200.Engine(0)
    rng = np.random.default_rng(2026)
    gens = {"g1": (64, w.g1_b(o.G1_GEN)), "g2": (128, w.g2_b(o.G2_GEN))}
    for lg in [int(x) for x in args.log2.split(",")]:
        n = 1 << lg
        d_k = torch.from_numpy(rng.integers(0, 256, size=(n, 32), dtype=np.uint8)).to(dev)
        for g, (width, gen) in gens.items():
            d_gen = torch.frombuffer(bytearray(gen), dtype=torch.uint8).to(dev).expand(n, width).contiguous()
            outs = {p: (torch.empty((n, width), dtype=torch.uint8, device=dev), torch.empty(n, dtype=torch.uint8,
                                                                                           device=dev))
                    for p in ("ladder", "generator")}
            ladder = getattr(eng, g + "_mul_batch_dev")
            fixed = getattr(eng, g + "_mul_generator_batch_dev")
            run = {"ladder": lambda: ladder(d_gen, d_k, *outs["ladder"]),
                   "generator": lambda: fixed(d_k, *outs["generator"])}
            for _ in range(args.warmup):
                for f in run.values():
                    f()
            torch.cuda.synchronize()
            ms = {p: [] for p in run}
            for _ in range(args.reps):
                for p, f in run.items():
                    ms[p].append(timed(f))
            same = all(torch.equal(a, b) for a, b in zip(outs["ladder"], outs["generator"]))
            med = {p: statistics.median(v) for p, v in ms.items()}
            rec = {"group": g, "n": n, "ladder_ms": round(med["ladder"], 3), "generator_ms": round(med["generator"], 3),
                   "speedup": round(med["ladder"] / med["generator"], 2),
                   "ladder_per_s": round(n / med["ladder"] * 1e3), "generator_per_s": round(n / med["generator"] * 1e3),
                   "ladder_ms_all": [round(x, 3) for x in ms["ladder"]],
                   "generator_ms_all": [round(x, 3) for x in ms["generator"]], "byte_identical": same}
            lines.append(json.dumps(rec))
            print(lines[-1], flush=True)
            if not same:
                sys.exit("generator path differs from the ladder at %s n=%d" % (g, n))
            del d_gen, outs
    eng.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python3
"""Pointwise G1 / G2 addition (g1_add_batch_dev / g2_add_batch_dev) and the EIP-196 ecMul body, timed with CUDA events.

Three parts, each in its own process so that each loads one build of the library:
  shipped   the library as built, from 2^10 to 2^24 points, on both sides of SY_G1_ADD_AFF_MIN_BATCH and
            SY_G2_ADD_AFF_MIN_BATCH
  always    a build with both thresholds 1: every batch writes projective points and k_g*_batch_affine shares one
            inversion between SY_AFF_K points
  never     a build with both thresholds 2^62: every thread inverts its own point
The last two run from 2^8 to 2^17 points and locate the crossovers the thresholds are set from.  The three
must give the same bytes at every size they share (a checksum of the outputs is compared).  The shipped part also
times eip196_mul_batch against g1_mul_batch on the same points and scalars (host forms, 2^16 and 2^20 inputs).

Inputs are seeded random field elements (the addition has no data-dependent branches, so validity does not change
its time).  Prints the device name and power limit first and one JSON line per measurement.

    python tools/group_law_time.py [--reps 9] [--variants-dir DIR] [--out profiles/r03d_group_law.log]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
VARIANTS = {"always": 1, "never": 1 << 62}


def power_limit() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def build_variant(path: str, min_batch: int) -> None:
    from sylow_b200 import build as b
    if os.path.exists(path) and not any(os.path.getmtime(d) > os.path.getmtime(path) for d in b._deps()):
        return
    cmd = ["nvcc"] + b.NVCC_FLAGS + ["-DSY_G%d_ADD_AFF_MIN_BATCH=%dull" % (g, min_batch) for g in (1, 2)] + \
        ["-o", path] + b.sources()
    subprocess.run(cmd, check=True, capture_output=True)


def worker(name: str, log2s, reps: int, eip: bool):
    import numpy as np
    import torch
    import sylow_b200

    dev = torch.device("cuda", 0)
    eng = sylow_b200.Engine(0)
    gen = torch.Generator(device=dev)

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        return a.elapsed_time(b)

    for g, width in (("g1", 64), ("g2", 128)):
        add = getattr(eng, g + "_add_batch_dev")
        for lg in log2s:
            n = 1 << lg
            gen.manual_seed(lg * 2 + (g == "g2"))
            a = torch.randint(0, 256, (n, width), dtype=torch.uint8, device=dev, generator=gen)
            b = torch.randint(0, 256, (n, width), dtype=torch.uint8, device=dev, generator=gen)
            a[:, 31::32] &= 0x1F
            b[:, 31::32] &= 0x1F
            out = torch.empty((n, width), dtype=torch.uint8, device=dev)
            out_inf = torch.empty(n, dtype=torch.uint8, device=dev)
            for _ in range(3):
                add(a, b, out, out_inf)
            torch.cuda.synchronize()
            ms = [timed(lambda: add(a, b, out, out_inf)) for _ in range(reps)]
            chk = int(out.to(torch.int64).sum().item()) * 1000003 + int(out.to(torch.int64)[:, :8].sum().item())
            med = statistics.median(ms)
            print(json.dumps({"part": name, "op": g + "_add_batch_dev", "n": n, "ms": round(med, 4),
                              "per_s": round(n / med * 1e3), "ms_all": [round(x, 4) for x in ms], "checksum": chk}),
                  flush=True)
            del a, b, out, out_inf
            torch.cuda.empty_cache()
    if not eip:
        return
    rng = np.random.default_rng(196)
    for lg in (16, 20):
        n = 1 << lg
        k = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
        pts, _ = eng.g1_mul_generator_batch(k)  # valid, finite points
        s = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
        inputs = np.concatenate([eng.g1_to_be_bytes_batch(pts, scrubbed=True), s[:, ::-1]], axis=1)
        ms = {"eip196_mul_batch": [], "g1_mul_batch": []}
        for r in range(3 + reps):
            for op, fn in (("eip196_mul_batch", lambda: eng.eip196_mul_batch(inputs)),
                           ("g1_mul_batch", lambda: eng.g1_mul_batch(pts, s))):
                t = timed(fn)
                if r >= 3:
                    ms[op].append(t)
        e_out, e_st = eng.eip196_mul_batch(inputs)
        m_out, m_inf = eng.g1_mul_batch(pts, s)
        same = bool((e_st == 0).all()) and bool((e_out == eng.g1_to_be_bytes_batch(m_out, m_inf, scrubbed=True)).all())
        rec = {"part": name, "op": "eip196_mul_vs_g1_mul", "n": n, "same_bytes": same}
        for op, v in ms.items():
            rec[op + "_ms"] = round(statistics.median(v), 3)
            rec[op + "_per_s"] = round(n / statistics.median(v) * 1e3)
        print(json.dumps(rec), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9, help="timed calls per size (at least 5), after 3 untimed ones")
    ap.add_argument("--variants-dir", default=None, help="where the two threshold variants are built (default: temp)")
    ap.add_argument("--out", default=None, help="also write the report to this file")
    ap.add_argument("--worker", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--log2", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.reps < 5:
        sys.exit("--reps must be at least 5")
    if args.worker:
        worker(args.worker, [int(x) for x in args.log2.split(",")], args.reps, args.worker == "shipped")
        return
    import torch
    if not torch.cuda.is_available():
        sys.exit("group_law_time.py needs a CUDA device")
    props = torch.cuda.get_device_properties(0)
    lines = ["device: %s, %d SMs; power.limit, clocks.max.sm: %s" % (props.name, props.multi_processor_count,
                                                                    power_limit())]
    print(lines[-1], flush=True)
    vdir = args.variants_dir or tempfile.mkdtemp(prefix="sylow_group_law_")
    os.makedirs(vdir, exist_ok=True)
    from sylow_b200 import build as b
    parts = [("shipped", b.build_library(), ",".join(str(x) for x in range(10, 25)))]
    for name, mb in VARIANTS.items():
        path = os.path.join(vdir, "libsylow_b200_add_%s.so" % name)
        build_variant(path, mb)
        parts.append((name, path, ",".join(str(x) for x in range(8, 18))))
    recs = []
    for name, lib, log2 in parts:
        env = dict(os.environ, SYLOW_B200_LIB=lib)
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", name, "--log2", log2, "--reps",
                            str(args.reps)], env=env, capture_output=True, text=True, cwd=ROOT)
        if p.returncode:
            sys.exit("%s part failed:\n%s" % (name, p.stderr[-4000:]))
        for line in p.stdout.splitlines():
            lines.append(line)
            recs.append(json.loads(line))
            print(line, flush=True)
    sums = {}
    for r in recs:
        if "checksum" in r:
            sums.setdefault((r["op"], r["n"]), set()).add(r["checksum"])
    same = all(len(v) == 1 for v in sums.values())
    lines.append(json.dumps({"outputs_identical_across_parts": same}))
    print(lines[-1], flush=True)
    ms = {(r["part"], r["op"], r["n"]): r["ms"] for r in recs if "checksum" in r}
    for op in ("g1_add_batch_dev", "g2_add_batch_dev"):
        cross = [n for (p, o_, n) in ms if p == "always" and o_ == op and ms[("always", op, n)] < ms[("never", op, n)]]
        lines.append(json.dumps({"op": op, "shared_inversion_faster_at": sorted(cross)}))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    if not same:
        sys.exit("outputs differ between the threshold variants")


if __name__ == "__main__":
    main()

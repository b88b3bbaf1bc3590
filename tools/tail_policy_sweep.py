#!/usr/bin/env python3
"""Time the Miller-loop and final-exponentiation launches of one GPU for batch sizes around the wave boundaries under
the lane policies of sylow_b200.cu (SYLOW_B200_LANES, read per call from the environment): 0 one thread per item only,
1 automatic, 2 two lanes per item always.
  tools/tail_policy_sweep.py [sizes, comma-separated] [policies, comma-separated, e.g. 0,1]
Prints one JSON line per policy: ms per call of miller_loop_batch_dev / final_exp_batch_dev / pairing_batch_dev."""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch, sylow_b200

eng = sylow_b200.Engine(0)
dev = torch.device("cuda", 0)
sizes = [int(x) for x in sys.argv[1].split(",")] if len(sys.argv) > 1 else \
    [1, 64, 1024, 4096, 9472, 14000, 18944, 25000, 1 << 15, 1 << 16, 80776, 113664, 1 << 17, 1 << 18, 257328]
policies = sys.argv[2].split(",") if len(sys.argv) > 2 else ["0", "1", "2"]
nmax = max(sizes)
g1 = torch.randint(0, 255, (nmax, 64), dtype=torch.uint8, device=dev)
g2 = torch.randint(0, 255, (nmax, 128), dtype=torch.uint8, device=dev)
g1[:, 31::32] &= 0x1F
g2[:, 31::32] &= 0x1F
f = torch.empty((nmax, 384), dtype=torch.uint8, device=dev)
gt = torch.empty((nmax, 384), dtype=torch.uint8, device=dev)
ref = {}


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return round(a.elapsed_time(b) / reps, 4)


for lanes in policies:
    os.environ["SYLOW_B200_LANES"] = lanes
    out = {"lanes": lanes, "miller_ms": {}, "fexp_ms": {}, "pairing_ms": {}, "same_bits": True}
    for n in sizes:
        reps = 2 if n > (1 << 17) else 5
        a1, a2, af, ag = g1[:n], g2[:n], f[:n], gt[:n]
        out["miller_ms"][n] = timed(lambda: eng.miller_loop_batch_dev(a1, a2, af), reps)
        out["fexp_ms"][n] = timed(lambda: eng.final_exp_batch_dev(af, ag), reps)
        out["pairing_ms"][n] = timed(lambda: eng.pairing_batch_dev(a1, a2, ag), reps)
        # every policy must give the same bytes (checksum of the Gt values of this size)
        chk = int(ag.to(torch.int64).mul(torch.arange(1, 385, device=dev)).sum().item())
        if n in ref and ref[n] != chk:
            out["same_bits"] = False
        ref.setdefault(n, chk)
    print(json.dumps(out), flush=True)

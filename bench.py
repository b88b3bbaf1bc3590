#!/usr/bin/env python3
"""bench.py - BN254 pairings/sec and BLS verifies/sec on N B200s, beside the host-core CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--log2n 20] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[1]): a batch of 2^20 independent optimal-ate pairings on random
G1 x G2 points per GPU (weak scaling: every rank runs its own contiguous 2^20 slice, no data-path
collective).  One "step" = one pass of pairing_batch (fused Miller loop kernel + final-exponentiation
kernel) over the whole batch.  `value` is timed with CUDA events with inputs resident in HBM;
`e2e` goes through the host-pointer C-ABI call with pinned host buffers (H2D + D2H inside the timed
region).  The inputs (192 MiB) and outputs (384 MiB) are larger than the 126 MB L2.

Beside the headline the same JSON line carries
  * `strong`: ONE 2^20 batch sharded over the N ranks (BASELINE configs[1] as written), with its efficiency
    against N times the single-GPU rate;
  * `small_batches`: batches that cannot fill the GPU with one thread per pairing, with the two-lane kernels
    (csrc/pairing_lanes.cuh) and with the one-thread kernels only;
  * `verify_batch` (BASELINE configs[2], the other half of the metric): BLS verifies/s at 2^20 distinct signers
    per GPU - device-resident `value`, host-buffer `e2e` through sylow_b200_verify_batch (>= 5 repetitions), the
    random-weight (sound per signature) form beside the reference example's unweighted product, its own
    `roofline` and `cpu_baseline` (both CPU forms: `verify` per signature and the example's batch form);
  * `other_configs`: BASELINE configs[3] (Groth16-shaped checks) and [4] (2^22 scalar multiplications) with
    roofline blocks, and the SURVEY 8(f) rows;
  * `parity_checks`: cross-rank checks run inside the timed job - the bilinearity checksum
    prod e(a_i G1, b_i G2) = GT^(sum a_i b_i) over ALL ranks through the 384-byte all-gather, a valid sharded
    verify_batch, and one with a corrupted signature on the LAST rank that every rank must reject.
Every `roofline` block carries three readings of the integer-multiply pipe: the algorithmic fraction
(SURVEY 8(d) units / time / measured peak), ncu's fmaheavy-pipe utilisation, and the EXECUTED IMAD.WIDE rate over the
peak (the last two from the committed ncu captures, profiles/r02_ncu_summary.json), plus the analytic peak.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# SURVEY.md 8(d): algorithmic work units (Fp multiplications per item; 136 limb products per Fp multiplication)
LIMB_PRODUCTS_PER_FP_MUL = 136        # 8-limb CIOS: 64 (a*b) + 64 (m*p) + 8 (m)
FP_MUL_MILLER_FUSED = 8444            # fused Miller loop, per pair
FP_MUL_MILLER_TABLE = 6045            # Miller loop against a precomputed / shared G2 table
FP_MUL_FINAL_EXP = 8822 + 380         # final exponentiation + one Fermat inversion (the unit SURVEY counts)
FP_MUL_HASH_TO_G1 = 2900              # 2 SvdW maps + add (Keccak excluded)
FP_MUL_G1_MUL = 3440                  # the reference's 256-step ladder (we execute a GLV ladder: about 2 000)
FP_MUL_G2_MUL = 10300                 # (we execute a 4-dimensional GLS ladder: about 4 900)
FP12_SQR = 36                         # shared squaring of a glued loop (efficient-formula column of SURVEY 8a)
# one Groth16-shaped check: a fused pair + 3 table pairs sharing the 63 squarings + one final exponentiation
FP_MUL_GROTH16_CHECK = FP_MUL_MILLER_FUSED + 3 * (FP_MUL_MILLER_TABLE - 63 * FP12_SQR) + FP_MUL_FINAL_EXP
R_ORDER = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
NCU_SUMMARY = os.path.join(ROOT, "profiles", "r02_ncu_summary.json")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2n", type=int, default=20, help="log2 of pairings per GPU per step")
    ap.add_argument("--verify-log2n", type=int, default=20, help="log2 of signatures for the verify_batch leg (0 = skip)")
    ap.add_argument("--extras", type=int, default=1, help="also time the Groth16-shaped check and scalar-mul configs")
    ap.add_argument("--groth-log2n", type=int, default=18)
    ap.add_argument("--mul-log2n", type=int, default=22)
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="budget of each cpu_baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a fixed sample of rank 0's last-step pairings to DIR as .npy "
                         "(inputs are seeded, so two builds run with the same arguments can be compared)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle timed on the host cores ("port": sylow itself cannot be built here, DESIGN.md)
# ------------------------------------------------------------------------------------------------
def cpu_pairings_per_s(budget_s: float):
    """Times the CPU restatement of sylow's pairing on a bounded sample of the same workload, with
    every host core.  Returns (pairings/s, cores, kind, sample description)."""
    try:
        from oracle import c_oracle

        if c_oracle.available():
            return c_oracle.time_pairings(budget_s)
    except Exception as e:  # the C oracle is optional test infrastructure; fall back to the Python one
        print("bench: C oracle unavailable (%s); timing the Python oracle" % e, file=sys.stderr)
    import random

    from oracle import bn254_py as o
    from tests import wire as w

    rng = random.Random(1)
    pts = [(w.rand_g1(rng), w.rand_g2(rng)) for _ in range(4)]
    t0 = time.perf_counter()
    done = 0
    while time.perf_counter() - t0 < budget_s:
        p, q = pts[done % 4]
        o.pairing_affine(p, q)
        done += 1
    dt = time.perf_counter() - t0
    return done / dt, 1, "port", "%d pairings, Python big-int oracle, 1 thread" % done


def cpu_verifies(budget_s: float):
    """Both CPU forms of the BLS half of the metric on all host cores: `verify` per signature (src/lib.rs:223-236: hash +
    two full pairings) and the example's batch form (examples/verify_multiple_messages_same_signer.rs:40-60)."""
    try:
        from oracle import c_oracle

        if not c_oracle.available():
            return None
        v1, cores, kind, s1 = c_oracle.time_verifies(budget_s / 2, batch_form=False)
        v2, _, _, s2 = c_oracle.time_verifies(budget_s / 2, batch_form=True)
        return {"value": v2, "unit": "verifies/s", "cores": cores, "kind": kind, "sample": s2,
                "verify_each": {"value": v1, "unit": "verifies/s", "sample": s1}}
    except Exception as e:
        print("bench: CPU verify baseline unavailable (%s)" % e, file=sys.stderr)
        return None


PUBLISHED = {"pairing_ms": 8.183, "pairings_per_s_per_core": 1e3 / 8.183, "sign_us": 954.0,
             "source": "sylow_devguide.pdf (hardware unstated)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t_all = time.perf_counter()
    vals = []
    steps = max(1, args.steps)
    per_step = max(1.0, min(20.0, 120.0 / (steps + args.warmup)))
    for i in range(args.warmup + steps):
        v, cores, kind, sample = cpu_pairings_per_s(per_step)
        if i >= args.warmup:
            vals.append(v)
    value = sum(vals) / len(vals)
    line = {
        "impl": "reference", "metric": "pairings_per_s", "value": value, "unit": "pairings/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "2^%d independent optimal-ate pairings (Miller loop + final exponentiation) on "
                               "random G1xG2 points per GPU, BASELINE configs[1]" % args.log2n,
                   "pairings_per_gpu_per_step": 1 << args.log2n,
                   "sample": "each step times a bounded sample of that workload on all host cores"},
        "reference_published": PUBLISHED,
        "cpu_baseline": {"value": value, "unit": "pairings/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "pairings/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    cv = cpu_verifies(min(20.0, args.cpu_seconds * 2))
    if cv:
        line["verify_batch"] = {"value": cv["value"], "unit": "verifies/s", "cpu_baseline": cv,
                                "e2e": {"value": cv["value"], "unit": "verifies/s", "h2d_bytes_per_step": 0,
                                        "d2h_bytes_per_step": 0}}
    line["wall_s"] = time.perf_counter() - t_all
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self._stop_evt = threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 7:
                    self.samples.append(f)
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


def load_ncu_summary():
    try:
        with open(NCU_SUMMARY) as f:
            return json.load(f)
    except Exception:
        return {}


def roofline_block(kernel: str, label: str, n_items: int, fp_mul_per_item: float, ms: float, peak: float, analytic: float,
                   ncu: dict, algorithmic_bytes_per_item: int, unit_note: str = ""):
    """One roofline block.  achieved = SURVEY 8(d) algorithmic limb products per launch / measured launch time."""
    lp = n_items * fp_mul_per_item * LIMB_PRODUCTS_PER_FP_MUL / (ms * 1e-3)
    cap = (ncu or {}).get(kernel) or {}
    executed = None
    if cap.get("inst_executed") and cap.get("imad_wide_share") and cap.get("n"):
        # warp-level IMAD.WIDE(.X) instructions of the capture, scaled to this launch's items, x 32 lanes, over the LIVE time
        per_item = cap["inst_executed"] * cap["imad_wide_share"] * 32.0 / cap["n"]
        executed = per_item * n_items / (ms * 1e-3)
    blk = {
        "bound": "imad", "kernel": label, "achieved": lp / 1e12, "peak": peak / 1e12,
        "unit": "T limb-products/s (32x32->64 multiply-adds)", "frac": lp / peak,
        "ms_per_launch": ms, "fp_mul_per_item": fp_mul_per_item,
        "peak_source": "self-measured live (not in MEASURED_PEAKS.json): IMAD.WIDE.U32.X carry-chain probe on all SMs",
        "peak_analytic": analytic / 1e12,
        "peak_analytic_note": "SMs x 4 schedulers x 8 lanes/clk (one IMAD.WIDE warp instruction per 4 cycles) x SM clock under load",
        "ncu_fmaheavy_pipe_pct": cap.get("fmaheavy_pct"),
        "executed_imad_wide": None if executed is None else {"rate": executed / 1e12, "frac": executed / peak},
        "traffic": cap.get("dram_bytes") and cap["dram_bytes"] * n_items / cap["n"],
        "algorithmic_bytes": n_items * algorithmic_bytes_per_item,
        "hbm_gbs_load_store": n_items * algorithmic_bytes_per_item / (ms * 1e-3) / 1e9,
        "ncu_capture": cap.get("source"),
    }
    if unit_note:
        blk["unit_note"] = unit_note
    return blk


DUMP_ROWS = 1 << 15  # sampled pairings: 32768 x 96 limbs x 8 bytes = 24 MiB


def dump_pairing_outputs(out_dir: str, d_out) -> None:
    """Writes a fixed, seeded sample of the rows of d_out: pairing_batch.npy holds the Gt values as float64
    (rows, 12, 8) - 12 Fp coefficients of 8 little-endian 32-bit limbs each, every limb exact in float64 - and
    pairing_batch_rows.npy the batch indices of those rows."""
    import numpy as np
    import torch

    n = d_out.shape[0]
    rows = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    sample = d_out[torch.from_numpy(rows).to(d_out.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "pairing_batch.npy"), sample.view("<u4").reshape(len(rows), 12, 8).astype(np.float64))
    np.save(os.path.join(out_dir, "pairing_batch_rows.npy"), rows.astype(np.float64))


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    import sylow_b200
    from sylow_b200 import sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the CUDA path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    eng = sylow_b200.Engine(local)
    n = 1 << args.log2n
    K, W = args.steps, max(3, args.warmup)
    ncu = load_ncu_summary()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_true(x: bool) -> bool:
        if world == 1:
            return bool(x)
        t = torch.tensor([1 if x else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    def time_ms(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    # ---- synthetic inputs, generated on the device: P_i = a_i * G1, Q_i = b_i * G2 (seed 1 + rank)
    rs = np.random.RandomState(1 + rank)

    def rand_scalars(m):
        raw = rs.randint(0, 256, size=(m, 32), dtype=np.uint8)
        raw[:, 31] &= 0x1F  # < 2^253 < r: uniform enough for synthetic inputs, never 0 in practice
        return raw

    g1gen = np.zeros((1, 64), np.uint8)
    g1gen[0, 0], g1gen[0, 32] = 1, 2
    G2_GEN = (10857046999023057135944570762232829481370756359578518086990519993285655852781,
              11559732032986387107991004021392285783925812861821192530917403151452391805634,
              8495653923123431417604973247489272438418190587263600148770280649306958101930,
              4082367875863433681332203403145435568316851327593401208105741076214120093531)  # g2.rs:47-77
    g2gen = np.frombuffer(b"".join(c.to_bytes(32, "little") for c in G2_GEN), dtype=np.uint8).reshape(1, 128)
    t_gen = time.perf_counter()
    h_a, h_b = rand_scalars(n), rand_scalars(n)
    d_g1gen = torch.from_numpy(np.repeat(g1gen, n, axis=0)).to(dev)
    d_g2gen = torch.from_numpy(np.repeat(g2gen, n, axis=0)).to(dev)
    d_a = torch.from_numpy(h_a).to(dev)
    d_b = torch.from_numpy(h_b).to(dev)
    d_g1 = torch.empty((n, 64), dtype=torch.uint8, device=dev)
    d_g2 = torch.empty((n, 128), dtype=torch.uint8, device=dev)
    eng.g1_mul_batch_dev(d_g1gen, d_a, d_g1)
    eng.g2_mul_batch_dev(d_g2gen, d_b, d_g2)
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t_gen
    del d_g1gen, d_g2gen, d_a, d_b
    d_out = torch.empty((n, 384), dtype=torch.uint8, device=dev)

    # ---- IMAD roofline denominator, measured live (IMAD.WIDE.U32.X carry chains, all SMs)
    sms = torch.cuda.get_device_properties(local).multi_processor_count
    best = 0.0
    for _ in range(5):
        ms, ops = eng.imad_probe(12, sms * 8, 256, 2000)
        best = max(best, ops / (ms * 1e-3))
    peak = best  # one IMAD.WIDE.U32 = one 32x32->64 limb product

    # ---- warm-up, then the timed region (CUDA events on torch's current stream = the launch stream)
    for _ in range(W):
        eng.pairing_batch_dev(d_g1, d_g2, d_out)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = eng.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        eng.pairing_batch_dev(d_g1, d_g2, d_out)
    e1.record()
    torch.cuda.synchronize()
    launches = eng.launch_count - l0
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:  # before the legs below overwrite d_out
        dump_pairing_outputs(args.dump_outputs, d_out)
    value = world * n * K / (ms_total * 1e-3)
    analytic = sms * 32.0 * (clocks["sm_mhz"] or 1965.0) * 1e6

    # ---- per-kernel durations for the roofline (same buffers, same stream, CUDA events)
    d_f = torch.empty((n, 384), dtype=torch.uint8, device=dev)
    ms_miller = time_ms(lambda: eng.miller_loop_batch_dev(d_g1, d_g2, d_f))
    ms_fexp = time_ms(lambda: eng.final_exp_batch_dev(d_f, d_out))
    del d_f
    roof = roofline_block("k_miller", "k_miller (fused Miller loop)", n, FP_MUL_MILLER_FUSED, ms_miller, peak, analytic, ncu,
                          192 + 384)
    roof["final_exp"] = roofline_block(
        "k_final_exp", "k_final_exp", n, FP_MUL_FINAL_EXP, ms_fexp, peak, analytic, ncu, 768,
        "SURVEY's unit counts a 380-multiplication Fermat inversion; the kernel runs a binary-GCD inversion instead, so "
        "the algorithmic fraction overstates the multiplier work by about 3 %")

    # ---- e2e: host-pointer C-ABI call, pinned host buffers, H2D + D2H inside the timed region
    h_g1 = torch.empty((n, 64), dtype=torch.uint8).pin_memory()
    h_g2 = torch.empty((n, 128), dtype=torch.uint8).pin_memory()
    h_out = torch.empty((n, 384), dtype=torch.uint8).pin_memory()
    h_g1.copy_(d_g1)
    h_g2.copy_(d_g2)

    def e2e_step():
        st = eng._lib.sylow_b200_pairing_batch(eng._h, ctypes.c_void_p(h_g1.data_ptr()), None,
                                               ctypes.c_void_p(h_g2.data_ptr()), None, n,
                                               ctypes.c_void_p(h_out.data_ptr()))
        if st != 0:
            raise RuntimeError("pairing_batch failed: %d" % st)

    e2e_step()
    Ke = max(1, min(K, 5))
    barrier()
    t0 = time.perf_counter()
    for _ in range(Ke):
        e2e_step()
    dt = max_over_ranks(time.perf_counter() - t0)
    e2e_value = world * n * Ke / dt
    same = bool((h_out[:4096].to(dev) == d_out[:4096]).all().item())

    # ---- strong scaling: ONE batch of 2^log2n pairings, contiguous slice per rank (BASELINE configs[1] as written)
    ns = n // world
    for _ in range(2):
        eng.pairing_batch_dev(d_g1[:ns], d_g2[:ns], d_out[:ns])
    barrier()
    Ks = max(3, min(K, 10))
    e0.record()
    for _ in range(Ks):
        eng.pairing_batch_dev(d_g1[:ns], d_g2[:ns], d_out[:ns])
    e1.record()
    torch.cuda.synchronize()
    ms_strong = max_over_ranks(e0.elapsed_time(e1)) / Ks
    barrier()
    strong_value = ns * world / (ms_strong * 1e-3)
    strong = {"pairings_total": ns * world, "pairings_per_gpu": ns, "value": strong_value, "unit": "pairings/s",
              "ms_per_step": ms_strong, "steps": Ks,
              "efficiency": strong_value / value,
              "efficiency_note": "one 2^%d batch over %d GPUs / (%d x the per-GPU rate of the weak-scaling headline)"
                                 % (args.log2n, world, world),
              "waves_per_gpu": {"k_miller": ns / (sms * 256.0), "k_final_exp": ns / (sms * 384.0)}}

    # ---- batches too small to fill the GPU with one thread per pairing: the two-lane kernels (csrc/pairing_lanes.cuh)
    # against the one-thread kernels on the same inputs (the library reads SYLOW_B200_LANES on every call)
    small = {"unit": "ms per batch", "note": "pairing_batch_dev; two lanes per Miller loop / final exponentiation when "
             "the batch fits one two-lane wave (148 x 128 items), and for wave remainders of larger batches"}
    for m in (1, 1024, 9472, 18944):
        row = {}
        for key, mode in (("two_lanes", None), ("one_thread", "0")):
            if mode is None:
                os.environ.pop("SYLOW_B200_LANES", None)
            else:
                os.environ["SYLOW_B200_LANES"] = mode
            row[key] = time_ms(lambda: eng.pairing_batch_dev(d_g1[:m], d_g2[:m], d_out[:m]), reps=5)
        os.environ.pop("SYLOW_B200_LANES", None)
        small[str(m)] = row

    # ---- cross-rank parity checks (cheap; every N): run BEFORE the long legs so a wrong build fails early
    parity = {}
    m_chk = min(2048, ns)
    d_part = torch.empty(384, dtype=torch.uint8, device=dev)
    eng.miller_product_dev(d_g1[:m_chk], d_g2[:m_chk], d_part)
    parts = sharding.all_gather_partials(d_part.cpu().numpy(), device=dev)
    gt_all = eng.final_exp_batch(eng.fp12_product(parts).reshape(1, 384))
    s_loc = sum(int.from_bytes(h_a[i].tobytes(), "little") * int.from_bytes(h_b[i].tobytes(), "little")
                for i in range(m_chk)) % R_ORDER
    if world > 1:
        sums = [None] * world
        dist.all_gather_object(sums, s_loc)
        s_all = sum(sums) % R_ORDER
    else:
        s_all = s_loc
    gt_gen = eng.pairing_batch(g1gen, g2gen)
    try:
        with open(os.path.join(ROOT, "tests", "golden", "reference_kats.json")) as f:
            kat = json.load(f)["gt_generator"]["fp12"]
        gt_ref = b"".join(int(x, 16).to_bytes(32, "little") for x in kat)
        parity["gt_generator_matches_reference_constant"] = bytes(gt_gen[0]) == gt_ref  # src/groups/gt.rs:20-109
    except Exception:
        parity["gt_generator_matches_reference_constant"] = None
    gt_pow = eng.gt_mul_batch(gt_gen, np.frombuffer(s_all.to_bytes(32, "little"), np.uint8).reshape(1, 32))
    parity["bilinearity_checksum_all_ranks"] = all_true(bool((gt_all == gt_pow).all()))
    parity["bilinearity_pairs"] = m_chk * world

    # ---- the other half of the metric: BLS verify_batch (hash-to-curve + Miller loops + ONE final exponentiation)
    verify = None
    if args.verify_log2n > 0:
        nv = 1 << args.verify_log2n
        msgs = np.zeros((nv, 32), np.uint8)
        msgs[:, :8] = (np.arange(nv, dtype=np.uint64) + np.uint64(rank * nv)).view(np.uint8).reshape(nv, 8)
        msgs[:, 8:] = rs.randint(0, 256, size=(nv, 24), dtype=np.uint8)
        offs = (np.arange(nv + 1, dtype=np.uint64) * 32)
        sks = rand_scalars(nv)
        packed = (msgs.reshape(-1), offs)
        sigs = eng.sign_batch(sks, packed)
        d_sk = torch.from_numpy(sks).to(dev)
        d_pk = torch.empty((nv, 128), dtype=torch.uint8, device=dev)
        eng.g2_mul_batch_dev(torch.from_numpy(np.repeat(g2gen, nv, axis=0)).to(dev), d_sk, d_pk)
        d_msgs = torch.from_numpy(msgs.reshape(-1)).to(dev)
        d_offs = torch.from_numpy(offs.view(np.int64)).to(dev)
        d_sigs = torch.from_numpy(sigs).to(dev)
        seed = bytes((7 * i + 1) & 0xFF for i in range(32))  # every rank uses the same seed; weights follow the global index

        def verify_dev(weighted):
            # per-GPU partial (hash + Miller loops + tree product), then the ONE exchange of the path: all-gather of
            # the 384-byte partials over NCCL, product + one final exponentiation
            eng.verify_batch_partial_dev(d_pk, d_msgs, d_offs, d_sigs, d_part, weight_seed=seed if weighted else None,
                                         first_index=rank * nv)
            return eng.verify_batch_finish(sharding.all_gather_partials(d_part.cpu().numpy(), device=dev))

        def timed(fn, reps):
            ok = fn()
            barrier()
            t0 = time.perf_counter()
            for _ in range(reps):
                ok = fn() and ok
            return max_over_ranks(time.perf_counter() - t0) / reps, ok

        dt_v, ok = timed(lambda: verify_dev(False), 5)
        dt_w, ok_w = timed(lambda: verify_dev(True), 3)
        # host-buffer e2e: pinned host arrays through the C ABI, H2D of keys + messages + signatures inside the timed region
        h_pk = torch.empty((nv, 128), dtype=torch.uint8).pin_memory()
        h_pk.copy_(d_pk)
        h_sg = torch.from_numpy(sigs).pin_memory()
        h_ms = torch.from_numpy(msgs.reshape(-1).copy()).pin_memory()
        h_of = torch.from_numpy(offs.view(np.int64).copy()).pin_memory()
        seed_buf = (ctypes.c_uint8 * 32)(*seed)
        dst = sylow_b200.api.DST
        part_host = np.empty(384, np.uint8)

        def verify_host(weighted):
            sp = ctypes.cast(seed_buf, ctypes.c_void_p) if weighted else None
            if world == 1:
                okc = ctypes.c_int(0)
                st = eng._lib.sylow_b200_verify_batch(eng._h, ctypes.c_void_p(h_pk.data_ptr()), None,
                                                      ctypes.c_void_p(h_ms.data_ptr()), ctypes.c_void_p(h_of.data_ptr()),
                                                      ctypes.c_void_p(h_sg.data_ptr()), None, nv, dst, len(dst), 0, sp,
                                                      ctypes.byref(okc))
                if st != 0:
                    raise RuntimeError("verify_batch failed: %d" % st)
                return bool(okc.value)
            st = eng._lib.sylow_b200_verify_batch_partial(eng._h, ctypes.c_void_p(h_pk.data_ptr()), None,
                                                          ctypes.c_void_p(h_ms.data_ptr()), ctypes.c_void_p(h_of.data_ptr()),
                                                          ctypes.c_void_p(h_sg.data_ptr()), None, nv, dst, len(dst), 0, sp,
                                                          rank * nv, part_host.ctypes.data_as(ctypes.c_void_p))
            if st != 0:
                raise RuntimeError("verify_batch_partial failed: %d" % st)
            return eng.verify_batch_finish(sharding.all_gather_partials(part_host, device=dev))

        dt_e, ok_e = timed(lambda: verify_host(False), 5)
        dt_ew, ok_ew = timed(lambda: verify_host(True), 3)
        ms_v_kernels = time_ms(lambda: eng.verify_batch_partial_dev(d_pk, d_msgs, d_offs, d_sigs, d_part), reps=3)
        d_hm = torch.empty((nv, 64), dtype=torch.uint8, device=dev)
        ms_hash = time_ms(lambda: eng.hash_to_g1_batch_dev(d_msgs, d_offs, d_hm), reps=3)
        # the Miller stage (k_glued<4,0>, which has no entry point of its own, plus the signature sum and the product
        # tree, about 3 %) = the partial product minus the hash, both event-timed on the same buffers
        ms_vm = max(ms_v_kernels - ms_hash, 1e-3)
        # negative case inside the job: the LAST signature of the LAST rank is replaced; every rank must say False
        bad = sigs.copy()
        if rank == world - 1:
            bad[nv - 1] = bad[0]
        m_neg = min(nv, 1 << 14)
        lo = nv - m_neg
        neg_msgs = (msgs[lo:].reshape(-1).copy(), np.arange(m_neg + 1, dtype=np.uint64) * 32)

        def sharded(sg, weighted):
            p = eng.verify_batch_partial(d_pk[lo:].cpu().numpy(), neg_msgs, sg[lo:], weight_seed=seed if weighted else None,
                                         first_index=rank * nv + lo)
            return eng.verify_batch_finish(sharding.all_gather_partials(p, device=dev))

        parity["verify_batch_valid_all_ranks"] = all_true(sharded(sigs, False) and sharded(sigs, True))
        parity["verify_batch_corrupt_last_rank_rejected_by_all"] = all_true((not sharded(bad, False)) and
                                                                            (not sharded(bad, True)))
        parity["verify_batch_signatures"] = m_neg * world
        # S = 1 variant (the reference example's own setting: one signer, many messages), host-pointer call
        same_signer = None
        if world == 1:
            sk1 = np.repeat(sks[:1], nv, axis=0)
            sigs1 = eng.sign_batch(sk1, packed)
            pk1, _ = eng.g2_mul_batch(g2gen, sks[:1])
            eng.verify_batch_same_signer(pk1[0], packed, sigs1)
            t1 = time.perf_counter()
            ok1 = eng.verify_batch_same_signer(pk1[0], packed, sigs1)
            same_signer = {"verifies_per_s": nv / (time.perf_counter() - t1), "batch_ok": bool(ok1),
                           "note": "one signer: n hashes + 2n point additions + two Miller loops per batch, host buffers (e2e)"}
        v_roof = roofline_block("verify", "verify_batch_partial (k_hash_to_g1 + k_g1_batch_affine + k_glued<4,0> + sums)", nv,
                                FP_MUL_HASH_TO_G1 + FP_MUL_MILLER_FUSED, ms_v_kernels, peak, analytic, None, 128 + 32 + 64,
                                "per signature: hash-to-curve 2 900 + fused Miller loop 8 444 Fp multiplications (SURVEY's "
                                "units).  The kernels execute fewer: four signatures share a thread and ONE Fp12 squaring per "
                                "loop digit (63 x 36 multiplications saved for 3 of every 4 pairs), the hash runs binary-GCD / "
                                "Jacobi iterations instead of 5 of its 7 ladders, and the signature side is one point "
                                "addition per signature plus ONE Miller loop per batch - so this fraction can exceed 1; "
                                "the per-kernel blocks carry the executed rates")
        v_roof["kernels"] = {
            "k_hash_to_g1": roofline_block("k_hash_to_g1", "k_hash_to_g1 (+ k_g1_batch_affine)", nv, FP_MUL_HASH_TO_G1, ms_hash,
                                           peak, analytic, ncu, 32 + 64,
                                           "SURVEY's unit counts 7 Fermat ladders; 5 of them are binary-GCD / Jacobi "
                                           "iterations here (ALU work, no multiplier), so the executed rate is far lower"),
            "k_glued<4,0>": roofline_block("k_glued<4,0>", "k_glued<4,0>: four (-H(m_i), pk_i) pairs per thread, shared squarings (+ signature sum, product tree)",
                                           nv, FP_MUL_MILLER_FUSED, ms_vm, peak, analytic,
                                           {"k_glued<4,0>": dict(ncu.get("k_glued<4,0>") or {}, n=4 * (ncu.get("k_glued<4,0>") or {}).get("n", 0))}
                                           if ncu.get("k_glued<4,0>") else None, 192 + 96,
                                           "unit = one separate fused Miller loop per pair (8 444); executed: 8 444 - 3/4 x 2 268")}
        verify = {"metric": "bls_verifies_per_s", "value": world * nv / dt_v, "unit": "verifies/s",
                  "signatures_per_gpu": nv, "distinct_signers": nv, "batch_ok": bool(ok and ok_e),
                  "ms_per_batch": dt_v * 1e3, "reps": 5,
                  "form": "aggregate product of the reference example: prod e(sig_i, G2gen) e(-H(m_i), pk_i) == 1",
                  "e2e": {"value": world * nv / dt_e, "unit": "verifies/s", "h2d_bytes_per_step": nv * (128 + 64 + 32 + 8),
                          "d2h_bytes_per_step": 384 + 4, "reps": 5,
                          "call": "sylow_b200_verify_batch" if world == 1 else
                                  "sylow_b200_verify_batch_partial + NCCL all-gather + sylow_b200_verify_batch_finish"},
                  "weighted": {"value": world * nv / dt_w, "e2e": world * nv / dt_ew, "unit": "verifies/s",
                               "batch_ok": bool(ok_w and ok_ew),
                               "note": "random 64-bit weights (sound per signature): two 64-bit G1 ladders per signature on top"},
                  "ms_partial_kernels": ms_v_kernels, "ms_hash_to_curve": ms_hash, "ms_miller": ms_vm,
                  "verifies_per_s_kernels_only": world * nv / (max_over_ranks(ms_v_kernels) * 1e-3),
                  "same_signer": same_signer, "roofline": v_roof,
                  "note": "per GPU: hash-to-curve + one fused Miller loop per signature, signatures summed into one "
                          "Miller loop against the generator, tree product; all-gather of the 384-byte partials; one "
                          "final exponentiation per batch"}
        del d_hm, d_pk, d_sigs, d_msgs

    # ---- further BASELINE configs, as extra keys (device-resident inputs, CUDA events)
    extras = {}
    if args.extras:
        # config #4: Groth16-shaped 4-pair product check, three G2 points fixed across all checks
        nc = 1 << args.groth_log2n
        co = eng.g2_precompute(d_g2[:3].cpu().numpy())
        d_tab = torch.empty(3 * 87 * 192, dtype=torch.uint8, device=dev)
        eng.tables_to_device(co, d_tab)
        torch.cuda.synchronize()
        d_g1c = d_g1[: 4 * nc].contiguous() if 4 * nc <= n else d_g1.repeat((4 * nc + n - 1) // n, 1)[: 4 * nc].contiguous()
        d_g2c = d_g2[:nc].contiguous()
        d_ok = torch.empty(nc, dtype=torch.uint8, device=dev)
        ms_g = time_ms(lambda: eng.pairing_check_fixed_batch_dev(d_g1c, d_g2c, d_tab, 1, 3, d_ok), reps=3)
        extras["groth16_4pair_checks_per_s"] = world * nc / (max_over_ranks(ms_g) * 1e-3)
        extras["groth16_checks_per_gpu"] = nc
        extras["groth16_roofline"] = roofline_block(
            "k_glued<1,3>", "k_glued<1,3> + k_check_products (4-pair glued loop, one final exponentiation per check)", nc,
            FP_MUL_GROTH16_CHECK, ms_g, peak, analytic, ncu, 4 * 64 + 128 + 1,
            "per check: fused pair 8 444 + 3 table pairs x (6 045 - 63 shared squarings x 36) + final exponentiation 9 202")
        # config #5: variable-base scalar multiplication, 254-bit scalars
        nm = 1 << args.mul_log2n
        d_k = torch.from_numpy(rand_scalars(nm)).to(dev)
        d_p1 = d_g1[:nm].contiguous() if nm <= n else d_g1.repeat((nm + n - 1) // n, 1)[:nm].contiguous()
        d_p2 = d_g2[:nm].contiguous() if nm <= n else d_g2.repeat((nm + n - 1) // n, 1)[:nm].contiguous()
        d_o1 = torch.empty((nm, 64), dtype=torch.uint8, device=dev)
        d_o2 = torch.empty((nm, 128), dtype=torch.uint8, device=dev)
        ms_1 = time_ms(lambda: eng.g1_mul_batch_dev(d_p1, d_k, d_o1), reps=3)
        ms_2 = time_ms(lambda: eng.g2_mul_batch_dev(d_p2, d_k, d_o2), reps=3)
        extras["g1_scalar_muls_per_s"] = world * nm / (max_over_ranks(ms_1) * 1e-3)
        extras["g2_scalar_muls_per_s"] = world * nm / (max_over_ranks(ms_2) * 1e-3)
        extras["scalar_muls_per_gpu"] = nm
        note = ("SURVEY's unit is the reference's 256-step NAF ladder; the kernel runs a GLV / GLS ladder with about "
                "half as many multiplications, so the algorithmic fraction exceeds the executed one")
        extras["g1_mul_roofline"] = roofline_block("k_g1_mul", "k_g1_mul + k_g1_batch_affine", nm, FP_MUL_G1_MUL, ms_1, peak,
                                                   analytic, ncu, 64 + 32 + 64, note)
        extras["g2_mul_roofline"] = roofline_block("k_g2_mul", "k_g2_mul + k_g2_batch_affine", nm, FP_MUL_G2_MUL, ms_2, peak,
                                                   analytic, ncu, 128 + 32 + 128, note)
        del d_k, d_p1, d_p2, d_o1, d_o2
        # SURVEY 8(f) rank 4: threshold aggregation, 2^15 sets of 8 partial signatures (host buffers, wall clock)
        tt = 8
        nsets = max(1, min(1 << 15, n // tt))
        ids = np.tile(np.arange(1, tt + 1, dtype=np.uint64), (nsets, 1)) + (np.arange(nsets, dtype=np.uint64) % 5)[:, None]
        h_sig = d_g1[: nsets * tt].cpu().numpy().reshape(nsets, tt, 64)
        eng.threshold_aggregate_batch(ids, h_sig)
        t0 = time.perf_counter()
        eng.threshold_aggregate_batch(ids, h_sig)
        extras["threshold_aggregations_per_s"] = world * nsets / max_over_ranks(time.perf_counter() - t0)
        extras["threshold_shares_per_set"] = tt

        # SURVEY 8(f) ranks 1-3 through the host-pointer calls (wall clock, copies included; 2^17 items, 2^15 for Gt)
        def wall(fn):
            fn()
            t0 = time.perf_counter()
            fn()
            return max_over_ranks(time.perf_counter() - t0)

        nx = min(1 << 17, n)
        h1 = d_g1[:nx].cpu().numpy()
        h2 = d_g2[:nx].cpu().numpy()
        hk = rand_scalars(nx)
        hm = (np.arange(nx, dtype=np.uint64).view(np.uint8).reshape(nx, 8).copy().reshape(-1),
              np.arange(nx + 1, dtype=np.uint64) * 8)
        extras["next_rows"] = {
            "items": nx,
            "g1_validate_per_s": world * nx / wall(lambda: eng.g1_validate_batch(h1)),
            "g2_validate_per_s": world * nx / wall(lambda: eng.g2_validate_batch(h2)),
            "g2_be_roundtrip_per_s": world * nx / wall(
                lambda: eng.g2_from_be_bytes_batch(eng.g2_to_be_bytes_batch(h2), eip_mode=False)),
            "sign_per_s": world * nx / wall(lambda: eng.sign_batch(hk, hm)),
            "note": "host buffers, wall clock: G1Affine::new / G2Projective::new checks, big-endian codec round trip, sign",
        }
        # one large multi-scalar multiplication (bucket method) next to the same sum by ladders + tree sum
        nm2 = min(1 << 20, n)
        hp, hs = d_g1[:nm2].cpu().numpy(), rand_scalars(nm2)
        t_b = wall(lambda: eng.g1_msm_bucket(hp, hs))
        extras["next_rows"]["g1_msm_2pow%d_ms" % int(np.log2(nm2))] = {"bucket": t_b * 1e3}
        ng = min(1 << 15, n)
        hgt = d_out[:ng].cpu().numpy()
        extras["next_rows"]["gt_mul_per_s"] = world * ng / wall(lambda: eng.gt_mul_batch(hgt, hk[:ng]))

    cpu = cpu_v = None
    if rank == 0 and world == 1:
        v, cores, kind, sample = cpu_pairings_per_s(args.cpu_seconds)
        cpu = {"value": v, "unit": "pairings/s", "cores": cores, "kind": kind, "sample": sample}
        if verify:
            cpu_v = cpu_verifies(args.cpu_seconds)

    if rank == 0:
        line = {
            "metric": "pairings_per_s", "value": value, "unit": "pairings/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32x8 Montgomery (integer)", "data": "synthetic",
            "config": {"workload": "2^%d independent optimal-ate pairings (Miller loop + final exponentiation) on "
                                   "random G1xG2 points per GPU, BASELINE configs[1]" % args.log2n,
                       "pairings_per_gpu_per_step": n, "l2_policy": "inputs+outputs (576 MiB) larger than L2",
                       "parallelism": "contiguous slice per GPU, no data-path collective", "input_gen_s": t_gen},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "pairings/s", "h2d_bytes_per_step": n * 192,
                    "d2h_bytes_per_step": n * 384, "steps": Ke, "matches_device_path": same},
            "gpu_launches": launches,
            "roofline": roof,
            "strong": strong,
            "small_batches": small,
            "parity_checks": parity,
            "reference_published": PUBLISHED,
        }
        if cpu:
            line["cpu_baseline"] = cpu
        if verify:
            if cpu_v:
                verify["cpu_baseline"] = cpu_v
            line["verify_batch"] = verify
        if extras:
            line["other_configs"] = extras
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

"""Batched BN254 engine: Python host binding over the C ABI (include/sylow_b200.h).

Arrays are numpy uint8 in the C-ABI wire formats (see the header): G1 (n, 64), G2 (n, 128),
Fp12/Gt (n, 384), scalars (n, 32), infinity flags (n,) uint8.  The `_dev` methods take torch CUDA
uint8 tensors and enqueue on torch's current stream (used by bench.py for the HBM-resident number).
All compute happens in libsylow_b200.so on the GPU; nothing here computes field arithmetic.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence, Tuple

import numpy as np

from . import _lib

DST = b"WARLOCK-CHAOS-V01-CS01-SHA-256"  # reference src/lib.rs:90


def _u8(a, shape_tail: Optional[int], name: str) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.uint8)
    if shape_tail is not None:
        if a.ndim == 1 and a.size == shape_tail:
            a = a.reshape(1, shape_tail)
        if a.ndim != 2 or a.shape[1] != shape_tail:
            raise ValueError("%s must have shape (n, %d), got %s" % (name, shape_tail, a.shape))
    return a


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def pack_messages(msgs: Sequence[bytes]) -> Tuple[np.ndarray, np.ndarray]:
    """Concatenate messages into (buffer uint8, offsets uint64 of length n+1)."""
    offs = np.zeros(len(msgs) + 1, dtype=np.uint64)
    if len(msgs):
        offs[1:] = np.cumsum([len(m) for m in msgs], dtype=np.uint64)
    buf = np.frombuffer(b"".join(msgs), dtype=np.uint8).copy() if int(offs[-1]) else np.zeros(0, dtype=np.uint8)
    return buf, offs


class Engine:
    """One context: bound to one CUDA device (`Engine(0)`, one process per GPU) or, given a list of devices
    (`Engine([0, 1, 2, 3])`, sylow_b200_create_multi), sharding every batched host-buffer call over them."""

    def __init__(self, device=0):
        self._lib = _lib.load()
        h = ctypes.c_void_p()
        if isinstance(device, (list, tuple)):
            ids = (ctypes.c_int * len(device))(*[int(d) for d in device])
            st = self._lib.sylow_b200_create_multi(ctypes.byref(h), ids, len(device))
            self.device = int(device[0]) if device else 0
        else:
            st = self._lib.sylow_b200_create(ctypes.byref(h), int(device))
            self.device = int(device)
        if st != 0:
            raise _lib.SylowB200Error(st, "sylow_b200_create(device=%r)" % (device,))
        self._h = h

    @property
    def device_count(self) -> int:
        return int(self._lib.sylow_b200_device_count(self._h))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.sylow_b200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, st: int, where: str):
        if st != 0:
            raise _lib.SylowB200Error(st, where, self._lib.sylow_b200_last_cuda_error(self._h))

    @property
    def launch_count(self) -> int:
        return int(self._lib.sylow_b200_launch_count(self._h))

    # ------------------------------------------------------------------ pairing
    def _pairs(self, g1, g2, g1_inf, g2_inf):
        g1 = _u8(g1, 64, "g1")
        g2 = _u8(g2, 128, "g2")
        n = g1.shape[0]
        if g2.shape[0] != n:
            raise ValueError("g1 and g2 batch sizes differ: %d vs %d" % (n, g2.shape[0]))
        g1_inf = None if g1_inf is None else np.ascontiguousarray(g1_inf, dtype=np.uint8).reshape(n)
        g2_inf = None if g2_inf is None else np.ascontiguousarray(g2_inf, dtype=np.uint8).reshape(n)
        return g1, g2, g1_inf, g2_inf, n

    def pairing_batch(self, g1, g2, g1_inf=None, g2_inf=None) -> np.ndarray:
        g1, g2, g1_inf, g2_inf, n = self._pairs(g1, g2, g1_inf, g2_inf)
        out = np.empty((n, 384), dtype=np.uint8)
        self._ck(self._lib.sylow_b200_pairing_batch(self._h, _ptr(g1), _ptr(g1_inf), _ptr(g2), _ptr(g2_inf), n,
                                                    _ptr(out)), "pairing_batch")
        return out

    def miller_loop_batch(self, g1, g2, g1_inf=None, g2_inf=None) -> np.ndarray:
        g1, g2, g1_inf, g2_inf, n = self._pairs(g1, g2, g1_inf, g2_inf)
        out = np.empty((n, 384), dtype=np.uint8)
        self._ck(self._lib.sylow_b200_miller_loop_batch(self._h, _ptr(g1), _ptr(g1_inf), _ptr(g2), _ptr(g2_inf), n,
                                                        _ptr(out)), "miller_loop_batch")
        return out

    def miller_product(self, g1, g2, g1_inf=None, g2_inf=None) -> np.ndarray:
        g1, g2, g1_inf, g2_inf, n = self._pairs(g1, g2, g1_inf, g2_inf)
        out = np.empty(384, dtype=np.uint8)
        self._ck(self._lib.sylow_b200_miller_product(self._h, _ptr(g1), _ptr(g1_inf), _ptr(g2), _ptr(g2_inf), n,
                                                     _ptr(out)), "miller_product")
        return out

    def final_exp_batch(self, f) -> np.ndarray:
        f = _u8(f, 384, "f")
        out = np.empty_like(f)
        self._ck(self._lib.sylow_b200_final_exp_batch(self._h, _ptr(f), f.shape[0], _ptr(out)), "final_exp_batch")
        return out

    def fp12_product(self, f) -> np.ndarray:
        f = _u8(f, 384, "f")
        out = np.empty(384, dtype=np.uint8)
        self._ck(self._lib.sylow_b200_fp12_product(self._h, _ptr(f), f.shape[0], _ptr(out)), "fp12_product")
        return out

    def pairing_check_batch(self, g1, g2, pairs_per_check: int, g1_inf=None, g2_inf=None) -> np.ndarray:
        g1, g2, g1_inf, g2_inf, n = self._pairs(g1, g2, g1_inf, g2_inf)
        k = int(pairs_per_check)
        if k <= 0 or n % k:
            raise ValueError("batch of %d pairs is not a multiple of pairs_per_check=%d" % (n, k))
        ok = np.empty(n // k, dtype=np.uint8)
        self._ck(self._lib.sylow_b200_pairing_check_batch(self._h, _ptr(g1), _ptr(g1_inf), _ptr(g2), _ptr(g2_inf), k,
                                                          n // k, _ptr(ok)), "pairing_check_batch")
        return ok.astype(bool)

    # ------------------------------------------------------------------ precomputed G2
    def g2_precompute(self, g2) -> np.ndarray:
        """G2Affine::precompute: (n, 87, 3, 64) uint8 canonical line coefficients."""
        g2 = _u8(g2, 128, "g2")
        out = np.empty((g2.shape[0], 87 * 192), dtype=np.uint8)
        self._ck(self._lib.sylow_b200_g2_precompute(self._h, _ptr(g2), g2.shape[0], _ptr(out)), "g2_precompute")
        return out

    def miller_loop_precomputed(self, coeffs, g1, g1_inf=None) -> np.ndarray:
        coeffs = np.ascontiguousarray(coeffs, dtype=np.uint8).reshape(87 * 192)
        g1 = _u8(g1, 64, "g1")
        n = g1.shape[0]
        g1_inf = None if g1_inf is None else np.ascontiguousarray(g1_inf, dtype=np.uint8).reshape(n)
        out = np.empty((n, 384), dtype=np.uint8)
        self._ck(self._lib.sylow_b200_miller_loop_precomputed(self._h, _ptr(coeffs), _ptr(g1), _ptr(g1_inf), n,
                                                              _ptr(out)), "miller_loop_precomputed")
        return out

    def _table_pairs(self, coeffs, g1, g1_inf):
        g1 = _u8(g1, 64, "g1")
        n = g1.shape[0]
        coeffs = np.ascontiguousarray(coeffs, dtype=np.uint8).reshape(-1, 87 * 192)
        if coeffs.shape[0] != n:
            raise ValueError("one table per pair: %d tables for %d G1 points" % (coeffs.shape[0], n))
        g1_inf = None if g1_inf is None else np.ascontiguousarray(g1_inf, dtype=np.uint8).reshape(n)
        return coeffs, g1, g1_inf, n

    def miller_loop_precomputed_batch(self, coeffs, g1, g1_inf=None) -> np.ndarray:
        """G2PreComputed::miller_loop with one canonical table per pair: coeffs (n, 16704), g1 (n, 64) -> (n, 384)."""
        coeffs, g1, g1_inf, n = self._table_pairs(coeffs, g1, g1_inf)
        out = np.empty((n, 384), dtype=np.uint8)
        self._ck(self._lib.sylow_b200_miller_loop_precomputed_batch(self._h, _ptr(coeffs), _ptr(g1), _ptr(g1_inf), n,
                                                                    _ptr(out)), "miller_loop_precomputed_batch")
        return out

    def miller_product_precomputed(self, coeffs, g1, g1_inf=None) -> np.ndarray:
        """glued_miller_loop(&[G2PreComputed], &[G1Affine]): one canonical table per pair; infinite G1 pairs skipped."""
        coeffs, g1, g1_inf, n = self._table_pairs(coeffs, g1, g1_inf)
        out = np.empty(384, dtype=np.uint8)
        self._ck(self._lib.sylow_b200_miller_product_precomputed(self._h, _ptr(coeffs), _ptr(g1), _ptr(g1_inf), n,
                                                                 _ptr(out)), "miller_product_precomputed")
        return out

    def pairing_check_fixed_batch(self, g1, g2_var, coeffs_fixed, k_var: int, k_fixed: int, g1_inf=None,
                                  g2_var_inf=None) -> np.ndarray:
        g1 = _u8(g1, 64, "g1")
        k = k_var + k_fixed
        if k <= 0 or g1.shape[0] % k:
            raise ValueError("g1 rows (%d) not a multiple of k_var + k_fixed = %d" % (g1.shape[0], k))
        n_checks = g1.shape[0] // k
        g2_var = None if k_var == 0 else _u8(g2_var, 128, "g2_var")
        if k_var and g2_var.shape[0] != n_checks * k_var:
            raise ValueError("g2_var must have n_checks * k_var rows")
        coeffs_fixed = np.ascontiguousarray(coeffs_fixed, dtype=np.uint8).reshape(k_fixed, 87 * 192)
        g1_inf = None if g1_inf is None else np.ascontiguousarray(g1_inf, dtype=np.uint8).reshape(-1)
        g2_var_inf = None if g2_var_inf is None else np.ascontiguousarray(g2_var_inf, dtype=np.uint8).reshape(-1)
        ok = np.empty(n_checks, dtype=np.uint8)
        self._ck(self._lib.sylow_b200_pairing_check_fixed_batch(self._h, _ptr(g1), _ptr(g1_inf), _ptr(g2_var),
                                                                _ptr(g2_var_inf), k_var, _ptr(coeffs_fixed), k_fixed,
                                                                n_checks, _ptr(ok)), "pairing_check_fixed_batch")
        return ok.astype(bool)

    def tables_to_device(self, coeffs_fixed, d_tables):
        coeffs_fixed = np.ascontiguousarray(coeffs_fixed, dtype=np.uint8).reshape(-1, 87 * 192)
        self._ck(self._lib.sylow_b200_tables_to_device(self._h, _ptr(coeffs_fixed), coeffs_fixed.shape[0],
                                                       self._tp(d_tables), self._stream()), "tables_to_device")

    def pairing_check_fixed_batch_dev(self, d_g1, d_g2_var, d_tables, k_var, k_fixed, d_ok, d_g1_inf=None,
                                      d_g2_var_inf=None):
        n_checks = d_g1.shape[0] // (k_var + k_fixed)
        self._ck(self._lib.sylow_b200_pairing_check_fixed_batch_dev(self._h, self._tp(d_g1), self._tp(d_g1_inf),
                                                                    self._tp(d_g2_var), self._tp(d_g2_var_inf), k_var,
                                                                    self._tp(d_tables), k_fixed, n_checks,
                                                                    self._tp(d_ok), self._stream()),
                 "pairing_check_fixed_batch_dev")

    # ------------------------------------------------------------------ validation
    def g1_validate_batch(self, g1, g1_inf=None) -> np.ndarray:
        """int8 status per point: 0 ok, ERR_DECODE, ERR_NOT_ON_CURVE (G1Affine::new)."""
        g1 = _u8(g1, 64, "g1")
        n = g1.shape[0]
        g1_inf = None if g1_inf is None else np.ascontiguousarray(g1_inf, dtype=np.uint8).reshape(n)
        st = np.empty(n, dtype=np.int8)
        self._ck(self._lib.sylow_b200_g1_validate_batch(self._h, _ptr(g1), _ptr(g1_inf), n, _ptr(st)), "g1_validate_batch")
        return st

    def g2_validate_batch(self, g2, g2_inf=None) -> np.ndarray:
        """int8 status per point: 0 ok, ERR_DECODE, ERR_NOT_ON_CURVE, ERR_NOT_IN_SUBGROUP (G2Projective::new)."""
        g2 = _u8(g2, 128, "g2")
        n = g2.shape[0]
        g2_inf = None if g2_inf is None else np.ascontiguousarray(g2_inf, dtype=np.uint8).reshape(n)
        st = np.empty(n, dtype=np.int8)
        self._ck(self._lib.sylow_b200_g2_validate_batch(self._h, _ptr(g2), _ptr(g2_inf), n, _ptr(st)), "g2_validate_batch")
        return st

    # ------------------------------------------------------------------ big-endian codecs
    def _from_be(self, fn, width, be, eip_mode):
        be = _u8(be, width, "be")
        n = be.shape[0]
        out = np.empty((n, width), dtype=np.uint8)
        inf = np.empty(n, dtype=np.uint8)
        st = np.empty(n, dtype=np.int8)
        self._ck(fn(self._h, _ptr(be), n, int(bool(eip_mode)), _ptr(out), _ptr(inf), _ptr(st)), fn.__name__)
        return out, inf, st

    def g1_from_be_bytes_batch(self, be, eip_mode=False):
        return self._from_be(self._lib.sylow_b200_g1_from_be_bytes_batch, 64, be, eip_mode)

    def g2_from_be_bytes_batch(self, be, eip_mode=False):
        return self._from_be(self._lib.sylow_b200_g2_from_be_bytes_batch, 128, be, eip_mode)

    def _to_be(self, fn, width, pts, inf, scrubbed):
        pts = _u8(pts, width, "pts")
        n = pts.shape[0]
        inf = None if inf is None else np.ascontiguousarray(inf, dtype=np.uint8).reshape(n)
        out = np.empty((n, width), dtype=np.uint8)
        self._ck(fn(self._h, _ptr(pts), _ptr(inf), n, int(bool(scrubbed)), _ptr(out)), fn.__name__)
        return out

    def g1_to_be_bytes_batch(self, g1, g1_inf=None, scrubbed=False):
        return self._to_be(self._lib.sylow_b200_g1_to_be_bytes_batch, 64, g1, g1_inf, scrubbed)

    def g2_to_be_bytes_batch(self, g2, g2_inf=None, scrubbed=False):
        return self._to_be(self._lib.sylow_b200_g2_to_be_bytes_batch, 128, g2, g2_inf, scrubbed)

    def eip197_pairing_check_batch(self, inputs, pairs_per_check: int):
        """inputs: (n_checks, k*192) big-endian calldata; returns (ok bool array, int8 status array)."""
        k = int(pairs_per_check)
        inputs = np.ascontiguousarray(inputs, dtype=np.uint8)
        if inputs.ndim == 1:
            inputs = inputs.reshape(1, -1)
        if inputs.shape[1] != k * 192:
            raise ValueError("each input must be k*192 bytes")
        n = inputs.shape[0]
        ok = np.empty(n, dtype=np.uint8)
        st = np.empty(n, dtype=np.int8)
        self._ck(self._lib.sylow_b200_eip197_pairing_check_batch(self._h, _ptr(inputs), k, n, _ptr(ok), _ptr(st)),
                 "eip197_pairing_check_batch")
        return ok.astype(bool), st

    # ------------------------------------------------------------------ scalar multiplication
    def _mul(self, fn, width, pts, scalars, pts_inf):
        pts = _u8(pts, width, "pts")
        scalars = _u8(scalars, 32, "scalars")
        n = pts.shape[0]
        if scalars.shape[0] != n:
            raise ValueError("pts and scalars batch sizes differ")
        pts_inf = None if pts_inf is None else np.ascontiguousarray(pts_inf, dtype=np.uint8).reshape(n)
        out = np.empty((n, width), dtype=np.uint8)
        out_inf = np.empty(n, dtype=np.uint8)
        self._ck(fn(self._h, _ptr(pts), _ptr(pts_inf), _ptr(scalars), n, _ptr(out), _ptr(out_inf)), fn.__name__)
        return out, out_inf

    def g1_mul_batch(self, pts, scalars, pts_inf=None):
        return self._mul(self._lib.sylow_b200_g1_mul_batch, 64, pts, scalars, pts_inf)

    def g2_mul_batch(self, pts, scalars, pts_inf=None):
        return self._mul(self._lib.sylow_b200_g2_mul_batch, 128, pts, scalars, pts_inf)

    def gt_mul_batch(self, gt, scalars) -> np.ndarray:
        """`Gt * Fr`: gt[i]^scalars[i] (gt must be final-exponentiation outputs)."""
        gt = _u8(gt, 384, "gt")
        scalars = _u8(scalars, 32, "scalars")
        if gt.shape[0] != scalars.shape[0]:
            raise ValueError("gt and scalars batch sizes differ")
        out = np.empty_like(gt)
        self._ck(self._lib.sylow_b200_gt_mul_batch(self._h, _ptr(gt), _ptr(scalars), gt.shape[0], _ptr(out)), "gt_mul_batch")
        return out

    def g1_sum(self, pts, pts_inf=None):
        """sum of the points (signature aggregation): (64-byte affine point, infinity flag)."""
        pts = _u8(pts, 64, "pts")
        n = pts.shape[0]
        pts_inf = None if pts_inf is None else np.ascontiguousarray(pts_inf, dtype=np.uint8).reshape(n)
        out = np.empty(64, dtype=np.uint8)
        inf = np.zeros(1, dtype=np.uint8)
        self._ck(self._lib.sylow_b200_g1_sum(self._h, _ptr(pts), _ptr(pts_inf), n, _ptr(out), _ptr(inf)), "g1_sum")
        return out, int(inf[0])

    def g1_msm(self, pts, scalars, pts_inf=None):
        """sum_i scalars[i] * pts[i] (Lagrange-weighted aggregation)."""
        pts = _u8(pts, 64, "pts")
        scalars = _u8(scalars, 32, "scalars")
        n = pts.shape[0]
        pts_inf = None if pts_inf is None else np.ascontiguousarray(pts_inf, dtype=np.uint8).reshape(n)
        out = np.empty(64, dtype=np.uint8)
        inf = np.zeros(1, dtype=np.uint8)
        self._ck(self._lib.sylow_b200_g1_msm(self._h, _ptr(pts), _ptr(pts_inf), _ptr(scalars), n, _ptr(out), _ptr(inf)),
                 "g1_msm")
        return out, int(inf[0])

    def g1_msm_bucket(self, pts, scalars, pts_inf=None, window_bits: int = 0):
        """sum_i scalars[i] * pts[i] by the bucket (Pippenger) method; window_bits = 0 picks the window from n."""
        pts = _u8(pts, 64, "pts")
        scalars = _u8(scalars, 32, "scalars")
        n = pts.shape[0]
        pts_inf = None if pts_inf is None else np.ascontiguousarray(pts_inf, dtype=np.uint8).reshape(n)
        out = np.empty(64, dtype=np.uint8)
        inf = np.zeros(1, dtype=np.uint8)
        self._ck(self._lib.sylow_b200_g1_msm_bucket(self._h, _ptr(pts), _ptr(pts_inf), _ptr(scalars), n, int(window_bits),
                                                    _ptr(out), _ptr(inf)), "g1_msm_bucket")
        return out, int(inf[0])

    def lagrange_coefficients_batch(self, ids):
        """ids: (n_sets, t) participant ids -> (n_sets, t, 32) Lagrange coefficients at 0 in Fr (examples/dkg.rs:216-226)."""
        ids = np.ascontiguousarray(ids, dtype=np.uint64)
        if ids.ndim != 2:
            raise ValueError("ids must be (n_sets, t)")
        n_sets, t = ids.shape
        out = np.empty((n_sets, t, 32), dtype=np.uint8)
        self._ck(self._lib.sylow_b200_lagrange_coefficients_batch(self._h, _ptr(ids), n_sets, t, _ptr(out)),
                 "lagrange_coefficients_batch")
        return out

    def threshold_aggregate_batch(self, ids, sigs, sigs_inf=None):
        """ids (n_sets, t), sigs (n_sets, t, 64) partial signatures -> (n_sets, 64) aggregated signatures + flags:
        sum_i lambda_i * sig_i per set (examples/dkg.rs:190-206)."""
        ids = np.ascontiguousarray(ids, dtype=np.uint64)
        if ids.ndim != 2:
            raise ValueError("ids must be (n_sets, t)")
        n_sets, t = ids.shape
        sigs = np.ascontiguousarray(sigs, dtype=np.uint8)
        if sigs.shape != (n_sets, t, 64):
            raise ValueError("sigs must be (n_sets, t, 64)")
        sigs_inf = None if sigs_inf is None else np.ascontiguousarray(sigs_inf, dtype=np.uint8).reshape(n_sets * t)
        out = np.empty((n_sets, 64), dtype=np.uint8)
        inf = np.zeros(n_sets, dtype=np.uint8)
        self._ck(self._lib.sylow_b200_threshold_aggregate_batch(self._h, _ptr(ids), _ptr(sigs), _ptr(sigs_inf), n_sets, t,
                                                                _ptr(out), _ptr(inf)), "threshold_aggregate_batch")
        return out, inf

    # ------------------------------------------------------------------ hash / BLS
    @staticmethod
    def _flags(f, n):
        return None if f is None else np.ascontiguousarray(f, dtype=np.uint8).reshape(n)

    @staticmethod
    def _seed(weight_seed):
        """32 secret random bytes (batch verification) or None (the reference example's unweighted product)."""
        if weight_seed is None:
            return None
        seed = np.frombuffer(bytes(weight_seed), dtype=np.uint8).copy()
        if seed.size != 32:
            raise ValueError("weight_seed must be 32 bytes")
        return seed

    def verify_batch_same_signer(self, pk, msgs, sigs, dst: bytes = DST, pk_inf: bool = False, sigs_inf=None,
                                 weight_seed=None) -> bool:
        pk = np.ascontiguousarray(pk, dtype=np.uint8).reshape(128)
        sigs = _u8(sigs, 64, "sigs")
        buf, offs = self._msgs(msgs)
        n = offs.size - 1
        ok = ctypes.c_int(0)
        seed = self._seed(weight_seed)
        self._ck(self._lib.sylow_b200_verify_batch_same_signer(self._h, _ptr(pk), int(bool(pk_inf)), _ptr(buf), _ptr(offs),
                                                               _ptr(sigs), _ptr(self._flags(sigs_inf, n)), n, dst, len(dst),
                                                               _lib.HASH_KECCAK256, _ptr(seed), ctypes.byref(ok)),
                 "verify_batch_same_signer")
        return bool(ok.value)

    def batch_weights(self, weight_seed, first_index: int, n: int) -> np.ndarray:
        out = np.empty(n, dtype=np.uint64)
        self._ck(self._lib.sylow_b200_batch_weights(self._h, _ptr(self._seed(weight_seed)), int(first_index), n, _ptr(out)),
                 "batch_weights")
        return out

    @staticmethod
    def _msgs(msgs):
        if isinstance(msgs, tuple):
            buf, offs = msgs
            return np.ascontiguousarray(buf, dtype=np.uint8), np.ascontiguousarray(offs, dtype=np.uint64)
        return pack_messages(msgs)

    def hash_to_g1_batch(self, msgs, dst: bytes = DST, hash_id: int = _lib.HASH_KECCAK256):
        buf, offs = self._msgs(msgs)
        n = offs.size - 1
        out = np.empty((n, 64), dtype=np.uint8)
        out_inf = np.empty(n, dtype=np.uint8)
        self._ck(self._lib.sylow_b200_hash_to_g1_batch(self._h, _ptr(buf), _ptr(offs), n, dst, len(dst),
                                                       hash_id, _ptr(out), _ptr(out_inf)),
                 "hash_to_g1_batch")
        return out, out_inf

    def expand_message_batch(self, msgs, dst: bytes, len_in_bytes: int, hash_id: int = _lib.HASH_KECCAK256) -> np.ndarray:
        """Expander::expand_message (XMD) per message: (n, len_in_bytes) uint8."""
        buf, offs = self._msgs(msgs)
        n = offs.size - 1
        out = np.empty((n, int(len_in_bytes)), dtype=np.uint8)
        self._ck(self._lib.sylow_b200_expand_message_batch(self._h, _ptr(buf), _ptr(offs), n, dst, len(dst), hash_id,
                                                           int(len_in_bytes), _ptr(out)), "expand_message_batch")
        return out

    def hash_to_field_batch(self, msgs, dst: bytes = DST, hash_id: int = _lib.HASH_KECCAK256) -> np.ndarray:
        """Expander::hash_to_field(msg, 2, 48): (n, 64) = two canonical Fp per message."""
        buf, offs = self._msgs(msgs)
        n = offs.size - 1
        out = np.empty((n, 64), dtype=np.uint8)
        self._ck(self._lib.sylow_b200_hash_to_field_batch(self._h, _ptr(buf), _ptr(offs), n, dst, len(dst), hash_id,
                                                          _ptr(out)), "hash_to_field_batch")
        return out

    def sign_batch(self, sks, msgs, dst: bytes = DST, return_inf: bool = False):
        sks = _u8(sks, 32, "sks")
        buf, offs = self._msgs(msgs)
        n = offs.size - 1
        out = np.empty((n, 64), dtype=np.uint8)
        inf = np.zeros(n, dtype=np.uint8)
        self._ck(self._lib.sylow_b200_sign_batch(self._h, _ptr(sks), _ptr(buf), _ptr(offs), n, dst, len(dst),
                                                 _lib.HASH_KECCAK256, _ptr(out), _ptr(inf)), "sign_batch")
        return (out, inf) if return_inf else out

    def verify_each(self, pks, msgs, sigs, dst: bytes = DST, pks_inf=None, sigs_inf=None) -> np.ndarray:
        pks = _u8(pks, 128, "pks")
        sigs = _u8(sigs, 64, "sigs")
        buf, offs = self._msgs(msgs)
        n = offs.size - 1
        ok = np.empty(n, dtype=np.uint8)
        self._ck(self._lib.sylow_b200_verify_each(self._h, _ptr(pks), _ptr(self._flags(pks_inf, n)), _ptr(buf), _ptr(offs),
                                                  _ptr(sigs), _ptr(self._flags(sigs_inf, n)), n, dst, len(dst),
                                                  _lib.HASH_KECCAK256, _ptr(ok)), "verify_each")
        return ok.astype(bool)

    def verify_batch_partial(self, pks, msgs, sigs, dst: bytes = DST, pks_inf=None, sigs_inf=None, weight_seed=None,
                             first_index: int = 0) -> np.ndarray:
        pks = _u8(pks, 128, "pks")
        sigs = _u8(sigs, 64, "sigs")
        buf, offs = self._msgs(msgs)
        n = offs.size - 1
        out = np.empty(384, dtype=np.uint8)
        seed = self._seed(weight_seed)
        self._ck(self._lib.sylow_b200_verify_batch_partial(self._h, _ptr(pks), _ptr(self._flags(pks_inf, n)), _ptr(buf),
                                                           _ptr(offs), _ptr(sigs), _ptr(self._flags(sigs_inf, n)), n,
                                                           dst, len(dst), _lib.HASH_KECCAK256, _ptr(seed),
                                                           int(first_index), _ptr(out)),
                 "verify_batch_partial")
        return out

    def verify_batch_finish(self, partials) -> bool:
        partials = _u8(partials, 384, "partials")
        ok = ctypes.c_int(0)
        self._ck(self._lib.sylow_b200_verify_batch_finish(self._h, _ptr(partials), partials.shape[0],
                                                          ctypes.byref(ok)), "verify_batch_finish")
        return bool(ok.value)

    def verify_batch(self, pks, msgs, sigs, dst: bytes = DST, pks_inf=None, sigs_inf=None, weight_seed=None) -> bool:
        """weight_seed=None: the reference example's aggregate check (prod e(sig_i, G2) e(-H_i, pk_i) == 1);
        32 random bytes: batch verification with random 64-bit weights (sound per signature)."""
        pks = _u8(pks, 128, "pks")
        sigs = _u8(sigs, 64, "sigs")
        buf, offs = self._msgs(msgs)
        n = offs.size - 1
        ok = ctypes.c_int(0)
        seed = self._seed(weight_seed)
        self._ck(self._lib.sylow_b200_verify_batch(self._h, _ptr(pks), _ptr(self._flags(pks_inf, n)), _ptr(buf), _ptr(offs),
                                                   _ptr(sigs), _ptr(self._flags(sigs_inf, n)), n, dst, len(dst),
                                                   _lib.HASH_KECCAK256, _ptr(seed), ctypes.byref(ok)), "verify_batch")
        return bool(ok.value)

    # ------------------------------------------------------------------ diagnostics
    def fp_op_batch(self, op: int, a, b) -> np.ndarray:
        a = _u8(a, 32, "a")
        b = _u8(b, 32, "b")
        out = np.empty_like(a)
        self._ck(self._lib.sylow_b200_fp_op_batch(self._h, op, _ptr(a), _ptr(b), a.shape[0], _ptr(out)), "fp_op_batch")
        return out

    def fp12_op_batch(self, op: int, a, b) -> np.ndarray:
        a = _u8(a, 384, "a")
        b = _u8(b, 384, "b")
        out = np.empty_like(a)
        self._ck(self._lib.sylow_b200_fp12_op_batch(self._h, op, _ptr(a), _ptr(b), a.shape[0], _ptr(out)),
                 "fp12_op_batch")
        return out

    def imad_probe(self, variant: int, blocks: int, threads: int, iters: int) -> Tuple[float, float]:
        ms = ctypes.c_float(0)
        ops = ctypes.c_double(0)
        self._ck(self._lib.sylow_b200_imad_probe(self._h, variant, blocks, threads, iters, ctypes.byref(ms),
                                                 ctypes.byref(ops)), "imad_probe")
        return float(ms.value), float(ops.value)

    # ------------------------------------------------------------------ device-resident (torch) variants
    @staticmethod
    def _tp(t):
        return None if t is None else ctypes.c_void_p(t.data_ptr())

    @staticmethod
    def _stream():
        import torch

        h = torch.cuda.current_stream().cuda_stream
        # torch's default stream has handle 0, which the C ABI reads as "use the context's own stream";
        # name the legacy default stream explicitly (cudaStreamLegacy == 0x1) so CUDA events recorded
        # on torch's stream bracket the kernels.
        return ctypes.c_void_p(h if h else 1)

    def pairing_batch_dev(self, d_g1, d_g2, d_out, d_g1_inf=None, d_g2_inf=None):
        n = d_g1.shape[0]
        self._ck(self._lib.sylow_b200_pairing_batch_dev(self._h, self._tp(d_g1), self._tp(d_g1_inf), self._tp(d_g2),
                                                        self._tp(d_g2_inf), n, self._tp(d_out), self._stream()),
                 "pairing_batch_dev")

    def miller_loop_batch_dev(self, d_g1, d_g2, d_out, d_g1_inf=None, d_g2_inf=None):
        n = d_g1.shape[0]
        self._ck(self._lib.sylow_b200_miller_loop_batch_dev(self._h, self._tp(d_g1), self._tp(d_g1_inf),
                                                            self._tp(d_g2), self._tp(d_g2_inf), n, self._tp(d_out),
                                                            self._stream()), "miller_loop_batch_dev")

    def miller_product_dev(self, d_g1, d_g2, d_out, d_g1_inf=None, d_g2_inf=None):
        n = d_g1.shape[0]
        self._ck(self._lib.sylow_b200_miller_product_dev(self._h, self._tp(d_g1), self._tp(d_g1_inf), self._tp(d_g2),
                                                         self._tp(d_g2_inf), n, self._tp(d_out), self._stream()),
                 "miller_product_dev")

    def g2_precompute_dev(self, d_g2, d_tables):
        """Device-form tables of the (n, 128) points d_g2 into d_tables (n * 16704 bytes of device memory)."""
        self._ck(self._lib.sylow_b200_g2_precompute_dev(self._h, self._tp(d_g2), d_g2.shape[0], self._tp(d_tables),
                                                        self._stream()), "g2_precompute_dev")

    def miller_product_precomputed_dev(self, d_tables, d_g1, d_out, d_table_idx=None, d_g1_inf=None):
        """Miller product over resident device-form tables: pair i is d_g1[i] against table d_table_idx[i] (int32 or
        uint32 tensor; None: table i).  An index past the last table makes the product zero."""
        if d_table_idx is not None and d_table_idx.element_size() != 4:
            raise ValueError("d_table_idx must hold 32-bit indices")
        n_tables = d_tables.numel() // (87 * 192)
        self._ck(self._lib.sylow_b200_miller_product_precomputed_dev(self._h, self._tp(d_tables), n_tables,
                                                                     self._tp(d_table_idx), self._tp(d_g1),
                                                                     self._tp(d_g1_inf), d_g1.shape[0], self._tp(d_out),
                                                                     self._stream()),
                 "miller_product_precomputed_dev")

    def final_exp_batch_dev(self, d_f, d_out):
        self._ck(self._lib.sylow_b200_final_exp_batch_dev(self._h, self._tp(d_f), d_f.shape[0], self._tp(d_out),
                                                          self._stream()), "final_exp_batch_dev")

    def pairing_check_batch_dev(self, d_g1, d_g2, pairs_per_check, d_ok, d_g1_inf=None, d_g2_inf=None):
        n = d_g1.shape[0]
        self._ck(self._lib.sylow_b200_pairing_check_batch_dev(self._h, self._tp(d_g1), self._tp(d_g1_inf),
                                                              self._tp(d_g2), self._tp(d_g2_inf), pairs_per_check,
                                                              n // pairs_per_check, self._tp(d_ok), self._stream()),
                 "pairing_check_batch_dev")

    def g1_mul_batch_dev(self, d_pts, d_scalars, d_out, d_out_inf=None, d_pts_inf=None):
        self._ck(self._lib.sylow_b200_g1_mul_batch_dev(self._h, self._tp(d_pts), self._tp(d_pts_inf),
                                                       self._tp(d_scalars), d_pts.shape[0], self._tp(d_out),
                                                       self._tp(d_out_inf), self._stream()), "g1_mul_batch_dev")

    def g2_mul_batch_dev(self, d_pts, d_scalars, d_out, d_out_inf=None, d_pts_inf=None):
        self._ck(self._lib.sylow_b200_g2_mul_batch_dev(self._h, self._tp(d_pts), self._tp(d_pts_inf),
                                                       self._tp(d_scalars), d_pts.shape[0], self._tp(d_out),
                                                       self._tp(d_out_inf), self._stream()), "g2_mul_batch_dev")

    def hash_to_g1_batch_dev(self, d_msgs, d_offsets, d_out, d_out_inf=None, dst: bytes = DST):
        n = d_offsets.shape[0] - 1
        self._ck(self._lib.sylow_b200_hash_to_g1_batch_dev(self._h, self._tp(d_msgs), self._tp(d_offsets), n, dst,
                                                           len(dst), _lib.HASH_KECCAK256, self._tp(d_out),
                                                           self._tp(d_out_inf), self._stream()),
                 "hash_to_g1_batch_dev")

    def verify_batch_partial_dev(self, d_pks, d_msgs, d_offsets, d_sigs, d_f_out, dst: bytes = DST, d_pks_inf=None,
                                 d_sigs_inf=None, weight_seed=None, first_index: int = 0):
        n = d_offsets.shape[0] - 1
        seed = self._seed(weight_seed)
        self._ck(self._lib.sylow_b200_verify_batch_partial_dev(self._h, self._tp(d_pks), self._tp(d_pks_inf),
                                                               self._tp(d_msgs), self._tp(d_offsets), self._tp(d_sigs),
                                                               self._tp(d_sigs_inf), n, dst, len(dst),
                                                               _lib.HASH_KECCAK256, _ptr(seed), int(first_index),
                                                               self._tp(d_f_out), self._stream()),
                 "verify_batch_partial_dev")

    def hash_failed_dev(self) -> bool:
        """True if a hash-to-curve of the last hashing `_dev` call failed (synchronises the stream, clears the flag)."""
        f = ctypes.c_int(0)
        self._ck(self._lib.sylow_b200_hash_failed_dev(self._h, self._stream(), ctypes.byref(f)), "hash_failed_dev")
        return bool(f.value)

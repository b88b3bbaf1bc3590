"""Batched BN254 engine: Python host binding over the C ABI (include/sylow_b200.h).

Arrays are numpy uint8 in the C-ABI wire formats (see the header): G1 (n, 64), G2 (n, 128),
Fp12/Gt (n, 384), scalars (n, 32), infinity flags (n,) uint8.  The `_dev` methods take torch CUDA
uint8 tensors and enqueue on torch's current stream (used by bench.py for the HBM-resident number).
All compute happens in libsylow_b200.so on the GPU; nothing here computes field arithmetic.

Every host-buffer method checks each per-item array against the batch size it passes to the library and raises
ValueError before the call: the library reads n items from every such array.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence, Tuple

import numpy as np

from . import _lib

DST = b"WARLOCK-CHAOS-V01-CS01-SHA-256"  # reference src/lib.rs:90
TABLE = 87 * 192  # bytes of one canonical G2PreComputed table (87 line-coefficient triples)


def _rows(a, width: int, name: str, n: Optional[int] = None) -> np.ndarray:
    """a as contiguous uint8 rows of `width` bytes (a single row of that size is a batch of one); n: required rows."""
    a = np.ascontiguousarray(a, dtype=np.uint8)
    if a.ndim == 1 and a.size == width:
        a = a.reshape(1, width)
    if a.ndim != 2 or a.shape[1] != width:
        raise ValueError("%s must have shape (n, %d), got %s" % (name, width, a.shape))
    if n is not None and a.shape[0] != n:
        raise ValueError("%s must have %d rows, got %d" % (name, n, a.shape[0]))
    return a


def _flags(f, n: int, name: str) -> Optional[np.ndarray]:
    """Optional per-item uint8 flags (None: no item flagged); n of them when given."""
    if f is None:
        return None
    f = np.ascontiguousarray(f, dtype=np.uint8)
    if f.size != n:
        raise ValueError("%s must hold %d flags, got %d" % (name, n, f.size))
    return f.reshape(n)


def _tables(coeffs, n: Optional[int] = None) -> np.ndarray:
    """Canonical G2PreComputed tables of any shape holding whole tables ((k, 87, 3, 64) too) as (k, TABLE) rows."""
    return _rows(np.ascontiguousarray(coeffs, dtype=np.uint8).reshape(-1, TABLE), TABLE, "coeffs", n)


def pack_messages(msgs: Sequence[bytes]) -> Tuple[np.ndarray, np.ndarray]:
    """Concatenate messages into (buffer uint8, offsets uint64 of length n+1)."""
    offs = np.zeros(len(msgs) + 1, dtype=np.uint64)
    if len(msgs):
        offs[1:] = np.cumsum([len(m) for m in msgs], dtype=np.uint64)
    buf = np.frombuffer(b"".join(msgs), dtype=np.uint8).copy() if int(offs[-1]) else np.zeros(0, dtype=np.uint8)
    return buf, offs


def _msgs(msgs) -> Tuple[np.ndarray, np.ndarray, int]:
    """(buffer, offsets, n) of a list of byte strings or of a packed (buffer, offsets) pair, whose buffer must hold the
    offsets[-1] bytes the library reads."""
    if isinstance(msgs, tuple):
        buf = np.ascontiguousarray(msgs[0], dtype=np.uint8)
        offs = np.ascontiguousarray(msgs[1], dtype=np.uint64).reshape(-1)
        if offs.size == 0:
            raise ValueError("offsets of n messages must hold n + 1 entries")
        if buf.size < int(offs[-1]):
            raise ValueError("message buffer holds %d bytes, offsets end at %d" % (buf.size, int(offs[-1])))
    else:
        buf, offs = pack_messages(msgs)
    return buf, offs, offs.size - 1


def _seed(weight_seed) -> Optional[np.ndarray]:
    """32 secret random bytes (batch verification) or None (the reference example's unweighted product)."""
    if weight_seed is None:
        return None
    seed = np.frombuffer(bytes(weight_seed), dtype=np.uint8).copy()
    if seed.size != 32:
        raise ValueError("weight_seed must be 32 bytes")
    return seed


def _offsets(offsets, n_items: Optional[int] = None, name: str = "offsets") -> np.ndarray:
    """n + 1 non-decreasing uint64 offsets of n checks; n_items: the items the arrays hold, which offsets[-1] must equal
    (the library reads offsets[-1] of them)."""
    offs = np.ascontiguousarray(offsets, dtype=np.uint64).reshape(-1)
    if offs.size == 0:
        raise ValueError("%s of n checks must hold n + 1 entries" % name)
    if (offs[1:] < offs[:-1]).any():
        raise ValueError("%s must not decrease" % name)
    if n_items is not None and int(offs[-1]) != n_items:
        raise ValueError("%s end at %d, the arrays hold %d pairs" % (name, int(offs[-1]), n_items))
    return offs


def _pairs(g1, g2, g1_inf, g2_inf):
    """(g1, g1_inf, g2, g2_inf, n) of n pairs, in the argument order of the pairing entry points."""
    g1 = _rows(g1, 64, "g1")
    n = g1.shape[0]
    return g1, _flags(g1_inf, n, "g1_inf"), _rows(g2, 128, "g2", n), _flags(g2_inf, n, "g2_inf"), n


def _table_pairs(coeffs, g1, g1_inf):
    """(coeffs, g1, g1_inf, n) of n pairs with one table each."""
    g1 = _rows(g1, 64, "g1")
    n = g1.shape[0]
    return _tables(coeffs, n), g1, _flags(g1_inf, n, "g1_inf"), n


def _signed(pks, msgs, sigs, pks_inf, sigs_inf):
    """(pks, pks_inf, buf, offs, sigs, sigs_inf, n) of n (key, message, signature) triples, in the argument order of
    the verify entry points."""
    buf, offs, n = _msgs(msgs)
    return (_rows(pks, 128, "pks", n), _flags(pks_inf, n, "pks_inf"), buf, offs, _rows(sigs, 64, "sigs", n),
            _flags(sigs_inf, n, "sigs_inf"), n)


def groth16_vk_dev_bytes(n_public: int) -> int:
    """SYLOW_B200_GROTH16_VK_DEV_BYTES: bytes of a prepared Groth16 key in device memory."""
    return 3 * TABLE + 128 + int(n_public) * 32 * 128 * 64


def _vk(vk, n_public: int) -> np.ndarray:
    """A Groth16 verifying key, alpha || beta || gamma || delta || IC_0 .. IC_n_public, as one row of bytes."""
    if int(n_public) < 0:
        raise ValueError("n_public must be >= 0")
    return _rows(np.ascontiguousarray(vk, dtype=np.uint8).reshape(-1), 448 + 64 * (int(n_public) + 1), "vk", 1)


def _groth16(vk, proofs, inputs, n_public: int, proofs_inf):
    """(vk, n_public, proofs, proofs_inf, inputs, n) in the argument order of the Groth16 host entry points."""
    l = int(n_public)
    proofs = _rows(proofs, 256, "proofs")
    n = proofs.shape[0]
    if l:
        inputs = np.ascontiguousarray(inputs, dtype=np.uint8)
        if inputs.size != n * 32 * l:
            raise ValueError("inputs must hold %d x %d x 32 bytes, got %d" % (n, l, inputs.size))
        inputs = inputs.reshape(n, 32 * l)
    else:
        inputs = None
    return _vk(vk, l), l, proofs, _flags(proofs_inf, 3 * n, "proofs_inf"), inputs, n


def _ids(ids) -> np.ndarray:
    ids = np.ascontiguousarray(ids, dtype=np.uint64)
    if ids.ndim != 2:
        raise ValueError("ids must be (n_sets, t)")
    return ids


def _arg(a):
    """numpy arrays and torch tensors as the address of their data; everything else as it is."""
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(ctypes.c_void_p)
    if hasattr(a, "data_ptr"):
        return ctypes.c_void_p(a.data_ptr())
    return a


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

    def _call(self, symbol: str, *args):
        """symbol(context, *args) with arrays and tensors passed by address; a non-zero status raises."""
        st = getattr(self._lib, symbol)(self._h, *[_arg(a) for a in args])
        if st != 0:
            raise _lib.SylowB200Error(st, symbol, self._lib.sylow_b200_last_cuda_error(self._h))

    @property
    def launch_count(self) -> int:
        return int(self._lib.sylow_b200_launch_count(self._h))

    # ------------------------------------------------------------------ pairing
    def pairing_batch(self, g1, g2, g1_inf=None, g2_inf=None) -> np.ndarray:
        args = _pairs(g1, g2, g1_inf, g2_inf)
        out = np.empty((args[-1], 384), dtype=np.uint8)
        self._call("sylow_b200_pairing_batch", *args, out)
        return out

    def miller_loop_batch(self, g1, g2, g1_inf=None, g2_inf=None) -> np.ndarray:
        args = _pairs(g1, g2, g1_inf, g2_inf)
        out = np.empty((args[-1], 384), dtype=np.uint8)
        self._call("sylow_b200_miller_loop_batch", *args, out)
        return out

    def miller_product(self, g1, g2, g1_inf=None, g2_inf=None) -> np.ndarray:
        out = np.empty(384, dtype=np.uint8)
        self._call("sylow_b200_miller_product", *_pairs(g1, g2, g1_inf, g2_inf), out)
        return out

    def final_exp_batch(self, f) -> np.ndarray:
        f = _rows(f, 384, "f")
        out = np.empty_like(f)
        self._call("sylow_b200_final_exp_batch", f, f.shape[0], out)
        return out

    def fp12_product(self, f) -> np.ndarray:
        f = _rows(f, 384, "f")
        out = np.empty(384, dtype=np.uint8)
        self._call("sylow_b200_fp12_product", f, f.shape[0], out)
        return out

    def pairing_check_batch(self, g1, g2, pairs_per_check: int, g1_inf=None, g2_inf=None) -> np.ndarray:
        g1, g1_inf, g2, g2_inf, n = _pairs(g1, g2, g1_inf, g2_inf)
        k = int(pairs_per_check)
        if k <= 0 or n % k:
            raise ValueError("batch of %d pairs is not a multiple of pairs_per_check=%d" % (n, k))
        ok = np.empty(n // k, dtype=np.uint8)
        self._call("sylow_b200_pairing_check_batch", g1, g1_inf, g2, g2_inf, k, n // k, ok)
        return ok.astype(bool)

    def pairing_check_ragged_batch(self, g1, g2, offsets, g1_inf=None, g2_inf=None) -> np.ndarray:
        """Check c multiplies the pairs [offsets[c], offsets[c + 1]): n_checks + 1 non-decreasing offsets ending at the
        number of pairs (offsets[0] may be above 0: the pairs before it are not read); an empty check holds."""
        g1, g1_inf, g2, g2_inf, n = _pairs(g1, g2, g1_inf, g2_inf)
        offs = _offsets(offsets, n)
        ok = np.empty(offs.size - 1, dtype=np.uint8)
        self._call("sylow_b200_pairing_check_ragged_batch", g1, g1_inf, g2, g2_inf, offs, offs.size - 1, ok)
        return ok.astype(bool)

    # ------------------------------------------------------------------ precomputed G2
    def g2_precompute(self, g2) -> np.ndarray:
        """G2Affine::precompute: (n, 87, 3, 64) uint8 canonical line coefficients."""
        g2 = _rows(g2, 128, "g2")
        out = np.empty((g2.shape[0], TABLE), dtype=np.uint8)
        self._call("sylow_b200_g2_precompute", g2, g2.shape[0], out)
        return out

    def miller_loop_precomputed(self, coeffs, g1, g1_inf=None) -> np.ndarray:
        g1 = _rows(g1, 64, "g1")
        n = g1.shape[0]
        out = np.empty((n, 384), dtype=np.uint8)
        self._call("sylow_b200_miller_loop_precomputed", _tables(coeffs, 1), g1, _flags(g1_inf, n, "g1_inf"), n, out)
        return out

    def miller_loop_precomputed_batch(self, coeffs, g1, g1_inf=None) -> np.ndarray:
        """G2PreComputed::miller_loop with one canonical table per pair: coeffs (n, 16704), g1 (n, 64) -> (n, 384)."""
        args = _table_pairs(coeffs, g1, g1_inf)
        out = np.empty((args[-1], 384), dtype=np.uint8)
        self._call("sylow_b200_miller_loop_precomputed_batch", *args, out)
        return out

    def miller_product_precomputed(self, coeffs, g1, g1_inf=None) -> np.ndarray:
        """glued_miller_loop(&[G2PreComputed], &[G1Affine]): one canonical table per pair; infinite G1 pairs skipped."""
        out = np.empty(384, dtype=np.uint8)
        self._call("sylow_b200_miller_product_precomputed", *_table_pairs(coeffs, g1, g1_inf), out)
        return out

    def pairing_check_fixed_batch(self, g1, g2_var, coeffs_fixed, k_var: int, k_fixed: int, g1_inf=None,
                                  g2_var_inf=None) -> np.ndarray:
        g1 = _rows(g1, 64, "g1")
        k = k_var + k_fixed
        if k <= 0 or g1.shape[0] % k:
            raise ValueError("g1 rows (%d) not a multiple of k_var + k_fixed = %d" % (g1.shape[0], k))
        n_checks = g1.shape[0] // k
        g2_var = None if k_var == 0 else _rows(g2_var, 128, "g2_var", n_checks * k_var)
        ok = np.empty(n_checks, dtype=np.uint8)
        self._call("sylow_b200_pairing_check_fixed_batch", g1, _flags(g1_inf, g1.shape[0], "g1_inf"), g2_var,
                   _flags(g2_var_inf, n_checks * k_var, "g2_var_inf"), k_var, _tables(coeffs_fixed, k_fixed), k_fixed,
                   n_checks, ok)
        return ok.astype(bool)

    def tables_to_device(self, coeffs_fixed, d_tables):
        coeffs_fixed = _tables(coeffs_fixed)
        self._call("sylow_b200_tables_to_device", coeffs_fixed, coeffs_fixed.shape[0], d_tables, self._stream())

    def pairing_check_fixed_batch_dev(self, d_g1, d_g2_var, d_tables, k_var, k_fixed, d_ok, d_g1_inf=None,
                                      d_g2_var_inf=None):
        n_checks = d_g1.shape[0] // (k_var + k_fixed)
        self._call("sylow_b200_pairing_check_fixed_batch_dev", d_g1, d_g1_inf, d_g2_var, d_g2_var_inf, k_var, d_tables,
                   k_fixed, n_checks, d_ok, self._stream())

    # ------------------------------------------------------------------ validation
    def g1_validate_batch(self, g1, g1_inf=None) -> np.ndarray:
        """int8 status per point: 0 ok, ERR_DECODE, ERR_NOT_ON_CURVE (G1Affine::new)."""
        g1 = _rows(g1, 64, "g1")
        n = g1.shape[0]
        st = np.empty(n, dtype=np.int8)
        self._call("sylow_b200_g1_validate_batch", g1, _flags(g1_inf, n, "g1_inf"), n, st)
        return st

    def g2_validate_batch(self, g2, g2_inf=None) -> np.ndarray:
        """int8 status per point: 0 ok, ERR_DECODE, ERR_NOT_ON_CURVE, ERR_NOT_IN_SUBGROUP (G2Projective::new)."""
        g2 = _rows(g2, 128, "g2")
        n = g2.shape[0]
        st = np.empty(n, dtype=np.int8)
        self._call("sylow_b200_g2_validate_batch", g2, _flags(g2_inf, n, "g2_inf"), n, st)
        return st

    # ------------------------------------------------------------------ big-endian codecs
    def _from_be(self, symbol, width, be, eip_mode):
        be = _rows(be, width, "be")
        n = be.shape[0]
        out = np.empty((n, width), dtype=np.uint8)
        inf = np.empty(n, dtype=np.uint8)
        st = np.empty(n, dtype=np.int8)
        self._call(symbol, be, n, int(bool(eip_mode)), out, inf, st)
        return out, inf, st

    def g1_from_be_bytes_batch(self, be, eip_mode=False):
        return self._from_be("sylow_b200_g1_from_be_bytes_batch", 64, be, eip_mode)

    def g2_from_be_bytes_batch(self, be, eip_mode=False):
        return self._from_be("sylow_b200_g2_from_be_bytes_batch", 128, be, eip_mode)

    def _to_be(self, symbol, width, pts, inf, scrubbed):
        pts = _rows(pts, width, "pts")
        n = pts.shape[0]
        out = np.empty((n, width), dtype=np.uint8)
        self._call(symbol, pts, _flags(inf, n, "inf"), n, int(bool(scrubbed)), out)
        return out

    def g1_to_be_bytes_batch(self, g1, g1_inf=None, scrubbed=False):
        return self._to_be("sylow_b200_g1_to_be_bytes_batch", 64, g1, g1_inf, scrubbed)

    def g2_to_be_bytes_batch(self, g2, g2_inf=None, scrubbed=False):
        return self._to_be("sylow_b200_g2_to_be_bytes_batch", 128, g2, g2_inf, scrubbed)

    def eip197_pairing_check_batch(self, inputs, pairs_per_check: int):
        """inputs: (n_checks, k*192) big-endian calldata; returns (ok bool array, int8 status array)."""
        k = int(pairs_per_check)
        inputs = _rows(inputs, k * 192, "inputs")
        n = inputs.shape[0]
        ok = np.empty(n, dtype=np.uint8)
        st = np.empty(n, dtype=np.int8)
        self._call("sylow_b200_eip197_pairing_check_batch", inputs, k, n, ok, st)
        return ok.astype(bool), st

    def eip197_pairing_check_ragged_batch(self, inputs):
        """EIP-197 ecPairing bodies over inputs of any length: a list of bytes (or a packed (buffer, offsets) pair, as
        for messages); returns (ok bool array, int8 status array).  A length that is not a multiple of 192 gives
        ok = False and status ERR_ARG; an empty input succeeds."""
        buf, offs, n = _msgs(inputs)
        offs = _offsets(offs)
        ok = np.empty(n, dtype=np.uint8)
        st = np.empty(n, dtype=np.int8)
        self._call("sylow_b200_eip197_pairing_check_ragged_batch", buf, offs, n, ok, st)
        return ok.astype(bool), st

    def _eip196(self, symbol, width, inputs):
        inputs = _rows(inputs, width, "inputs")
        n = inputs.shape[0]
        out = np.empty((n, 64), dtype=np.uint8)
        st = np.empty(n, dtype=np.int8)
        self._call(symbol, inputs, n, out, st)
        return out, st

    def eip196_add_batch(self, inputs):
        """EIP-196 ecAdd bodies: inputs (n, 128) big-endian x1 || y1 || x2 || y2 (the caller pads or truncates calldata
        to 128 bytes); returns (out (n, 64) big-endian, all zero for infinity and for a failed input; int8 status: 0,
        ERR_DECODE or ERR_NOT_ON_CURVE)."""
        return self._eip196("sylow_b200_eip196_add_batch", 128, inputs)

    def eip196_mul_batch(self, inputs):
        """EIP-196 ecMul bodies: inputs (n, 96) big-endian x || y || s, s any 256-bit integer; returns like
        eip196_add_batch."""
        return self._eip196("sylow_b200_eip196_mul_batch", 96, inputs)

    # ------------------------------------------------------------------ group law
    def _add(self, symbol, width, a, b, a_inf, b_inf, subtract):
        a = _rows(a, width, "a")
        n = a.shape[0]
        out = np.empty((n, width), dtype=np.uint8)
        out_inf = np.empty(n, dtype=np.uint8)
        self._call(symbol, a, _flags(a_inf, n, "a_inf"), _rows(b, width, "b", n), _flags(b_inf, n, "b_inf"), n,
                   int(bool(subtract)), out, out_inf)
        return out, out_inf

    def g1_add_batch(self, a, b, a_inf=None, b_inf=None, subtract=False):
        """a[i] + b[i] (a[i] - b[i] with subtract) in G1, affine: (out (n, 64), out_inf (n,))."""
        return self._add("sylow_b200_g1_add_batch", 64, a, b, a_inf, b_inf, subtract)

    def g2_add_batch(self, a, b, a_inf=None, b_inf=None, subtract=False):
        """a[i] + b[i] (a[i] - b[i] with subtract) in G2, affine: (out (n, 128), out_inf (n,))."""
        return self._add("sylow_b200_g2_add_batch", 128, a, b, a_inf, b_inf, subtract)

    # ------------------------------------------------------------------ scalar multiplication
    def _mul(self, symbol, width, pts, scalars, pts_inf):
        pts = _rows(pts, width, "pts")
        n = pts.shape[0]
        out = np.empty((n, width), dtype=np.uint8)
        out_inf = np.empty(n, dtype=np.uint8)
        self._call(symbol, pts, _flags(pts_inf, n, "pts_inf"), _rows(scalars, 32, "scalars", n), n, out, out_inf)
        return out, out_inf

    def g1_mul_batch(self, pts, scalars, pts_inf=None):
        return self._mul("sylow_b200_g1_mul_batch", 64, pts, scalars, pts_inf)

    def g2_mul_batch(self, pts, scalars, pts_inf=None):
        return self._mul("sylow_b200_g2_mul_batch", 128, pts, scalars, pts_inf)

    def _mul_generator(self, symbol, width, scalars):
        scalars = _rows(scalars, 32, "scalars")
        n = scalars.shape[0]
        out = np.empty((n, width), dtype=np.uint8)
        out_inf = np.empty(n, dtype=np.uint8)
        self._call(symbol, scalars, n, out, out_inf)
        return out, out_inf

    def g1_mul_generator_batch(self, scalars):
        """scalars[i] * G1 generator: the values of g1_mul_batch on the repeated generator, from a fixed-base table."""
        return self._mul_generator("sylow_b200_g1_mul_generator_batch", 64, scalars)

    def g2_mul_generator_batch(self, scalars):
        """scalars[i] * G2 generator (KeyPair::generate's public key), like g1_mul_generator_batch."""
        return self._mul_generator("sylow_b200_g2_mul_generator_batch", 128, scalars)

    def gt_mul_batch(self, gt, scalars) -> np.ndarray:
        """`Gt * Fr`: gt[i]^scalars[i] (gt must be final-exponentiation outputs)."""
        gt = _rows(gt, 384, "gt")
        out = np.empty_like(gt)
        self._call("sylow_b200_gt_mul_batch", gt, _rows(scalars, 32, "scalars", gt.shape[0]), gt.shape[0], out)
        return out

    def g1_sum(self, pts, pts_inf=None):
        """sum of the points (signature aggregation): (64-byte affine point, infinity flag)."""
        pts = _rows(pts, 64, "pts")
        n = pts.shape[0]
        out = np.empty(64, dtype=np.uint8)
        inf = np.zeros(1, dtype=np.uint8)
        self._call("sylow_b200_g1_sum", pts, _flags(pts_inf, n, "pts_inf"), n, out, inf)
        return out, int(inf[0])

    def g1_msm(self, pts, scalars, pts_inf=None):
        """sum_i scalars[i] * pts[i] (Lagrange-weighted aggregation)."""
        pts = _rows(pts, 64, "pts")
        n = pts.shape[0]
        out = np.empty(64, dtype=np.uint8)
        inf = np.zeros(1, dtype=np.uint8)
        self._call("sylow_b200_g1_msm", pts, _flags(pts_inf, n, "pts_inf"), _rows(scalars, 32, "scalars", n), n, out,
                   inf)
        return out, int(inf[0])

    def g1_msm_bucket(self, pts, scalars, pts_inf=None, window_bits: int = 0):
        """sum_i scalars[i] * pts[i] by the bucket (Pippenger) method; window_bits = 0 picks the window from n."""
        pts = _rows(pts, 64, "pts")
        n = pts.shape[0]
        out = np.empty(64, dtype=np.uint8)
        inf = np.zeros(1, dtype=np.uint8)
        self._call("sylow_b200_g1_msm_bucket", pts, _flags(pts_inf, n, "pts_inf"), _rows(scalars, 32, "scalars", n), n,
                   int(window_bits), out, inf)
        return out, int(inf[0])

    def lagrange_coefficients_batch(self, ids):
        """ids: (n_sets, t) participant ids -> (n_sets, t, 32) Lagrange coefficients at 0 in Fr (examples/dkg.rs:216-226)."""
        ids = _ids(ids)
        n_sets, t = ids.shape
        out = np.empty((n_sets, t, 32), dtype=np.uint8)
        self._call("sylow_b200_lagrange_coefficients_batch", ids, n_sets, t, out)
        return out

    def threshold_aggregate_batch(self, ids, sigs, sigs_inf=None):
        """ids (n_sets, t), sigs (n_sets, t, 64) partial signatures -> (n_sets, 64) aggregated signatures + flags:
        sum_i lambda_i * sig_i per set (examples/dkg.rs:190-206)."""
        ids = _ids(ids)
        n_sets, t = ids.shape
        sigs = np.ascontiguousarray(sigs, dtype=np.uint8)
        if sigs.shape != (n_sets, t, 64):
            raise ValueError("sigs must be (n_sets, t, 64)")
        out = np.empty((n_sets, 64), dtype=np.uint8)
        inf = np.zeros(n_sets, dtype=np.uint8)
        self._call("sylow_b200_threshold_aggregate_batch", ids, sigs, _flags(sigs_inf, n_sets * t, "sigs_inf"), n_sets,
                   t, out, inf)
        return out, inf

    # ------------------------------------------------------------------ hash / BLS
    def verify_batch_same_signer(self, pk, msgs, sigs, dst: bytes = DST, pk_inf: bool = False, sigs_inf=None,
                                 weight_seed=None) -> bool:
        pk = np.ascontiguousarray(pk, dtype=np.uint8).reshape(128)
        buf, offs, n = _msgs(msgs)
        ok = ctypes.c_int(0)
        self._call("sylow_b200_verify_batch_same_signer", pk, int(bool(pk_inf)), buf, offs, _rows(sigs, 64, "sigs", n),
                   _flags(sigs_inf, n, "sigs_inf"), n, dst, len(dst), _lib.HASH_KECCAK256, _seed(weight_seed),
                   ctypes.byref(ok))
        return bool(ok.value)

    def batch_weights(self, weight_seed, first_index: int, n: int) -> np.ndarray:
        out = np.empty(n, dtype=np.uint64)
        self._call("sylow_b200_batch_weights", _seed(weight_seed), int(first_index), n, out)
        return out

    def hash_to_g1_batch(self, msgs, dst: bytes = DST, hash_id: int = _lib.HASH_KECCAK256):
        buf, offs, n = _msgs(msgs)
        out = np.empty((n, 64), dtype=np.uint8)
        out_inf = np.empty(n, dtype=np.uint8)
        self._call("sylow_b200_hash_to_g1_batch", buf, offs, n, dst, len(dst), hash_id, out, out_inf)
        return out, out_inf

    def expand_message_batch(self, msgs, dst: bytes, len_in_bytes: int, hash_id: int = _lib.HASH_KECCAK256) -> np.ndarray:
        """Expander::expand_message (XMD) per message: (n, len_in_bytes) uint8."""
        buf, offs, n = _msgs(msgs)
        out = np.empty((n, int(len_in_bytes)), dtype=np.uint8)
        self._call("sylow_b200_expand_message_batch", buf, offs, n, dst, len(dst), hash_id, int(len_in_bytes), out)
        return out

    def hash_to_field_batch(self, msgs, dst: bytes = DST, hash_id: int = _lib.HASH_KECCAK256) -> np.ndarray:
        """Expander::hash_to_field(msg, 2, 48): (n, 64) = two canonical Fp per message."""
        buf, offs, n = _msgs(msgs)
        out = np.empty((n, 64), dtype=np.uint8)
        self._call("sylow_b200_hash_to_field_batch", buf, offs, n, dst, len(dst), hash_id, out)
        return out

    def sign_batch(self, sks, msgs, dst: bytes = DST, return_inf: bool = False):
        buf, offs, n = _msgs(msgs)
        out = np.empty((n, 64), dtype=np.uint8)
        inf = np.zeros(n, dtype=np.uint8)
        self._call("sylow_b200_sign_batch", _rows(sks, 32, "sks", n), buf, offs, n, dst, len(dst), _lib.HASH_KECCAK256,
                   out, inf)
        return (out, inf) if return_inf else out

    def verify_each(self, pks, msgs, sigs, dst: bytes = DST, pks_inf=None, sigs_inf=None) -> np.ndarray:
        args = _signed(pks, msgs, sigs, pks_inf, sigs_inf)
        ok = np.empty(args[-1], dtype=np.uint8)
        self._call("sylow_b200_verify_each", *args, dst, len(dst), _lib.HASH_KECCAK256, ok)
        return ok.astype(bool)

    def verify_batch_partial(self, pks, msgs, sigs, dst: bytes = DST, pks_inf=None, sigs_inf=None, weight_seed=None,
                             first_index: int = 0) -> np.ndarray:
        args = _signed(pks, msgs, sigs, pks_inf, sigs_inf)
        out = np.empty(384, dtype=np.uint8)
        self._call("sylow_b200_verify_batch_partial", *args, dst, len(dst), _lib.HASH_KECCAK256, _seed(weight_seed),
                   int(first_index), out)
        return out

    def verify_batch_finish(self, partials) -> bool:
        partials = _rows(partials, 384, "partials")
        ok = ctypes.c_int(0)
        self._call("sylow_b200_verify_batch_finish", partials, partials.shape[0], ctypes.byref(ok))
        return bool(ok.value)

    def verify_batch(self, pks, msgs, sigs, dst: bytes = DST, pks_inf=None, sigs_inf=None, weight_seed=None) -> bool:
        """weight_seed=None: the reference example's aggregate check (prod e(sig_i, G2) e(-H_i, pk_i) == 1);
        32 random bytes: batch verification with random 64-bit weights (sound per signature)."""
        args = _signed(pks, msgs, sigs, pks_inf, sigs_inf)
        ok = ctypes.c_int(0)
        self._call("sylow_b200_verify_batch", *args, dst, len(dst), _lib.HASH_KECCAK256, _seed(weight_seed),
                   ctypes.byref(ok))
        return bool(ok.value)

    # ------------------------------------------------------------------ Groth16
    def groth16_prepare_vk(self, vk, n_public: int, d_vk_out):
        """Validate the host key (448 + 64 (n_public + 1) bytes) and build its device form in d_vk_out, a torch CUDA
        uint8 tensor of groth16_vk_dev_bytes(n_public) bytes; an invalid key raises with its status."""
        self._call("sylow_b200_groth16_prepare_vk", _vk(vk, n_public), int(n_public), d_vk_out, self._stream())

    def groth16_verify_each(self, vk, proofs, inputs, n_public: int, proofs_inf=None) -> np.ndarray:
        """One verdict per proof: proofs (n, 256) A || B || C, inputs (n, n_public * 32) canonical Fr, proofs_inf
        (n, 3) flags or None.  Proof points are not validated (g1/g2_validate_batch first)."""
        args = _groth16(vk, proofs, inputs, n_public, proofs_inf)
        ok = np.empty(args[-1], dtype=np.uint8)
        self._call("sylow_b200_groth16_verify_each", *args, ok)
        return ok.astype(bool)

    def groth16_verify_batch(self, vk, proofs, inputs, n_public: int, weight_seed, proofs_inf=None) -> bool:
        """One verdict for the batch, with random 64-bit weights from weight_seed (32 secret random bytes)."""
        ok = ctypes.c_int(0)
        self._call("sylow_b200_groth16_verify_batch", *_groth16(vk, proofs, inputs, n_public, proofs_inf),
                   _seed(weight_seed), ctypes.byref(ok))
        return bool(ok.value)

    def groth16_verify_each_dev(self, d_vk, n_public: int, d_proofs, d_inputs, d_ok, d_proofs_inf=None):
        self._call("sylow_b200_groth16_verify_each_dev", d_vk, int(n_public), d_proofs, d_proofs_inf, d_inputs,
                   d_proofs.shape[0], d_ok, self._stream())

    def groth16_verify_batch_partial_dev(self, d_vk, n_public: int, d_proofs, d_inputs, d_f_out, weight_seed,
                                         first_index: int = 0, d_proofs_inf=None):
        """The 384-byte share of the proofs d_proofs (global index of the first: first_index); combine the shares with
        verify_batch_finish."""
        self._call("sylow_b200_groth16_verify_batch_partial_dev", d_vk, int(n_public), d_proofs, d_proofs_inf,
                   d_inputs, d_proofs.shape[0], _seed(weight_seed), int(first_index), d_f_out, self._stream())

    # ------------------------------------------------------------------ diagnostics
    def fp_op_batch(self, op: int, a, b) -> np.ndarray:
        a = _rows(a, 32, "a")
        out = np.empty_like(a)
        self._call("sylow_b200_fp_op_batch", op, a, _rows(b, 32, "b", a.shape[0]), a.shape[0], out)
        return out

    def fp12_op_batch(self, op: int, a, b) -> np.ndarray:
        a = _rows(a, 384, "a")
        out = np.empty_like(a)
        self._call("sylow_b200_fp12_op_batch", op, a, _rows(b, 384, "b", a.shape[0]), a.shape[0], out)
        return out

    def imad_probe(self, variant: int, blocks: int, threads: int, iters: int) -> Tuple[float, float]:
        ms = ctypes.c_float(0)
        ops = ctypes.c_double(0)
        self._call("sylow_b200_imad_probe", variant, blocks, threads, iters, ctypes.byref(ms), ctypes.byref(ops))
        return float(ms.value), float(ops.value)

    # ------------------------------------------------------------------ device-resident (torch) variants
    @staticmethod
    def _stream():
        import torch

        h = torch.cuda.current_stream().cuda_stream
        # torch's default stream has handle 0, which the C ABI reads as "use the context's own stream";
        # name the legacy default stream explicitly (cudaStreamLegacy == 0x1) so CUDA events recorded
        # on torch's stream bracket the kernels.
        return ctypes.c_void_p(h if h else 1)

    def pairing_batch_dev(self, d_g1, d_g2, d_out, d_g1_inf=None, d_g2_inf=None):
        self._call("sylow_b200_pairing_batch_dev", d_g1, d_g1_inf, d_g2, d_g2_inf, d_g1.shape[0], d_out, self._stream())

    def miller_loop_batch_dev(self, d_g1, d_g2, d_out, d_g1_inf=None, d_g2_inf=None):
        self._call("sylow_b200_miller_loop_batch_dev", d_g1, d_g1_inf, d_g2, d_g2_inf, d_g1.shape[0], d_out,
                   self._stream())

    def miller_product_dev(self, d_g1, d_g2, d_out, d_g1_inf=None, d_g2_inf=None):
        self._call("sylow_b200_miller_product_dev", d_g1, d_g1_inf, d_g2, d_g2_inf, d_g1.shape[0], d_out, self._stream())

    def g2_precompute_dev(self, d_g2, d_tables):
        """Device-form tables of the (n, 128) points d_g2 into d_tables (n * 16704 bytes of device memory)."""
        self._call("sylow_b200_g2_precompute_dev", d_g2, d_g2.shape[0], d_tables, self._stream())

    def miller_product_precomputed_dev(self, d_tables, d_g1, d_out, d_table_idx=None, d_g1_inf=None):
        """Miller product over resident device-form tables: pair i is d_g1[i] against table d_table_idx[i] (int32 or
        uint32 tensor; None: table i).  An index past the last table makes the product zero."""
        if d_table_idx is not None and d_table_idx.element_size() != 4:
            raise ValueError("d_table_idx must hold 32-bit indices")
        self._call("sylow_b200_miller_product_precomputed_dev", d_tables, d_tables.numel() // TABLE, d_table_idx, d_g1,
                   d_g1_inf, d_g1.shape[0], d_out, self._stream())

    def final_exp_batch_dev(self, d_f, d_out):
        self._call("sylow_b200_final_exp_batch_dev", d_f, d_f.shape[0], d_out, self._stream())

    def pairing_check_batch_dev(self, d_g1, d_g2, pairs_per_check, d_ok, d_g1_inf=None, d_g2_inf=None):
        self._call("sylow_b200_pairing_check_batch_dev", d_g1, d_g1_inf, d_g2, d_g2_inf, pairs_per_check,
                   d_g1.shape[0] // pairs_per_check, d_ok, self._stream())

    def pairing_check_ragged_batch_dev(self, d_g1, d_g2, offsets, d_ok, d_g1_inf=None, d_g2_inf=None):
        """pairing_check_ragged_batch on torch CUDA tensors (d_g1 (n, 64), d_g2 (n, 128), flags (n,), d_ok (n_checks,)
        uint8) with host (numpy) offsets; enqueued on torch's current stream."""
        n = d_g1.shape[0]
        offs = _offsets(offsets, n)
        for t, name, want in ((d_g2, "d_g2", n), (d_g1_inf, "d_g1_inf", n), (d_g2_inf, "d_g2_inf", n),
                              (d_ok, "d_ok", offs.size - 1)):
            if t is not None and t.shape[0] != want:
                raise ValueError("%s must have %d rows, got %d" % (name, want, t.shape[0]))
        self._call("sylow_b200_pairing_check_ragged_batch_dev", d_g1, d_g1_inf, d_g2, d_g2_inf, offs, offs.size - 1,
                   d_ok, self._stream())

    def g1_mul_batch_dev(self, d_pts, d_scalars, d_out, d_out_inf=None, d_pts_inf=None):
        self._call("sylow_b200_g1_mul_batch_dev", d_pts, d_pts_inf, d_scalars, d_pts.shape[0], d_out, d_out_inf,
                   self._stream())

    def g2_mul_batch_dev(self, d_pts, d_scalars, d_out, d_out_inf=None, d_pts_inf=None):
        self._call("sylow_b200_g2_mul_batch_dev", d_pts, d_pts_inf, d_scalars, d_pts.shape[0], d_out, d_out_inf,
                   self._stream())

    def g1_add_batch_dev(self, d_a, d_b, d_out, d_out_inf=None, d_a_inf=None, d_b_inf=None, subtract=False):
        self._call("sylow_b200_g1_add_batch_dev", d_a, d_a_inf, d_b, d_b_inf, d_a.shape[0], int(bool(subtract)), d_out,
                   d_out_inf, self._stream())

    def g2_add_batch_dev(self, d_a, d_b, d_out, d_out_inf=None, d_a_inf=None, d_b_inf=None, subtract=False):
        self._call("sylow_b200_g2_add_batch_dev", d_a, d_a_inf, d_b, d_b_inf, d_a.shape[0], int(bool(subtract)), d_out,
                   d_out_inf, self._stream())

    def g1_mul_generator_batch_dev(self, d_scalars, d_out, d_out_inf=None):
        self._call("sylow_b200_g1_mul_generator_batch_dev", d_scalars, d_scalars.shape[0], d_out, d_out_inf,
                   self._stream())

    def g2_mul_generator_batch_dev(self, d_scalars, d_out, d_out_inf=None):
        self._call("sylow_b200_g2_mul_generator_batch_dev", d_scalars, d_scalars.shape[0], d_out, d_out_inf,
                   self._stream())

    def hash_to_g1_batch_dev(self, d_msgs, d_offsets, d_out, d_out_inf=None, dst: bytes = DST):
        self._call("sylow_b200_hash_to_g1_batch_dev", d_msgs, d_offsets, d_offsets.shape[0] - 1, dst, len(dst),
                   _lib.HASH_KECCAK256, d_out, d_out_inf, self._stream())

    def verify_batch_partial_dev(self, d_pks, d_msgs, d_offsets, d_sigs, d_f_out, dst: bytes = DST, d_pks_inf=None,
                                 d_sigs_inf=None, weight_seed=None, first_index: int = 0):
        self._call("sylow_b200_verify_batch_partial_dev", d_pks, d_pks_inf, d_msgs, d_offsets, d_sigs, d_sigs_inf,
                   d_offsets.shape[0] - 1, dst, len(dst), _lib.HASH_KECCAK256, _seed(weight_seed), int(first_index),
                   d_f_out, self._stream())

    def hash_failed_dev(self) -> bool:
        """True if a hash-to-curve of the last hashing `_dev` call failed (synchronises the stream, clears the flag)."""
        f = ctypes.c_int(0)
        self._call("sylow_b200_hash_failed_dev", self._stream(), ctypes.byref(f))
        return bool(f.value)

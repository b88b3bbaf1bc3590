"""Object-level mirror of sylow's public API (reference src/lib.rs:71-84) on top of the batched engine.

Same names and argument meaning as the Rust crate - `Fp`, `Fr`, `G1Affine`, `G1Projective`, `G2Affine`,
`G2Projective`, `Gt`, `pairing`, `glued_pairing`, `KeyPair`, `sign`, `verify`, `XMDExpander` - so tests can be
written the way the reference's own tests are (src/pairing.rs:1038-1251).  Every operation is a batch of one on
the GPU engine; nothing here does field or curve arithmetic on the CPU.  For throughput use `Engine` directly
(`pairing_batch`, `verify_batch`, `g1_mul_batch`, ...): these wrappers exist for API parity, not speed.

Differences from the Rust types, all forced by the byte-level boundary (INTEGRATION.md section 5): points are kept
in affine form (`G1Projective` / `G2Projective` are aliases whose equality is point equality, like the
reference's cross-multiplied `ct_eq`), and field elements are Python ints holding the canonical residue.
"""
from __future__ import annotations

import secrets
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

from . import _lib
from .api import DST, Engine

P = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47  # Fp modulus, reference fp.rs:51-56
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001  # Fr modulus, reference fp.rs:541-542
SECURITY_BITS = 128  # reference lib.rs:94

_engine: Optional[Engine] = None


def engine() -> Engine:
    """The process-wide engine on cuda:0 (created on first use; raises if there is no CUDA device)."""
    global _engine
    if _engine is None:
        _engine = Engine(0)
    return _engine


class GroupError(Exception):
    """reference src/groups/group.rs:37-47"""


class NotOnCurve(GroupError):
    pass


class NotInSubgroup(GroupError):
    pass


class CannotHashToGroup(GroupError):
    pass


class DecodeError(GroupError):
    pass


_STATUS = {_lib.ERR_NOT_ON_CURVE: NotOnCurve, _lib.ERR_NOT_IN_SUBGROUP: NotInSubgroup, _lib.ERR_DECODE: DecodeError}


def _fp(x: int) -> bytes:
    return int(x).to_bytes(32, "little")


def _arr(b: bytes, width: int) -> np.ndarray:
    return np.frombuffer(b, dtype=np.uint8).reshape(-1, width).copy()


class Fp(int):
    """Canonical residue mod p.  `Fp(x)` reduces like `Fp::new` (fp.rs:199-201)."""

    def __new__(cls, v: int = 0):
        return super().__new__(cls, int(v) % P)


class Fr(int):
    def __new__(cls, v: int = 0):
        return super().__new__(cls, int(v) % R)

    @classmethod
    def rand(cls) -> "Fr":
        return cls(secrets.randbelow(R - 1) + 1)


@dataclass(frozen=True)
class G1Affine:
    x: int = 0
    y: int = 1
    infinity: bool = True

    @classmethod
    def new(cls, x: int, y: int) -> "G1Affine":
        """Checked constructor, G1Affine::new (g1.rs:111-132): raises NotOnCurve."""
        st = int(engine().g1_validate_batch(_arr(_fp(x % (1 << 256)) + _fp(y % (1 << 256)), 64))[0])
        if st:
            raise _STATUS.get(st, GroupError)()
        return cls(int(x), int(y), False)

    @classmethod
    def generator(cls) -> "G1Affine":
        return cls(1, 2, False)  # g1.rs:54-60

    @classmethod
    def zero(cls) -> "G1Affine":
        return cls(0, 1, True)

    def is_zero(self) -> bool:
        return self.infinity

    def _b(self) -> bytes:
        return _fp(self.x) + _fp(self.y)

    def __neg__(self) -> "G1Affine":
        return self if self.infinity else G1Affine(self.x, (-self.y) % P, False)

    def __mul__(self, k: int) -> "G1Affine":
        """`&G1Projective * &Fp` (group.rs:639-667) followed by the affine conversion."""
        out, inf = engine().g1_mul_batch(_arr(self._b(), 64), _arr(_fp(int(k) % (1 << 256)), 32), [int(self.infinity)])
        return _g1_from(out[0], inf[0])

    __rmul__ = __mul__

    def _add(self, other: "G1Affine", subtract: bool) -> "G1Affine":
        """`&G1Projective + / - &G1Projective` (group.rs:528-624) followed by the affine conversion."""
        out, inf = engine().g1_add_batch(_arr(self._b(), 64), _arr(other._b(), 64), [int(self.infinity)],
                                         [int(other.infinity)], subtract)
        return _g1_from(out[0], inf[0])

    def __add__(self, other: "G1Affine") -> "G1Affine":
        return self._add(other, False)

    def __sub__(self, other: "G1Affine") -> "G1Affine":
        return self._add(other, True)

    def to_be_bytes(self) -> bytes:
        return bytes(engine().g1_to_be_bytes_batch(_arr(self._b(), 64), [int(self.infinity)])[0])

    @classmethod
    def from_be_bytes(cls, b: bytes) -> "G1Affine":
        out, inf, st = engine().g1_from_be_bytes_batch(_arr(bytes(b), 64))
        if st[0]:
            raise _STATUS.get(int(st[0]), GroupError)()
        return _g1_from(out[0], inf[0])

    @classmethod
    def rand(cls) -> "G1Affine":
        return cls.generator() * Fr.rand()  # g1.rs:296-298

    @classmethod
    def hash_to_curve(cls, expander: "XMDExpander", msg: bytes) -> "G1Affine":
        out, inf = engine().hash_to_g1_batch([bytes(msg)], expander.dst, expander.hash_id)
        return _g1_from(out[0], inf[0])


def _g1_from(row, inf) -> G1Affine:
    b = bytes(row)
    return G1Affine(int.from_bytes(b[:32], "little"), int.from_bytes(b[32:], "little"), bool(inf))


@dataclass(frozen=True)
class G2Affine:
    x: tuple = (0, 0)
    y: tuple = (1, 0)
    infinity: bool = True

    @classmethod
    def new(cls, x: Sequence[int], y: Sequence[int]) -> "G2Affine":
        """Curve + subgroup check, G2Projective::new (g2.rs:460-525): raises NotOnCurve / NotInSubgroup."""
        raw = b"".join(_fp(c % (1 << 256)) for c in (x[0], x[1], y[0], y[1]))
        st = int(engine().g2_validate_batch(_arr(raw, 128))[0])
        if st:
            raise _STATUS.get(st, GroupError)()
        return cls((int(x[0]), int(x[1])), (int(y[0]), int(y[1])), False)

    @classmethod
    def generator(cls) -> "G2Affine":
        return cls((10857046999023057135944570762232829481370756359578518086990519993285655852781,
                    11559732032986387107991004021392285783925812861821192530917403151452391805634),
                   (8495653923123431417604973247489272438418190587263600148770280649306958101930,
                    4082367875863433681332203403145435568316851327593401208105741076214120093531), False)  # g2.rs:47-77

    @classmethod
    def zero(cls) -> "G2Affine":
        return cls((0, 0), (1, 0), True)

    def is_zero(self) -> bool:
        return self.infinity

    def _b(self) -> bytes:
        return _fp(self.x[0]) + _fp(self.x[1]) + _fp(self.y[0]) + _fp(self.y[1])

    def __neg__(self) -> "G2Affine":
        return self if self.infinity else G2Affine(self.x, ((-self.y[0]) % P, (-self.y[1]) % P), False)

    def __mul__(self, k: int) -> "G2Affine":
        out, inf = engine().g2_mul_batch(_arr(self._b(), 128), _arr(_fp(int(k) % (1 << 256)), 32), [int(self.infinity)])
        return _g2_from(out[0], inf[0])

    __rmul__ = __mul__

    def _add(self, other: "G2Affine", subtract: bool) -> "G2Affine":
        out, inf = engine().g2_add_batch(_arr(self._b(), 128), _arr(other._b(), 128), [int(self.infinity)],
                                         [int(other.infinity)], subtract)
        return _g2_from(out[0], inf[0])

    def __add__(self, other: "G2Affine") -> "G2Affine":
        return self._add(other, False)

    def __sub__(self, other: "G2Affine") -> "G2Affine":
        return self._add(other, True)

    @classmethod
    def rand(cls) -> "G2Affine":
        return cls.generator() * Fr.rand()

    def precompute(self) -> "G2PreComputed":
        """G2Affine::precompute (pairing.rs:676-708)."""
        return G2PreComputed(self, engine().g2_precompute(_arr(self._b(), 128))[0])


def _g2_from(row, inf) -> G2Affine:
    c = [int.from_bytes(bytes(row[32 * i: 32 * i + 32]), "little") for i in range(4)]
    return G2Affine((c[0], c[1]), (c[2], c[3]), bool(inf))


G1Projective = G1Affine  # points live in affine form on this side of the boundary
G2Projective = G2Affine


@dataclass(frozen=True)
class Gt:
    """Opaque Fp12 in tower order (12 canonical residues); `+` multiplies, `-x` conjugates, `* Fr` exponentiates
    (gt.rs:115-215)."""
    c: tuple

    @classmethod
    def identity(cls) -> "Gt":
        return cls((1,) + (0,) * 11)

    @classmethod
    def generator(cls) -> "Gt":
        return pairing(G1Affine.generator(), G2Affine.generator())

    def _b(self) -> bytes:
        return b"".join(_fp(x) for x in self.c)

    def __add__(self, o: "Gt") -> "Gt":
        return _gt_from(engine().fp12_op_batch(0, _arr(self._b(), 384), _arr(o._b(), 384))[0])

    def __neg__(self) -> "Gt":
        return Gt(self.c[:6] + tuple((-x) % P for x in self.c[6:]))  # unitary_inverse: negate the w-part

    def __mul__(self, k: int) -> "Gt":
        return _gt_from(engine().gt_mul_batch(_arr(self._b(), 384), _arr(_fp(int(k) % R), 32))[0])


def _gt_from(row) -> Gt:
    b = bytes(row)
    return Gt(tuple(int.from_bytes(b[32 * i: 32 * i + 32], "little") for i in range(12)))


@dataclass(frozen=True)
class MillerLoopResult:
    c: tuple

    def final_exponentiation(self) -> Gt:
        """pairing.rs:245-492"""
        b = b"".join(_fp(x) for x in self.c)
        return _gt_from(engine().final_exp_batch(_arr(b, 384))[0])


@dataclass(frozen=True)
class G2PreComputed:
    q: G2Affine
    coeffs: np.ndarray  # 87 x (3 Fp2) canonical, 16704 bytes

    def miller_loop(self, g1: G1Affine) -> MillerLoopResult:
        """pairing.rs:590-619"""
        row = engine().miller_loop_precomputed(self.coeffs, _arr(g1._b(), 64), [int(g1.infinity)])[0]
        return MillerLoopResult(_gt_from(row).c)


def pairing(p: G1Affine, q: G2Affine) -> Gt:
    """pairing.rs:870-893"""
    out = engine().pairing_batch(_arr(p._b(), 64), _arr(q._b(), 128), [int(p.infinity)], [int(q.infinity)])
    return _gt_from(out[0])


def glued_miller_loop(g2s: Sequence, g1s: Sequence[G1Affine]) -> MillerLoopResult:
    """pairing.rs:970-1022.  g2s holds `G2PreComputed` values (the reference's signature: the engine runs the loop
    from their tables) or `G2Affine` points (the engine fuses the precomputation).  Pairs with an infinite point are
    skipped."""
    n = min(len(g1s), len(g2s))
    if n == 0:
        return MillerLoopResult(Gt.identity().c)
    if all(isinstance(q, G2PreComputed) for q in g2s[:n]):
        coeffs = np.stack([np.ascontiguousarray(q.coeffs, dtype=np.uint8).reshape(87 * 192) for q in g2s[:n]])
        g1 = _arr(b"".join(p._b() for p in g1s[:n]), 64)
        skip = [int(p.infinity or q.q.infinity) for p, q in zip(g1s[:n], g2s[:n])]  # a table has no infinity form
        row = engine().miller_product_precomputed(coeffs, g1, skip)
        return MillerLoopResult(_gt_from(row).c)
    if any(isinstance(q, G2PreComputed) for q in g2s[:n]):
        raise TypeError("g2s mixes G2PreComputed and G2Affine values")
    g1 = _arr(b"".join(p._b() for p in g1s[:n]), 64)
    g2 = _arr(b"".join(q._b() for q in g2s[:n]), 128)
    row = engine().miller_product(g1, g2, [int(p.infinity) for p in g1s[:n]], [int(q.infinity) for q in g2s[:n]])
    return MillerLoopResult(_gt_from(row).c)


def glued_pairing(g1s: Sequence[G1Affine], g2s: Sequence[G2Affine]) -> Gt:
    """pairing.rs:1029-1037"""
    return glued_miller_loop(g2s, g1s).final_exponentiation()


class XMDExpander:
    """XMDExpander::<Keccak256 | Sha256>::new(dst, 128) (hasher.rs:137-172)."""

    def __init__(self, dst: bytes = DST, security_param: int = SECURITY_BITS, hash_name: str = "keccak256"):
        if security_param != SECURITY_BITS:
            raise ValueError("only k = 128 is supported (both digests have 256-bit output)")
        self.dst = bytes(dst)
        self.hash_id = {"keccak256": _lib.HASH_KECCAK256, "sha256": _lib.HASH_SHA256}[hash_name]

    def expand_message(self, msg: bytes, len_in_bytes: int) -> bytes:
        return bytes(engine().expand_message_batch([bytes(msg)], self.dst, len_in_bytes, self.hash_id)[0])

    def hash_to_field(self, msg: bytes, count: int = 2, size: int = 48) -> List[Fp]:
        if (count, size) != (2, 48):
            raise ValueError("hash_to_field is fixed to count = 2, L = 48 like the reference's callers (g1.rs:308-309)")
        row = bytes(engine().hash_to_field_batch([bytes(msg)], self.dst, self.hash_id)[0])
        return [Fp(int.from_bytes(row[:32], "little")), Fp(int.from_bytes(row[32:], "little"))]


class XOFExpander(XMDExpander):
    """XOFExpander::<Shake128>::new(dst, 128) (hasher.rs:258-330)."""

    def __init__(self, dst: bytes = DST, security_param: int = SECURITY_BITS):
        if security_param != SECURITY_BITS:
            raise ValueError("only k = 128 is supported")
        self.dst = bytes(dst)
        self.hash_id = _lib.HASH_SHAKE128


@dataclass(frozen=True)
class KeyPair:
    """lib.rs:105-137"""
    secret_key: int
    public_key: G2Affine

    @classmethod
    def generate(cls) -> "KeyPair":
        sk = int(Fr.rand())
        out, inf = engine().g2_mul_generator_batch(_arr(_fp(sk), 32))
        return cls(sk, _g2_from(out[0], inf[0]))


def sign(k: int, msg: bytes) -> G1Affine:
    """lib.rs:179-187"""
    out, inf = engine().sign_batch(_arr(_fp(int(k) % (1 << 256)), 32), [bytes(msg)], return_inf=True)
    return _g1_from(out[0], int(inf[0]))


def verify(pubkey: G2Affine, msg: bytes, sig: G1Affine) -> bool:
    """lib.rs:223-236"""
    # an infinite key or signature makes its side's pairing the identity (pairing.rs:876-886): the library applies
    # that rule itself from the infinity flags
    ok = engine().verify_each(_arr(pubkey._b(), 128), [bytes(msg)], _arr(sig._b(), 64),
                              pks_inf=[int(pubkey.infinity)], sigs_inf=[int(sig.infinity)])
    return bool(ok[0])

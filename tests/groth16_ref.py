"""Groth16 for the tests: the verifier equation over oracle.bn254_py, and keys and proofs made with the trapdoor.

Points are the oracle's affine tuples (x, y, infinity).  A key is (alpha, beta, gamma, delta, [IC_0 .. IC_l]), a proof
(A, B, C).  The trapdoor: every point is a known multiple of a generator, alpha = al G1, beta = be G2, ..., IC_i = u_i G1,
and a proof of inputs x with random a, b is A = a G1, B = b G2, C = c G1 with
c = (a b - al be - (u_0 + sum_i x_i u_i) ga) / de mod r, which makes e(A, B) e(-alpha, beta) e(-L, gamma) e(-C, delta) = 1.
"""
import random

from oracle import bn254_py as o
from tests import wire as w

R = o.R_ORDER


def g1_mul(k):
    return o.proj_to_affine(o.FpOps, o.proj_mul(o.FpOps, o.affine_to_proj(o.FpOps, o.G1_GEN), k % R))


def g2_mul(k):
    return o.proj_to_affine(o.Fp2Ops, o.proj_mul(o.Fp2Ops, o.affine_to_proj(o.Fp2Ops, o.G2_GEN), k % R))


def public_term(ic, inputs):
    """L = IC_0 + sum_i x_i IC_i (affine)"""
    acc = o.affine_to_proj(o.FpOps, ic[0])
    for x, p in zip(inputs, ic[1:]):
        acc = o.proj_add(o.FpOps, acc, o.proj_mul(o.FpOps, o.affine_to_proj(o.FpOps, p), x))
    return o.proj_to_affine(o.FpOps, acc)


def groth16_verify(vk, proof, inputs) -> bool:
    """Every input < r, then glued_pairing([A, -alpha, -L, -C], [B, beta, gamma, delta]) == 1; a pair with an infinite
    point contributes 1."""
    alpha, beta, gamma, delta, ic = vk
    if len(inputs) != len(ic) - 1 or not all(0 <= x < R for x in inputs):
        return False
    a, b, c = proof
    g1s = [a, o.g1_affine_neg(alpha), o.g1_affine_neg(public_term(ic, inputs)), o.g1_affine_neg(c)]
    g2s = [b, beta, gamma, delta]
    keep = [i for i in range(4) if not g1s[i][2] and not g2s[i][2]]
    return o.glued_pairing([g1s[i] for i in keep], [g2s[i] for i in keep]) == o.FP12_ONE


class Trapdoor:
    """Scalars of a key with l public inputs; proof scalars (a, b, c) for any inputs."""

    def __init__(self, l, seed):
        self.rng = random.Random(seed)
        self.al, self.be, self.ga, self.de = (self.rng.randrange(1, R) for _ in range(4))
        self.u = [self.rng.randrange(1, R) for _ in range(l + 1)]

    def l_scalar(self, inputs):
        return (self.u[0] + sum(x * u for x, u in zip(inputs, self.u[1:]))) % R

    def proof_scalars(self, inputs):
        a, b = self.rng.randrange(1, R), self.rng.randrange(1, R)
        c = (a * b - self.al * self.be - self.l_scalar(inputs) * self.ga) * pow(self.de, -1, R) % R
        return a, b, c

    def vk(self):
        """the key as oracle points"""
        return (g1_mul(self.al), g2_mul(self.be), g2_mul(self.ga), g2_mul(self.de), [g1_mul(u) for u in self.u])


def vk_bytes(vk) -> bytes:
    alpha, beta, gamma, delta, ic = vk
    return w.g1_b(alpha) + w.g2_b(beta) + w.g2_b(gamma) + w.g2_b(delta) + b"".join(w.g1_b(p) for p in ic)


def proof_bytes(proof) -> bytes:
    return w.g1_b(proof[0]) + w.g2_b(proof[1]) + w.g1_b(proof[2])

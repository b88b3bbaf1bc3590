"""CPU tier: the Groth16 reference of tests/groth16_ref.py, on which the GPU tests rest: trapdoor-made proofs verify,
tampered ones do not."""
import random

from oracle import bn254_py as o
from tests import groth16_ref as g

R = o.R_ORDER


def _proof(td, xs):
    a, b, c = td.proof_scalars(xs)
    return [g.g1_mul(a), g.g2_mul(b), g.g1_mul(c)]


def test_trapdoor_proofs_verify_and_tampered_ones_fail():
    rng = random.Random(5)
    td = g.Trapdoor(2, 11)
    vk = td.vk()
    xs = [rng.randrange(R), rng.randrange(R)]
    proof = _proof(td, xs)
    assert g.groth16_verify(vk, proof, xs)
    bad_c = list(proof)
    bad_c[2] = o.proj_to_affine(o.FpOps, o.proj_add(o.FpOps, o.affine_to_proj(o.FpOps, proof[2]),
                                                    o.affine_to_proj(o.FpOps, o.G1_GEN)))
    assert not g.groth16_verify(vk, bad_c, xs)                 # C + G1
    assert not g.groth16_verify(vk, proof, [xs[1], xs[0]])     # other inputs
    assert not g.groth16_verify(vk, proof, [xs[0] + R, xs[1]])  # the same residue, not canonical
    other = _proof(td, xs)
    assert g.groth16_verify(vk, other, xs)
    assert not g.groth16_verify(vk, [proof[0], other[1], proof[2]], xs)  # B of another proof


def test_no_public_inputs():
    td = g.Trapdoor(0, 12)
    vk = td.vk()
    assert g.groth16_verify(vk, _proof(td, []), [])
    assert not g.groth16_verify(vk, _proof(td, []), [1])  # wrong number of inputs

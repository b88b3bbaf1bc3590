"""sylow_b200: B200-native batched BN254 engine behind sylow's API for its data-parallel hot path
(batched optimal-ate pairings, G1/G2 scalar multiplication, BLS verify / batch-verify).

The compute lives in libsylow_b200.so (hand-written sm_100a CUDA, C ABI in include/sylow_b200.h).
"""
from .api import DST, Engine, groth16_vk_dev_bytes, pack_messages  # noqa: F401
from ._lib import SylowB200Error  # noqa: F401

__all__ = ["Engine", "DST", "groth16_vk_dev_bytes", "pack_messages", "SylowB200Error"]

"""CPU tier: the ragged pairing-check methods of Engine against a stub of libsylow_b200.so (the stub of
test_engine_marshalling.py, which records every call).  Well-formed arguments reach the C function once, by address;
decreasing offsets, offsets that do not end at the number of pairs and flag arrays of the wrong length raise ValueError
before any call: the library would read past the caller's arrays."""
import ctypes

import numpy as np
import pytest

from tests.test_engine_marshalling import G1, G2, INF, INF2, N, eng  # noqa: F401  (eng: the stubbed Engine fixture)


class Dev:
    """Stands in for a torch CUDA tensor of `rows` rows: its address and its shape are used."""

    def __init__(self, rows, addr=0x7000):
        self.shape = (rows,)
        self.addr = addr

    def data_ptr(self):
        return self.addr


OFFS = np.array([0, 1, 1, 4], np.uint64)  # checks of 1, 0 and 3 pairs over the N = 4 pairs


def _call(eng):
    assert len(eng._lib.calls) == 1, eng._lib.calls
    return eng._lib.calls[0]


def test_pairing_check_ragged_batch(eng):
    ok = eng.pairing_check_ragged_batch(G1, G2, OFFS, INF, INF2)
    name, args, _ = _call(eng)
    assert name == "sylow_b200_pairing_check_ragged_batch"
    assert [a.value for a in args[1:5]] == [G1.ctypes.data, INF.ctypes.data, G2.ctypes.data, INF2.ctypes.data]
    assert ctypes.string_at(args[5].value, 32) == OFFS.tobytes() and args[6] == 3
    assert ok.dtype == bool and ok.shape == (3,)


def test_pairing_check_ragged_batch_offsets_past_zero(eng):
    eng.pairing_check_ragged_batch(G1, G2, [2, 3, 4])  # pairs 0 and 1 are not read
    assert _call(eng)[1][6] == 2


def test_eip197_ragged(eng):
    inputs = [b"\x01" * 192, b"", b"\x02" * 191, b"\x03" * 384]
    ok, st = eng.eip197_pairing_check_ragged_batch(inputs)
    name, args, _ = _call(eng)
    assert name == "sylow_b200_eip197_pairing_check_ragged_batch"
    assert ctypes.string_at(args[1].value, 767) == b"".join(inputs)
    assert np.frombuffer(ctypes.string_at(args[2].value, 40), np.uint64).tolist() == [0, 192, 192, 383, 767]
    assert args[3] == 4 and ok.shape == (4,) and st.dtype == np.int8


def test_dev(eng):
    d_ok = Dev(3, 0x9000)
    eng.pairing_check_ragged_batch_dev(Dev(N), Dev(N, 0x8000), OFFS, d_ok)
    name, args, _ = _call(eng)
    assert name == "sylow_b200_pairing_check_ragged_batch_dev"
    assert args[1].value == 0x7000 and args[2] is None and args[3].value == 0x8000 and args[4] is None
    assert ctypes.string_at(args[5].value, 32) == OFFS.tobytes() and args[6] == 3 and args[7].value == 0x9000


BAD = [
    ("decreasing offsets", lambda e: e.pairing_check_ragged_batch(G1, G2, [0, 3, 2, 4])),
    ("short last offset", lambda e: e.pairing_check_ragged_batch(G1, G2, [0, 1, 3])),
    ("long last offset", lambda e: e.pairing_check_ragged_batch(G1, G2, [0, 1, 5])),
    ("no offsets", lambda e: e.pairing_check_ragged_batch(G1, G2, [])),
    ("short g1_inf", lambda e: e.pairing_check_ragged_batch(G1, G2, OFFS, INF[:3])),
    ("long g2_inf", lambda e: e.pairing_check_ragged_batch(G1, G2, OFFS, None, np.zeros(5, np.uint8))),
    ("short g2", lambda e: e.pairing_check_ragged_batch(G1, G2[:3], OFFS)),
    ("eip197 decreasing offsets", lambda e: e.eip197_pairing_check_ragged_batch(
        (np.zeros(384, np.uint8), np.array([0, 192, 0], np.uint64)))),
    ("eip197 short buffer", lambda e: e.eip197_pairing_check_ragged_batch(
        (np.zeros(383, np.uint8), np.array([0, 192, 384], np.uint64)))),
    ("dev decreasing offsets", lambda e: e.pairing_check_ragged_batch_dev(Dev(N), Dev(N), [0, 2, 1, 4], Dev(3))),
    ("dev short last offset", lambda e: e.pairing_check_ragged_batch_dev(Dev(N), Dev(N), [0, 2, 3], Dev(2))),
    ("dev g2 rows", lambda e: e.pairing_check_ragged_batch_dev(Dev(N), Dev(3), OFFS, Dev(3))),
    ("dev flags", lambda e: e.pairing_check_ragged_batch_dev(Dev(N), Dev(N), OFFS, Dev(3), d_g1_inf=Dev(3))),
    ("dev verdicts", lambda e: e.pairing_check_ragged_batch_dev(Dev(N), Dev(N), OFFS, Dev(4))),
]


@pytest.mark.parametrize("call", [b[1] for b in BAD], ids=[b[0] for b in BAD])
def test_bad_arguments_are_rejected_before_the_call(eng, call):
    with pytest.raises(ValueError):
        call(eng)
    assert eng._lib.calls == []

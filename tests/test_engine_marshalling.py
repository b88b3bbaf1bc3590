"""CPU tier: how Engine's host-buffer methods hand their arguments to the C ABI.  A stub stands in for
libsylow_b200.so and records every call, so no GPU and no built library are needed.  Each method must call its C
function once, with the context, the caller's arrays by address (no copy), the integers of the prototype and outputs
that it returns.  A per-item array that does not match the batch size must raise ValueError before any call: the
library would read past its end."""
import ctypes

import numpy as np
import pytest

from sylow_b200.api import DST, Engine

N = 4
TABLE = 87 * 192


class Out:
    """An output of `nbytes` that the method converts before returning it; the stub fills it with 1s."""

    def __init__(self, nbytes):
        self.nbytes = nbytes


class Ret:
    """A pointer to the data of the returned array (of element i of a returned tuple)."""

    def __init__(self, i=None):
        self.i = i


class Data:
    """A pointer to these bytes, in a buffer the method builds (packed messages, a seed)."""

    def __init__(self, b):
        self.b = bytes(b)


class Ref:
    """A byref() output; the stub stores `value` in it."""

    def __init__(self, value):
        self.value = value


class Tensor:
    """Stands in for a torch tensor: only its address is used."""

    def data_ptr(self):
        return 0x7000


STREAM = ctypes.c_void_p(0x5000)


class StubLib:
    def __init__(self):
        self.calls = []
        self.expect = []

    def __getattr__(self, name):
        if not name.startswith("sylow_b200_"):
            raise AttributeError(name)

        def fn(*args):
            seen = []  # what only the call itself can observe: buffers freed when the method returns
            for e, a in zip(self.expect, args[1:]):
                if isinstance(e, Out):
                    ctypes.memset(a.value, 1, e.nbytes)
                elif isinstance(e, Ref):
                    a._obj.value = e.value
                seen.append(ctypes.string_at(a.value, len(e.b)) if isinstance(e, Data) and a is not None else None)
            self.calls.append((name, args, seen))
            return 0

        fn.__name__ = name
        return fn


@pytest.fixture
def eng(monkeypatch):
    monkeypatch.setattr(Engine, "_stream", staticmethod(lambda: STREAM))
    e = Engine.__new__(Engine)
    e._lib = StubLib()
    e._h = ctypes.c_void_p(0x1000)
    yield e
    e._h = None


def _rows(n, width, seed):
    return np.random.default_rng(seed).integers(0, 256, size=(n, width), dtype=np.uint8)


G1, G2, F, SC, SC2 = _rows(N, 64, 1), _rows(N, 128, 2), _rows(N, 384, 3), _rows(N, 32, 4), _rows(N, 32, 16)
INF, INF2 = np.array([0, 1, 0, 0], np.uint8), np.array([1, 0, 0, 1], np.uint8)
COEFFS, COEFF1 = _rows(N, TABLE, 5), _rows(1, TABLE, 6)
G2V, INF_V = _rows(2, 128, 7), np.array([0, 1], np.uint8)
BE64, BE128, EIP = _rows(N, 64, 8), _rows(N, 128, 9), _rows(N, 2 * 192, 10)
IDS, TSIGS, TINF = np.arange(1, 7, dtype=np.uint64).reshape(2, 3), _rows(6, 64, 11).reshape(2, 3, 64), np.zeros(6, np.uint8)
PK, PKS, SIGS = _rows(1, 128, 12).reshape(128), _rows(N, 128, 13), _rows(N, 64, 14)
MSGS = [b"a", b"bc", b"", b"def"]
BUF, OFFS = np.frombuffer(b"abcdef", np.uint8).copy(), np.array([0, 1, 3, 3, 6], np.uint64)
SEED = bytes(range(32))
PARTIALS = _rows(2, 384, 15)

M = [Data(BUF), Data(OFFS)]  # messages given as a list are packed by the method
K = [DST, len(DST), 0]  # dst, dst_len, keccak-256

# (method, args, kwargs, C function, expected arguments after the context, check of the result)
CASES = [
    ("pairing_batch", (G1, G2, INF, INF2), {}, "pairing_batch", [G1, INF, G2, INF2, N, Ret()], (N, 384)),
    ("pairing_batch", (G1, G2), {}, "pairing_batch", [G1, None, G2, None, N, Ret()], (N, 384)),
    ("miller_loop_batch", (G1, G2, INF), {}, "miller_loop_batch", [G1, INF, G2, None, N, Ret()], (N, 384)),
    ("miller_product", (G1, G2, None, INF2), {}, "miller_product", [G1, None, G2, INF2, N, Ret()], (384,)),
    ("final_exp_batch", (F,), {}, "final_exp_batch", [F, N, Ret()], (N, 384)),
    ("fp12_product", (F,), {}, "fp12_product", [F, N, Ret()], (384,)),
    ("pairing_check_batch", (G1, G2, 2, INF, INF2), {}, "pairing_check_batch",
     [G1, INF, G2, INF2, 2, 2, Out(2)], [True, True]),
    ("g2_precompute", (G2,), {}, "g2_precompute", [G2, N, Ret()], (N, TABLE)),
    ("miller_loop_precomputed", (COEFF1, G1, INF), {}, "miller_loop_precomputed", [COEFF1, G1, INF, N, Ret()], (N, 384)),
    ("miller_loop_precomputed_batch", (COEFFS, G1, INF), {}, "miller_loop_precomputed_batch",
     [COEFFS, G1, INF, N, Ret()], (N, 384)),
    ("miller_product_precomputed", (COEFFS, G1), {}, "miller_product_precomputed", [COEFFS, G1, None, N, Ret()], (384,)),
    ("pairing_check_fixed_batch", (G1, G2V, COEFF1, 1, 1), {"g1_inf": INF, "g2_var_inf": INF_V},
     "pairing_check_fixed_batch", [G1, INF, G2V, INF_V, 1, COEFF1, 1, 2, Out(2)], [True, True]),
    ("pairing_check_fixed_batch", (G1[:2], None, COEFF1, 0, 1), {}, "pairing_check_fixed_batch",
     [G1[:2], None, None, None, 0, COEFF1, 1, 2, Out(2)], [True, True]),
    ("tables_to_device", (COEFFS, Tensor()), {}, "tables_to_device", [COEFFS, N, Tensor(), STREAM], None),
    ("g1_validate_batch", (G1, INF), {}, "g1_validate_batch", [G1, INF, N, Ret()], (N,)),
    ("g2_validate_batch", (G2,), {}, "g2_validate_batch", [G2, None, N, Ret()], (N,)),
    ("g1_from_be_bytes_batch", (BE64, True), {}, "g1_from_be_bytes_batch", [BE64, N, 1, Ret(0), Ret(1), Ret(2)], None),
    ("g2_from_be_bytes_batch", (BE128,), {}, "g2_from_be_bytes_batch", [BE128, N, 0, Ret(0), Ret(1), Ret(2)], None),
    ("g1_to_be_bytes_batch", (G1, INF), {"scrubbed": True}, "g1_to_be_bytes_batch", [G1, INF, N, 1, Ret()], (N, 64)),
    ("g2_to_be_bytes_batch", (G2,), {}, "g2_to_be_bytes_batch", [G2, None, N, 0, Ret()], (N, 128)),
    ("eip197_pairing_check_batch", (EIP, 2), {}, "eip197_pairing_check_batch", [EIP, 2, N, Out(N), Ret(1)],
     lambda r: r[0].tolist() == [True] * N and r[1].dtype == np.int8),
    ("g1_mul_batch", (G1, SC, INF), {}, "g1_mul_batch", [G1, INF, SC, N, Ret(0), Ret(1)], None),
    ("g2_mul_batch", (G2, SC), {}, "g2_mul_batch", [G2, None, SC, N, Ret(0), Ret(1)], None),
    ("gt_mul_batch", (F, SC), {}, "gt_mul_batch", [F, SC, N, Ret()], (N, 384)),
    ("g1_sum", (G1, INF), {}, "g1_sum", [G1, INF, N, Ret(0), Out(1)], lambda r: r[1] == 1),
    ("g1_msm", (G1, SC, INF), {}, "g1_msm", [G1, INF, SC, N, Ret(0), Out(1)], lambda r: r[1] == 1),
    ("g1_msm_bucket", (G1, SC), {"window_bits": 9}, "g1_msm_bucket", [G1, None, SC, N, 9, Ret(0), Out(1)],
     lambda r: r[1] == 1),
    ("lagrange_coefficients_batch", (IDS,), {}, "lagrange_coefficients_batch", [IDS, 2, 3, Ret()], (2, 3, 32)),
    ("threshold_aggregate_batch", (IDS, TSIGS, TINF), {}, "threshold_aggregate_batch",
     [IDS, TSIGS, TINF, 2, 3, Ret(0), Ret(1)], None),
    ("verify_batch_same_signer", (PK, MSGS, SIGS), {"pk_inf": True, "sigs_inf": INF, "weight_seed": SEED},
     "verify_batch_same_signer", [PK, 1] + M + [SIGS, INF, N] + K + [Data(SEED), Ref(1)], True),
    ("verify_batch_same_signer", (PK, (BUF, OFFS), SIGS), {}, "verify_batch_same_signer",
     [PK, 0, BUF, OFFS, SIGS, None, N] + K + [None, Ref(1)], True),
    ("batch_weights", (SEED, 5, N), {}, "batch_weights", [Data(SEED), 5, N, Ret()], (N,)),
    ("hash_to_g1_batch", (MSGS,), {"dst": b"d", "hash_id": 1}, "hash_to_g1_batch",
     M + [N, b"d", 1, 1, Ret(0), Ret(1)], None),
    ("expand_message_batch", ((BUF, OFFS), b"dst", 48), {"hash_id": 2}, "expand_message_batch",
     [BUF, OFFS, N, b"dst", 3, 2, 48, Ret()], (N, 48)),
    ("hash_to_field_batch", (MSGS,), {}, "hash_to_field_batch", M + [N] + K + [Ret()], (N, 64)),
    ("sign_batch", (SC, MSGS), {"return_inf": True}, "sign_batch", [SC] + M + [N] + K + [Ret(0), Ret(1)], None),
    ("sign_batch", (SC, (BUF, OFFS)), {}, "sign_batch", [SC, BUF, OFFS, N] + K + [Ret(), Out(N)], (N, 64)),
    ("verify_each", (PKS, MSGS, SIGS), {"pks_inf": INF, "sigs_inf": INF2}, "verify_each",
     [PKS, INF] + M + [SIGS, INF2, N] + K + [Out(N)], [True] * N),
    ("verify_batch_partial", (PKS, (BUF, OFFS), SIGS), {"weight_seed": SEED, "first_index": 7}, "verify_batch_partial",
     [PKS, None, BUF, OFFS, SIGS, None, N] + K + [Data(SEED), 7, Ret()], (384,)),
    ("verify_batch_finish", (PARTIALS,), {}, "verify_batch_finish", [PARTIALS, 2, Ref(1)], True),
    ("verify_batch", (PKS, MSGS, SIGS), {"sigs_inf": INF}, "verify_batch",
     [PKS, None] + M + [SIGS, INF, N] + K + [None, Ref(1)], True),
    ("verify_batch", (PKS, MSGS, SIGS), {"weight_seed": SEED}, "verify_batch",
     [PKS, None] + M + [SIGS, None, N] + K + [Data(SEED), Ref(1)], True),
    ("fp_op_batch", (3, SC, SC2), {}, "fp_op_batch", [3, SC, SC2, N, Ret()], (N, 32)),
    ("fp12_op_batch", (7, F, F), {}, "fp12_op_batch", [7, F, F, N, Ret()], (N, 384)),
    ("imad_probe", (1, 2, 3, 4), {}, "imad_probe", [1, 2, 3, 4, Ref(1.5), Ref(2.5)], (1.5, 2.5)),
]


def _addr(p):
    assert isinstance(p, ctypes.c_void_p), p
    return p.value


@pytest.mark.parametrize("method,args,kwargs,symbol,expect,result", CASES,
                         ids=["%s-%d" % (c[0], i) for i, c in enumerate(CASES)])
def test_host_method_marshalling(eng, method, args, kwargs, symbol, expect, result):
    lib = eng._lib
    lib.expect = expect
    r = getattr(eng, method)(*args, **kwargs)
    assert len(lib.calls) == 1, lib.calls
    name, got, seen = lib.calls[0]
    assert name == "sylow_b200_" + symbol
    assert got[0] is eng._h
    assert len(got) - 1 == len(expect)
    for i, (e, a) in enumerate(zip(expect, got[1:])):
        if e is None or isinstance(e, (ctypes.c_void_p, bytes)):
            assert a is e or a == e, (i, a)
        elif isinstance(e, int):
            assert type(a) is int and a == e, (i, a)
        elif isinstance(e, np.ndarray):
            assert _addr(a) == e.ctypes.data, i  # the caller's array itself, not a copy
        elif isinstance(e, Tensor):
            assert _addr(a) == e.data_ptr(), i
        elif isinstance(e, Ret):
            assert _addr(a) == (r if e.i is None else r[e.i]).ctypes.data, i
        elif isinstance(e, Data):
            assert seen[i] == e.b, i
        elif isinstance(e, Out):
            assert _addr(a), i
        elif isinstance(e, Ref):
            assert type(a).__name__ == "CArgObject", i
        else:
            raise AssertionError(e)
    if isinstance(result, tuple) and isinstance(r, np.ndarray):
        assert r.shape == result
    elif callable(result):
        assert result(r)
    elif result is not None:
        assert (r.tolist() if isinstance(r, np.ndarray) else r) == result


SHORT = N - 1
BAD = [
    ("sign_batch", lambda e: e.sign_batch(SC[:SHORT], MSGS)),
    ("verify_each pks", lambda e: e.verify_each(PKS[:SHORT], MSGS, SIGS)),
    ("verify_each sigs", lambda e: e.verify_each(PKS, MSGS, SIGS[:SHORT])),
    ("verify_batch_partial pks", lambda e: e.verify_batch_partial(PKS[:SHORT], MSGS, SIGS)),
    ("verify_batch_partial sigs", lambda e: e.verify_batch_partial(PKS, MSGS, SIGS[:SHORT])),
    ("verify_batch pks", lambda e: e.verify_batch(PKS[:SHORT], MSGS, SIGS)),
    ("verify_batch sigs", lambda e: e.verify_batch(PKS, MSGS, SIGS[:SHORT])),
    ("verify_batch_same_signer sigs", lambda e: e.verify_batch_same_signer(PK, MSGS, SIGS[:SHORT])),
    ("g1_msm scalars", lambda e: e.g1_msm(G1, SC[:SHORT])),
    ("g1_msm_bucket scalars", lambda e: e.g1_msm_bucket(G1, SC[:SHORT])),
    ("fp_op_batch b", lambda e: e.fp_op_batch(0, SC, SC[:SHORT])),
    ("fp12_op_batch b", lambda e: e.fp12_op_batch(0, F, F[:SHORT])),
    ("pairing_check_fixed_batch g1_inf", lambda e: e.pairing_check_fixed_batch(G1, G2V, COEFF1, 1, 1,
                                                                                g1_inf=INF[:SHORT])),
    ("pairing_check_fixed_batch g2_var_inf", lambda e: e.pairing_check_fixed_batch(G1, G2V, COEFF1, 1, 1,
                                                                                    g2_var_inf=INF)),
    ("messages buffer", lambda e: e.hash_to_g1_batch((BUF[:5], OFFS))),
    ("messages buffer verify", lambda e: e.verify_batch(PKS, (BUF[:5], OFFS), SIGS)),
]


@pytest.mark.parametrize("call", [b[1] for b in BAD], ids=[b[0] for b in BAD])
def test_short_per_item_array_is_rejected_before_the_call(eng, call):
    with pytest.raises(ValueError):
        call(eng)
    assert eng._lib.calls == []

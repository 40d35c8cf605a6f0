"""CPU-only checks of blsgpu_verify_batch_grouped's host side: the Python mirror's length rules (they fire before any
engine call) and the C entry point's refusal of a NULL context."""
import ctypes

import numpy as np
import pytest


@pytest.fixture(scope="module", autouse=True)
def built_library():
    import __graft_entry__ as g
    g.build_engine()


@pytest.fixture
def detached():
    """An Engine whose context is NULL: whatever reaches the C ABI comes back as BLSGPU_E_ARG, no GPU needed."""
    import blsful_b200 as B
    e = B.Engine.__new__(B.Engine)
    e._lib = B.load_library()
    e._ctx = None
    return e


@pytest.mark.parametrize("impl", [1, 2])
def test_length_rules(detached, impl):
    import blsful_b200 as B
    pl, sl = B.pk_len(impl), B.sig_len(impl)
    with pytest.raises(B.BlsError) as e:
        detached.verify_batch_grouped(impl, 0, [bytes(pl), bytes(pl - 1)], [bytes(sl)] * 2, [0, 0], [b"m"])
    assert e.value.status == B.ST_INVALID_LENGTH
    with pytest.raises(B.BlsError) as e:
        detached.verify_batch_grouped(impl, 0, [bytes(pl)] * 2, [bytes(sl), bytes(sl + 1)], [0, 0], [b"m"])
    assert e.value.status == B.ST_INVALID_LENGTH
    with pytest.raises(B.BlsError) as e:   # one signature per public key
        detached.verify_batch_grouped(impl, 0, [bytes(pl)] * 2, [bytes(sl)], [0, 0], [b"m"])
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    with pytest.raises(B.BlsError) as e:   # one message index per item
        detached.verify_batch_grouped(impl, 0, [bytes(pl)] * 2, [bytes(sl)] * 2, [0], [b"m"])
    assert e.value.status == B.ST_MISMATCHED_LENGTHS


def test_null_context_is_an_argument_error(detached):
    import blsful_b200 as B
    lib = B.load_library()
    moff = np.array([0, 1], dtype=np.uint64)
    idx = np.zeros(1, dtype=np.uint32)
    pk, sg, msg, st = np.zeros(48, dtype=np.uint8), np.zeros(96, dtype=np.uint8), np.zeros(1, dtype=np.uint8), np.zeros(1, dtype=np.uint8)
    assert lib.blsgpu_verify_batch_grouped(None, 2, 0, 1, 1, pk.ctypes.data, sg.ctypes.data, idx.ctypes.data, 1, msg.ctypes.data,
                                           moff.ctypes.data, st.ctypes.data) == -1   # BLSGPU_E_ARG
    with pytest.raises(B.EngineError):
        detached.verify_batch_grouped(2, 0, [bytes(48)], [bytes(96)], [0], [b"m"])
    assert lib.blsgpu_verify_batch_grouped(ctypes.c_void_p(None), 2, 0, 1, 0, None, None, None, 0, None, None, None) == -1

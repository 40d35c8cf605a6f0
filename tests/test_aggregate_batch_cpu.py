"""CPU-only checks of blsgpu_aggregate_verify_batch's host side: the Python mirror's length rules (they fire before any
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
def test_wrong_pk_or_signature_length_is_invalid_length(detached, impl):
    import blsful_b200 as B
    pl, sl = B.pk_len(impl), B.sig_len(impl)
    good = (bytes(pl), b"m")
    with pytest.raises(B.BlsError) as e:
        detached.aggregate_verify_batch_status(impl, 0, [([bytes(pl), bytes(pl - 1)], [b"a", b"b"])], [bytes(sl)])
    assert e.value.status == B.ST_INVALID_LENGTH
    with pytest.raises(B.BlsError) as e:
        detached.aggregate_verify_batch_status(impl, 0, [([good[0]], [good[1]]), ([good[0]], [good[1]])], [bytes(sl), bytes(sl + 1)])
    assert e.value.status == B.ST_INVALID_LENGTH
    with pytest.raises(B.BlsError) as e:   # one message per public key, one signature per aggregate
        detached.aggregate_verify_batch_status(impl, 0, [([good[0]], [b"a", b"b"])], [bytes(sl)])
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    with pytest.raises(B.BlsError) as e:
        detached.aggregate_verify_batch_status(impl, 0, [([good[0]], [good[1]])], [bytes(sl), bytes(sl)])
    assert e.value.status == B.ST_MISMATCHED_LENGTHS


def test_null_context_is_an_argument_error(detached):
    import blsful_b200 as B
    lib = B.load_library()
    soff = np.array([0, 1], dtype=np.uint64)
    moff = np.array([0, 1], dtype=np.uint64)
    pk, sg, msg = np.zeros(48, dtype=np.uint8), np.zeros(96, dtype=np.uint8), np.zeros(1, dtype=np.uint8)
    st, idx = np.zeros(1, dtype=np.uint8), np.zeros(2, dtype=np.int64)
    assert lib.blsgpu_aggregate_verify_batch(None, 2, 0, 1, 1, soff.ctypes.data, pk.ctypes.data, msg.ctypes.data, moff.ctypes.data,
                                             sg.ctypes.data, st.ctypes.data, idx.ctypes.data) == -1   # BLSGPU_E_ARG
    with pytest.raises(B.EngineError):
        detached.aggregate_verify_batch_status(2, 0, [([bytes(48)], [b"m"])], [bytes(96)])
    assert lib.blsgpu_aggregate_verify_batch(ctypes.c_void_p(None), 2, 0, 1, 0, None, None, None, None, None, None, None) == -1

"""CPU-only checks of the key-set entry points' host side: the C functions refuse a NULL context, and the Python mirror's
length rules fire before any engine call."""
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


def test_null_context_is_an_argument_error():
    import blsful_b200 as B
    lib = B.load_library()
    pk, sg, msg, st = np.zeros(48, dtype=np.uint8), np.zeros(96, dtype=np.uint8), np.zeros(1, dtype=np.uint8), np.zeros(1, dtype=np.uint8)
    moff = np.array([0, 1], dtype=np.uint64)
    idx = np.zeros(1, dtype=np.uint32)
    out = ctypes.c_uint64(0)
    assert lib.blsgpu_keyset_create(None, 2, 1, 1, pk.ctypes.data, st.ctypes.data, ctypes.byref(out)) == -1
    assert out.value == 0
    assert lib.blsgpu_keyset_destroy(None, 1) == -1
    assert lib.blsgpu_verify_batch_keyed(None, 1, 0, 1, 1, idx.ctypes.data, sg.ctypes.data, msg.ctypes.data, moff.ctypes.data,
                                         st.ctypes.data) == -1
    assert lib.blsgpu_verify_batch_grouped_keyed(None, 1, 0, 1, 1, idx.ctypes.data, sg.ctypes.data, idx.ctypes.data, 1, msg.ctypes.data,
                                                 moff.ctypes.data, st.ctypes.data) == -1
    assert lib.blsgpu_verify_batch_keyed(ctypes.c_void_p(None), 0, 0, 1, 0, None, None, None, None, None) == -1


@pytest.mark.parametrize("impl", [1, 2])
def test_key_set_length_rule(detached, impl):
    import blsful_b200 as B
    pl = B.pk_len(impl)
    with pytest.raises(B.BlsError) as e:
        detached.key_set(impl, [bytes(pl), bytes(pl + 1)])
    assert e.value.status == B.ST_INVALID_LENGTH
    with pytest.raises(B.BlsError) as e:
        detached.key_set(impl, np.zeros(pl + 3, dtype=np.uint8))
    assert e.value.status == B.ST_INVALID_LENGTH
    with pytest.raises(B.EngineError):   # well-formed input reaches the C ABI, which refuses the NULL context
        detached.key_set(impl, [bytes(pl)])


@pytest.mark.parametrize("impl", [1, 2])
def test_keyed_length_rules(detached, impl):
    import blsful_b200 as B
    sl = B.sig_len(impl)
    ks = B.KeySet(detached, impl, 7, np.zeros(3, dtype=np.uint8))   # an id the NULL context does not hold
    assert len(ks) == 3
    with pytest.raises(B.BlsError) as e:
        detached.verify_batch_keyed(ks, 0, [0, 1], [bytes(sl), bytes(sl - 1)], [b"a", b"b"])
    assert e.value.status == B.ST_INVALID_LENGTH
    with pytest.raises(B.BlsError) as e:   # one signature per key index
        detached.verify_batch_keyed(ks, 0, [0, 1], [bytes(sl)], [b"a", b"b"])
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    with pytest.raises(B.BlsError) as e:   # one message per item
        detached.verify_batch_keyed(ks, 0, [0, 1], [bytes(sl)] * 2, [b"a"])
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    with pytest.raises(B.BlsError) as e:
        detached.verify_batch_grouped_keyed(ks, 0, [0, 1], [bytes(sl + 1), bytes(sl)], [0, 0], [b"m"])
    assert e.value.status == B.ST_INVALID_LENGTH
    with pytest.raises(B.BlsError) as e:   # one signature per key index
        detached.verify_batch_grouped_keyed(ks, 0, [0, 1, 2], [bytes(sl)] * 2, [0, 0], [b"m"])
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    with pytest.raises(B.BlsError) as e:   # one message index per item
        detached.verify_batch_grouped_keyed(ks, 0, [0, 1], [bytes(sl)] * 2, [0], [b"m"])
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    data, off = B.pack_messages([b"a", b"b"])
    with pytest.raises(B.BlsError) as e:   # packed: key indices for every item
        detached.verify_batch_keyed_packed(ks, 0, np.zeros(1, dtype=np.uint32), np.zeros(2 * sl, dtype=np.uint8), data, off)
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    with pytest.raises(B.EngineError):
        detached.verify_batch_keyed(ks, 0, [0, 1], [bytes(sl)] * 2, [b"a", b"b"])
    with pytest.raises(B.EngineError):
        detached.verify_batch_grouped_keyed(ks, 0, [0, 1], [bytes(sl)] * 2, [0, 0], [b"m"])
    ks.close()   # no context: nothing to free, and idempotent
    ks.close()
    assert ks.id == 0

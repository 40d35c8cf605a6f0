"""CPU-only checks of the multi-signature entry points' host side: the library exports them, the C functions refuse a NULL
context, and the Python mirror's length rules fire before any engine call."""
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


def test_the_library_exports_the_multisig_calls():
    import blsful_b200 as B
    lib = B.load_library()
    for name in ("blsgpu_verify_multisig_batch", "blsgpu_verify_multisig_batch_keyed", "blsgpu_sum_points_batch"):
        assert name in B.EXPORTED_SYMBOLS
        assert getattr(lib, name).restype is ctypes.c_int


def test_null_context_is_an_argument_error():
    import blsful_b200 as B
    lib = B.load_library()
    koff = np.array([0, 2], dtype=np.uint64)
    idx = np.zeros(2, dtype=np.uint32)
    pk, sg = np.zeros(2 * 48, dtype=np.uint8), np.zeros(96, dtype=np.uint8)
    msg, moff, st = np.zeros(1, dtype=np.uint8), np.array([0, 1], dtype=np.uint64), np.zeros(1, dtype=np.uint8)
    out, bad = np.zeros(48, dtype=np.uint8), np.zeros(1, dtype=np.int64)
    assert lib.blsgpu_verify_multisig_batch(None, 2, 0, 1, 1, koff.ctypes.data, pk.ctypes.data, sg.ctypes.data, msg.ctypes.data,
                                            moff.ctypes.data, st.ctypes.data) == -1
    assert lib.blsgpu_verify_multisig_batch_keyed(None, 1, 0, 1, 1, koff.ctypes.data, idx.ctypes.data, sg.ctypes.data, msg.ctypes.data,
                                                  moff.ctypes.data, st.ctypes.data) == -1
    assert lib.blsgpu_sum_points_batch(None, 1, 1, 1, koff.ctypes.data, pk.ctypes.data, out.ctypes.data, st.ctypes.data,
                                       bad.ctypes.data) == -1
    assert lib.blsgpu_verify_multisig_batch(None, 2, 0, 1, 0, None, None, None, None, None, None) == -1
    assert lib.blsgpu_verify_multisig_batch_keyed(None, 0, 0, 1, 0, None, None, None, None, None, None) == -1
    assert lib.blsgpu_sum_points_batch(None, 1, 1, 0, None, None, None, None, None) == -1


@pytest.mark.parametrize("impl", [1, 2])
def test_multisig_length_rules(detached, impl):
    import blsful_b200 as B
    pl, sl = B.pk_len(impl), B.sig_len(impl)
    ks = B.KeySet(detached, impl, 7, np.zeros(3, dtype=np.uint8))   # an id the NULL context does not hold
    sets = [[bytes(pl)] * 2, [bytes(pl)]]
    with pytest.raises(B.BlsError) as e:   # one signature per set
        detached.verify_multisig_batch(impl, 0, sets, [bytes(sl)], [b"a", b"b"])
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    with pytest.raises(B.BlsError) as e:   # one message per set
        detached.verify_multisig_batch(impl, 0, sets, [bytes(sl)] * 2, [b"a"])
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    with pytest.raises(B.BlsError) as e:
        detached.verify_multisig_batch(impl, 0, [[bytes(pl)], [bytes(pl + 1)]], [bytes(sl)] * 2, [b"a", b"b"])
    assert e.value.status == B.ST_INVALID_LENGTH
    with pytest.raises(B.BlsError) as e:
        detached.verify_multisig_batch(impl, 0, sets, [bytes(sl), bytes(sl - 1)], [b"a", b"b"])
    assert e.value.status == B.ST_INVALID_LENGTH
    data, off = B.pack_messages([b"a", b"b"])
    koff = np.array([0, 2, 3], dtype=np.uint64)
    with pytest.raises(B.BlsError) as e:   # packed: pk holds key_off[q] keys
        detached.verify_multisig_batch_packed(impl, 0, koff, np.zeros(2 * pl, dtype=np.uint8), np.zeros(2 * sl, dtype=np.uint8), data, off)
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    with pytest.raises(B.BlsError) as e:   # packed: q signatures
        detached.verify_multisig_batch_packed(impl, 0, koff, np.zeros(3 * pl, dtype=np.uint8), np.zeros(3 * sl, dtype=np.uint8), data, off)
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    with pytest.raises(B.BlsError) as e:   # keyed: one signature per set
        detached.verify_multisig_batch_keyed(ks, 0, [[0, 1], [2]], [bytes(sl)], [b"a", b"b"])
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    with pytest.raises(B.BlsError) as e:   # keyed: one message per set
        detached.verify_multisig_batch_keyed(ks, 0, [[0, 1], [2]], [bytes(sl)] * 2, [b"a"])
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    with pytest.raises(B.BlsError) as e:
        detached.verify_multisig_batch_keyed(ks, 0, [[0, 1], [2]], [bytes(sl), bytes(sl + 1)], [b"a", b"b"])
    assert e.value.status == B.ST_INVALID_LENGTH
    with pytest.raises(B.BlsError) as e:   # keyed packed: key_idx holds key_off[q] entries
        detached.verify_multisig_batch_keyed_packed(ks, 0, koff, np.zeros(2, dtype=np.uint32), np.zeros(2 * sl, dtype=np.uint8), data, off)
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    with pytest.raises(B.BlsError) as e:   # keyed packed: one message per set
        detached.verify_multisig_batch_keyed_packed(ks, 0, koff, np.zeros(3, dtype=np.uint32), np.zeros(2 * sl, dtype=np.uint8),
                                                    *B.pack_messages([b"a"]))
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    group = 2 if impl == 1 else 1
    with pytest.raises(B.BlsError) as e:
        detached.sum_points_batch(group, [[bytes(pl)], [bytes(pl - 1)]])
    assert e.value.status == B.ST_INVALID_LENGTH
    with pytest.raises(B.BlsError) as e:   # packed: set_off[q] points
        detached.sum_points_batch_packed(group, koff, np.zeros(2 * pl, dtype=np.uint8))
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    with pytest.raises(B.EngineError):   # well-formed input reaches the C ABI, which refuses the NULL context
        detached.verify_multisig_batch(impl, 0, sets, [bytes(sl)] * 2, [b"a", b"b"])
    with pytest.raises(B.EngineError):
        detached.verify_multisig_batch_keyed(ks, 0, [[0, 1], [2]], [bytes(sl)] * 2, [b"a", b"b"])
    with pytest.raises(B.EngineError):
        detached.sum_points_batch(group, sets)

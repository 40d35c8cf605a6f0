"""CPU-only checks of blsgpu_keyset_update / blsgpu_keyset_append: both refuse a NULL context, both are exported and declared
(test_abi_cpu.py checks the header, the export list and the Rust sys crate against each other), and the Python mirror's
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
    pk, st = np.zeros(48, dtype=np.uint8), np.zeros(1, dtype=np.uint8)
    idx = np.zeros(1, dtype=np.uint32)
    assert lib.blsgpu_keyset_update(None, 1, 1, 1, idx.ctypes.data, pk.ctypes.data, st.ctypes.data) == -1
    assert lib.blsgpu_keyset_append(None, 1, 1, 1, pk.ctypes.data, st.ctypes.data) == -1
    assert lib.blsgpu_keyset_update(None, 1, 1, 0, None, None, None) == -1
    assert lib.blsgpu_keyset_append(None, 1, 1, 0, None, None) == -1


def test_exported_and_registered():
    import blsful_b200 as B
    lib = B.load_library()
    for name in ("blsgpu_keyset_update", "blsgpu_keyset_append"):
        assert name in B.EXPORTED_SYMBOLS
        assert getattr(lib, name).argtypes is not None


@pytest.mark.parametrize("impl", [1, 2])
def test_update_and_append_length_rules(detached, impl):
    import blsful_b200 as B
    pl = B.pk_len(impl)
    ks = B.KeySet(detached, impl, 7, np.zeros(3, dtype=np.uint8))   # an id the NULL context does not hold
    with pytest.raises(B.BlsError) as e:
        detached.update_key_set(ks, [0, 1], [bytes(pl), bytes(pl - 1)])
    assert e.value.status == B.ST_INVALID_LENGTH
    with pytest.raises(B.BlsError) as e:
        detached.update_key_set(ks, [0], np.zeros(pl + 5, dtype=np.uint8))
    assert e.value.status == B.ST_INVALID_LENGTH
    with pytest.raises(B.BlsError) as e:   # one key per index
        detached.update_key_set(ks, [0, 1], [bytes(pl)])
    assert e.value.status == B.ST_MISMATCHED_LENGTHS
    with pytest.raises(B.BlsError) as e:
        detached.append_key_set(ks, [bytes(pl + 1)])
    assert e.value.status == B.ST_INVALID_LENGTH
    with pytest.raises(B.BlsError) as e:
        detached.append_key_set(ks, np.zeros(2 * pl - 1, dtype=np.uint8))
    assert e.value.status == B.ST_INVALID_LENGTH
    with pytest.raises(B.EngineError):   # well-formed input reaches the C ABI, which refuses the NULL context
        detached.update_key_set(ks, [0], [bytes(pl)])
    with pytest.raises(B.EngineError):
        detached.append_key_set(ks, [bytes(pl)])
    assert len(ks) == 3 and ks.status.tolist() == [0, 0, 0]   # a refused call leaves the mirror's statuses alone

"""blsgpu_verify_batch_records refuses a null pk_bytes, sig_bytes or msgs buffer whose offsets span bytes (BLSGPU_E_ARG)
instead of reading through it, and the context still verifies afterwards."""
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import bls_oracle as O

E_ARG = -1


@pytest.mark.parametrize("null", ["pk_bytes", "sig_bytes", "msgs"])
def test_records_with_a_null_buffer_are_refused(null):
    import blsful_b200 as B
    eng = B.Engine([0])
    try:
        rnd = random.Random(4242)
        n, impl = 8, 2
        k = np.frombuffer(b"".join(rnd.randrange(1, O.R).to_bytes(32, "big") for _ in range(n)), dtype=np.uint8)
        data, off = B.pack_messages([b"records-%d" % i for i in range(n)])
        pks, sigs = eng.testdata_sign(impl, 0, k, data, off)
        pk_off = np.arange(n + 1, dtype=np.uint64) * np.uint64(B.pk_len(impl))
        sig_off = np.arange(n + 1, dtype=np.uint64) * np.uint64(B.sig_len(impl))

        def call(null_name=None, msg_off=off):
            bufs = {"pk_bytes": pks, "sig_bytes": sigs, "msgs": data}
            ptr = {name: None if name == null_name else a.ctypes.data for name, a in bufs.items()}
            st = np.full(n, 0xAA, dtype=np.uint8)
            rc = eng._lib.blsgpu_verify_batch_records(eng._ctx, impl, 1, 0, n, ptr["pk_bytes"], pk_off.ctypes.data, ptr["sig_bytes"],
                                                      sig_off.ctypes.data, ptr["msgs"], msg_off.ctypes.data, st.ctypes.data)
            return rc, st

        rc, _ = call(null)
        assert rc == E_ARG
        assert b"is null" in eng._lib.blsgpu_last_error(eng._ctx)
        rc, st = call()
        assert rc == 0 and st.tolist() == [0] * n
        if null == "msgs":  # a null buffer stays legal when its records are empty
            rc, _ = call(null, msg_off=np.zeros(n + 1, dtype=np.uint64))
            assert rc == 0
    finally:
        eng.close()

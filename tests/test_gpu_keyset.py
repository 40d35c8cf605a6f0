"""Key sets and the keyed verify calls: every status must equal the unkeyed call's on the same items with the key bytes
written out (and, on a sample, the big-int oracle); rejections stay exact at scale; no public key is decoded by a keyed call;
ids are checked, and the set's device memory lives and dies with the set."""
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import bls_oracle as O


@pytest.fixture(scope="module")
def B():
    import blsful_b200
    return blsful_b200


@pytest.fixture(scope="module")
def eng(B):
    e = B.Engine([0])
    yield e
    e.close()


def _ident(length):
    return bytes([0xC0]) + bytes(length - 1)


def _off_curve(group):
    """A compressed encoding (Modern) whose x has no point on the curve: a decode error in either format."""
    if group == 1:
        x = 1
        while O.fp_sqrt((x ** 3 + 4) % O.P) is not None:
            x += 1
        e = bytearray(x.to_bytes(48, "big"))
    else:
        k = 1
        while O.f2_sqrt(O.f2_add(O.f2_mul(O.f2_sqr((k, 2)), (k, 2)), O.B2)) is not None:
            k += 1
        e = bytearray((2).to_bytes(48, "big") + k.to_bytes(48, "big"))
    e[0] |= 0x80
    return bytes(e)


def _neg(enc):
    return bytes([enc[0] ^ 0x20]) + enc[1:]


def _scalars(rnd, n):
    return [rnd.randrange(1, O.R).to_bytes(32, "big") for _ in range(n)]


def _groups(impl):
    return (1, 2) if impl == 2 else (2, 1)   # (public-key group, signature group)


def _sign(eng, B, impl, scheme, scalars, msgs):
    """(pks, sigs) as lists of Modern encodings, item i signed with scalars[i] over msgs[i]"""
    k = np.frombuffer(b"".join(scalars), dtype=np.uint8)
    pks, sigs = eng.testdata_sign(impl, scheme, k, *B.pack_messages(msgs))
    pl, sl = B.pk_len(impl), B.sig_len(impl)
    return [pks[i * pl:(i + 1) * pl].tobytes() for i in range(len(msgs))], [sigs[i * sl:(i + 1) * sl].tobytes() for i in range(len(msgs))]


K_SIGNERS, K_UNUSED = 30, 6
BAD_KEY, HEADER_KEY, IDENT_KEY = K_SIGNERS + K_UNUSED, K_SIGNERS + K_UNUSED + 1, K_SIGNERS + K_UNUSED + 2


@pytest.mark.parametrize("fmt", [O.MODERN, O.LEGACY])
@pytest.mark.parametrize("impl", [2, 1])
def test_mixed_batch_equals_the_unkeyed_calls_and_the_oracle(eng, B, impl, fmt):
    pkg, sgg = _groups(impl)
    pl, sl = B.pk_len(impl), B.sig_len(impl)
    for scheme in (0, 1, 2):
        rnd = random.Random(1000 * impl + 10 * fmt + scheme)
        secret = _scalars(rnd, K_SIGNERS + K_UNUSED)
        msgs = [b"keyed/%d/%d" % (scheme, j) for j in range(4)] + [b""]
        n = 420
        key_idx = [rnd.randrange(K_SIGNERS) for _ in range(n)]            # unsorted, repeating; keys 30..35 unused
        msg_idx = [0 if i < 200 else rnd.randrange(len(msgs)) for i in range(n)]
        rnd.shuffle(msg_idx)
        pks, sigs = _sign(eng, B, impl, scheme, [secret[k] for k in key_idx], [msgs[j] for j in msg_idx])
        _, sigs_other = _sign(eng, B, impl, scheme, [secret[k] for k in key_idx], [msgs[(j + 1) % len(msgs)] for j in msg_idx])
        kbytes = _sign(eng, B, impl, scheme, secret, [b"k"] * len(secret))[0] + [_off_curve(pkg), None, _ident(pl)]
        hdr = kbytes[0]
        D = _sign(eng, B, impl, 0, _scalars(rnd, 1), [b"D"])[1][0]
        on0 = [i for i in range(n) if msg_idx[i] == 0]
        names = {"bad_key": on0[3], "header_key": on0[4], "ident_key": on0[5], "undecodable_sig": on0[6], "ident_sig": on0[7],
                 "other_message": on0[8], "other_item": on0[9], "cancel_a": on0[10], "cancel_b": on0[150]}
        key_idx[names["bad_key"]], key_idx[names["header_key"]], key_idx[names["ident_key"]] = BAD_KEY, HEADER_KEY, IDENT_KEY
        sigs[names["undecodable_sig"]] = _off_curve(sgg)
        sigs[names["ident_sig"]] = _ident(sl)
        sigs[names["other_message"]] = sigs_other[names["other_message"]]
        sigs[names["other_item"]] = sigs[on0[20]] if key_idx[on0[20]] != key_idx[names["other_item"]] else sigs_other[names["other_item"]]
        a, b = names["cancel_a"], names["cancel_b"]   # errors that cancel in an unweighted sum
        sigs[a] = eng.sum_points(sgg, [sigs[a], D])
        sigs[b] = eng.sum_points(sgg, [sigs[b], _neg(D)])
        if fmt == O.LEGACY:
            def conv(group, encs):
                st, outs = eng.recode_points(group, encs, O.MODERN, O.LEGACY)
                return [o if s == 0 else O.modern_to_legacy(e) for e, s, o in zip(encs, st.tolist(), outs)]
            kbytes = conv(pkg, kbytes[:HEADER_KEY]) + [hdr if hdr[0] & 0x20 else _neg(hdr)] + conv(pkg, kbytes[IDENT_KEY:])
            sigs = conv(sgg, sigs)
        else:
            kbytes[HEADER_KEY] = bytes([hdr[0] & 0x7F]) + hdr[1:]   # no compression flag
        ks = eng.key_set(impl, kbytes, fmt)
        try:
            assert len(ks) == len(kbytes) and ks.impl_id == impl
            assert ks.status[BAD_KEY] in (O.ERR_DESERIALIZE, O.ERR_LEGACY_FORMAT)
            assert ks.status[HEADER_KEY] in (O.ERR_DESERIALIZE, O.ERR_LEGACY_FORMAT)
            assert ks.status[:BAD_KEY].tolist() == [0] * BAD_KEY and ks.status[IDENT_KEY] == 0
            item_pks = [kbytes[k] for k in key_idx]
            item_msgs = [msgs[j] for j in msg_idx]
            want = eng.verify_batch(impl, scheme, item_pks, sigs, item_msgs, fmt)
            keyed = eng.verify_batch_keyed(ks, scheme, key_idx, sigs, item_msgs, fmt)
            grouped = eng.verify_batch_grouped(impl, scheme, item_pks, sigs, msg_idx, msgs, fmt)
            grouped_keyed = eng.verify_batch_grouped_keyed(ks, scheme, key_idx, sigs, msg_idx, msgs, fmt)
            for got in (keyed, grouped, grouped_keyed):
                assert got.tolist() == want.tolist(), [(i, x, y) for i, (x, y) in enumerate(zip(got.tolist(), want.tolist())) if x != y]
            st = {name: int(want[i]) for name, i in names.items()}
            assert st["bad_key"] in (O.ERR_DESERIALIZE, O.ERR_LEGACY_FORMAT) and st["header_key"] in (O.ERR_DESERIALIZE, O.ERR_LEGACY_FORMAT)
            assert st["ident_key"] == O.ERR_PK_IDENTITY and st["ident_sig"] == O.ERR_SIG_IDENTITY
            assert st["undecodable_sig"] in (O.ERR_DESERIALIZE, O.ERR_LEGACY_FORMAT)
            assert st["other_message"] == st["other_item"] == st["cancel_a"] == st["cancel_b"] == 1
            assert sum(1 for s in want.tolist() if s) == len(names)
            if scheme == 0:   # a sample end to end against the big-int oracle
                for name in ("cancel_a", "ident_key", "header_key"):
                    i = names[name]
                    assert O.verify(impl, scheme, fmt, item_pks[i], sigs[i], item_msgs[i]) == keyed[i], name
                i = on0[0]
                assert O.verify(impl, scheme, fmt, item_pks[i], sigs[i], item_msgs[i]) == keyed[i] == 0
        finally:
            ks.close()


@pytest.fixture(scope="module")
def scale(eng, B):
    """2^20 G2Impl Basic items over a 2^16-key set and 1,000 messages (seeded key and message per item)"""
    rnd = random.Random(4096)
    n, k, q = 1 << 20, 1 << 16, 1000
    secret = np.frombuffer(b"".join(_scalars(rnd, k)), dtype=np.uint8).reshape(k, 32)
    nrng = np.random.default_rng(7)
    key_idx = nrng.integers(0, k, size=n, dtype=np.uint32)
    msg_idx = nrng.integers(0, q, size=n, dtype=np.uint32)
    msgs = [b"scale/%d" % j for j in range(q)]
    data_i, off_i = B.pack_messages([msgs[j] for j in msg_idx.tolist()])
    _, sg = eng.testdata_sign(2, 0, secret[key_idx].reshape(-1), data_i, off_i)
    kb, _ = eng.testdata_sign(2, 0, secret.reshape(-1), *B.pack_messages([b""] * k))
    data, off = B.pack_messages(msgs)
    return kb, key_idx, sg, msg_idx, data, off, data_i, off_i


def _plant(sg, n, bad):
    s = sg.copy().reshape(n, 96)
    for i in bad:       # another item's signature: a valid point that fails its own equation
        s[i] = sg.reshape(n, 96)[(i + 1) % n]
    return s.reshape(-1)


def test_failure_search_is_exact_at_scale(eng, B, scale):
    kb, key_idx, sg, msg_idx, data, off, data_i, off_i = scale
    n = key_idx.size
    ks = eng.key_set(2, kb)
    e2 = B.Engine([0])
    ks2 = e2.key_set(2, kb)
    try:
        assert not ks.status.any()
        rnd = random.Random(5)
        for nbad in (0, 1, 1000):
            bad = sorted(rnd.sample(range(n), nbad))
            planted = _plant(sg, n, bad)
            st = eng.verify_batch_keyed_packed(ks, 0, key_idx, planted, data_i, off_i)
            assert np.flatnonzero(st).tolist() == bad and (st[bad] == 1).all()
            st = eng.verify_batch_grouped_keyed_packed(ks, 0, key_idx, planted, msg_idx, data, off)
            assert np.flatnonzero(st).tolist() == bad and (st[bad] == 1).all()
        bad = sorted(rnd.sample(range(n), 1000))
        planted = _plant(sg, n, bad)
        e2.set_rlc_bits(128)
        assert np.flatnonzero(e2.verify_batch_keyed_packed(ks2, 0, key_idx, planted, data_i, off_i)).tolist() == bad
        assert np.flatnonzero(e2.verify_batch_grouped_keyed_packed(ks2, 0, key_idx, planted, msg_idx, data, off)).tolist() == bad
        e2.set_rlc_bits(64)
        e2.set_rlc_salt(bytes(range(32)))
        assert np.flatnonzero(e2.verify_batch_keyed_packed(ks2, 0, key_idx, planted, data_i, off_i)).tolist() == bad
        assert np.flatnonzero(e2.verify_batch_grouped_keyed_packed(ks2, 0, key_idx, planted, msg_idx, data, off)).tolist() == bad
    finally:
        e2.close()
        ks.close()


def test_several_miller_passes(eng, B, scale, monkeypatch):
    """BLSGPU_M6_CHUNK=1200: more items (and more leaves) than one pass of the Miller kernels holds"""
    kb, key_idx, sg, msg_idx, data, off, data_i, off_i = scale
    n = 130_000
    ks = eng.key_set(2, kb)
    try:
        bad = sorted(random.Random(9).sample(range(n), 25))
        planted = _plant(sg[:96 * n], n, bad)
        monkeypatch.setenv("BLSGPU_M6_CHUNK", "1200")
        st = eng.verify_batch_keyed_packed(ks, 0, key_idx[:n], planted, data_i[:int(off_i[n])], off_i[:n + 1])
        assert np.flatnonzero(st).tolist() == bad
        st = eng.verify_batch_grouped_keyed_packed(ks, 0, key_idx[:n], planted, msg_idx[:n], data, off)
        assert np.flatnonzero(st).tolist() == bad
    finally:
        ks.close()


@pytest.mark.parametrize("impl", [2, 1])
def test_keyed_calls_decode_no_public_key(eng, B, impl):
    rnd = random.Random(31 + impl)
    secret = _scalars(rnd, 8)
    idx = [rnd.randrange(8) for _ in range(64)]
    pks, sigs = _sign(eng, B, impl, 0, [secret[k] for k in idx], [b"m"] * 64)
    kb = _sign(eng, B, impl, 0, secret, [b"m"] * 8)[0]
    ks = eng.key_set(impl, kb)
    try:
        for call in (lambda: eng.verify_batch_keyed(ks, 0, idx, sigs, [b"m"] * 64),
                     lambda: eng.verify_batch_grouped_keyed(ks, 0, idx, sigs, [0] * 64, [b"m"])):
            assert call().tolist() == [0] * 64
            k = eng.last_kernel_ms()
            assert k["k_decode_pk"][1] == 0 and k["k_subgroup_check_pk"][1] == 0
            assert k["k_decode_sig"][1] == 1
        eng.verify_batch(impl, 0, pks, sigs, [b"m"] * 64)   # the unkeyed call still decodes its keys
        assert eng.last_kernel_ms()["k_decode_pk"][1] == 1
    finally:
        ks.close()


def test_ids_and_indices_are_checked_then_the_context_still_verifies(B):
    e, other = B.Engine([0]), B.Engine([0])
    try:
        rnd = random.Random(12)
        secret = _scalars(rnd, 4)
        idx = [3, 1, 1, 0, 2, 3]
        pks, sigs = _sign(e, B, 2, 0, [secret[k] for k in idx], [b"x"] * 6)
        kb = _sign(e, B, 2, 0, secret, [b"x"] * 4)[0]
        ks, gone, foreign = e.key_set(2, kb), e.key_set(2, kb), other.key_set(2, kb)
        assert ks.id and gone.id and foreign.id and len({ks.id, gone.id, foreign.id}) == 3
        gone_id = gone.id
        gone.close()
        gone.close()   # idempotent
        for ident in (gone_id, foreign.id, 0):
            fake = B.KeySet(e, 2, ident, np.zeros(4, dtype=np.uint8))
            with pytest.raises(B.EngineError, match=r"\(-1\)"):
                e.verify_batch_keyed(fake, 0, idx, sigs, [b"x"] * 6)
            with pytest.raises(B.EngineError, match=r"\(-1\)"):
                e.verify_batch_grouped_keyed(fake, 0, idx, sigs, [0] * 6, [b"x"])
            with pytest.raises(B.EngineError, match=r"\(-1\)"):
                e._check(e._lib.blsgpu_keyset_destroy(e._ctx, ident), "blsgpu_keyset_destroy")
        with pytest.raises(B.EngineError, match=r"key_idx\[4\]"):
            e.verify_batch_keyed(ks, 0, [3, 1, 1, 0, 4, 3], sigs, [b"x"] * 6)
        with pytest.raises(B.EngineError, match=r"key_idx\[1\]"):
            e.verify_batch_grouped_keyed(ks, 0, [3, 99, 1, 0, 2, 3], sigs, [0] * 6, [b"x"])
        sigs[2] = sigs[0]
        assert e.verify_batch_keyed(ks, 0, idx, sigs, [b"x"] * 6).tolist() == [0, 0, 1, 0, 0, 0]
        assert e.verify_batch_grouped_keyed(ks, 0, idx, sigs, [0] * 6, [b"x"]).tolist() == [0, 0, 1, 0, 0, 0]
        assert other.verify_batch_keyed(foreign, 0, idx, sigs, [b"x"] * 6).tolist() == [0, 0, 1, 0, 0, 0]
        empty = e.key_set(2, [])
        assert len(empty) == 0 and empty.id
        assert e.verify_batch_keyed(empty, 0, [], [], []).tolist() == []
        with pytest.raises(B.EngineError, match=r"key_idx\[0\]"):
            e.verify_batch_keyed(empty, 0, [0], sigs[:1], [b"x"])
        # the set survives a call that regrows the arena
        n = 1 << 17
        data, off = B.pack_messages([b"big"] * n)
        keys = np.frombuffer(b"".join(_scalars(rnd, 1)) * n, dtype=np.uint8)
        bpk, bsg = e.testdata_sign(2, 0, keys, data, off)
        assert not e.verify_batch_packed(2, 0, bpk, bsg, data, off).any()
        assert e.verify_batch_keyed(ks, 0, idx, sigs, [b"x"] * 6).tolist() == [0, 0, 1, 0, 0, 0]
        ks.close()
    finally:
        other.close()
        e.close()   # closes the live empty set with the context
    assert empty.id and empty.close() is None and empty.id == 0


def test_a_large_set_frees_its_device_memory(B, scale):
    import torch
    kb = np.tile(scale[0], 16)   # 2^20 keys
    e = B.Engine([0])
    try:
        e.key_set(2, kb[:48 * 4096]).close()   # loads the decode kernels before the measurement
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info(0)[0]
        ks = e.key_set(2, kb)
        assert len(ks) == 1 << 20 and not ks.status.any()
        assert torch.cuda.mem_get_info(0)[0] < free0 - 100 * 2 ** 20
        ks.close()
        assert abs(torch.cuda.mem_get_info(0)[0] - free0) <= 2 * 2 ** 20
        live = [e.key_set(2, kb[:48 * 1000]), e.key_set(2, kb[:48 * 10])]
    finally:
        e.close()   # frees the live sets; closing them afterwards is a no-op
    for ks in live:
        ks.close()
    assert abs(torch.cuda.mem_get_info(0)[0] - free0) <= 2 * 2 ** 20


def test_two_devices_give_the_statuses_of_one(B, scale):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    kb, key_idx, sg, msg_idx, data, off, data_i, off_i = scale
    n = 50_000
    bad = sorted(random.Random(2).sample(range(n), 7))
    planted = _plant(sg[:96 * n], n, bad)
    out = []
    for devs in ([0], [0, 1]):
        e = B.Engine(devs)
        try:
            ks = e.key_set(2, kb)
            out.append((e.verify_batch_keyed_packed(ks, 0, key_idx[:n], planted, data_i[:int(off_i[n])], off_i[:n + 1]).tolist(),
                        e.verify_batch_grouped_keyed_packed(ks, 0, key_idx[:n], planted, msg_idx[:n], data, off).tolist()))
        finally:
            e.close()
    assert out[0] == out[1] and [i for i, s in enumerate(out[0][0]) if s] == bad

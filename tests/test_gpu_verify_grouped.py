"""blsgpu_verify_batch_grouped: n signatures over q shared messages.  Every status must equal blsgpu_verify_batch's on the
same items with their messages written out (and, on a sample, the big-int oracle); rejections must be exact whatever the
grouping, including wrong signatures whose errors cancel in an unweighted sum."""
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import bls_oracle as O

L = 96  # items per leaf (GROUPED_LEAF in blsgpu.cu)


@pytest.fixture(scope="module")
def eng():
    import blsful_b200 as B
    e = B.Engine([0])
    yield e
    e.close()


@pytest.fixture(scope="module")
def B():
    import blsful_b200
    return blsful_b200


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
    """-P for a compressed (Modern) point that is not the identity: the sign flag flips"""
    return bytes([enc[0] ^ 0x20]) + enc[1:]


def _scalars(rnd, n):
    return np.frombuffer(b"".join(rnd.randrange(1, O.R).to_bytes(32, "big") for _ in range(n)), dtype=np.uint8)


def _groups(impl):
    return (1, 2) if impl == 2 else (2, 1)   # (public-key group, signature group)


def _sign(eng, B, impl, scheme, keys, msgs):
    """(pks, sigs) as lists of Modern encodings, item i signed with keys[i] over msgs[i]"""
    pks, sigs = eng.testdata_sign(impl, scheme, keys, *B.pack_messages(msgs))
    pl, sl = B.pk_len(impl), B.sig_len(impl)
    return [pks[i * pl:(i + 1) * pl].tobytes() for i in range(len(msgs))], [sigs[i * sl:(i + 1) * sl].tobytes() for i in range(len(msgs))]


def _expanded(eng, impl, scheme, pks, sigs, idx, msgs, fmt):
    return eng.verify_batch(impl, scheme, pks, sigs, [msgs[j] for j in idx], fmt)


GROUP_SIZES = [0, 1, 5, 6, 7, L - 1, L, L + 1, 6 * L + 1]


@pytest.mark.parametrize("fmt", [O.MODERN, O.LEGACY])
@pytest.mark.parametrize("impl", [2, 1])
def test_mixed_batch_equals_verify_batch_and_the_oracle(eng, B, impl, fmt):
    pkg, sgg = _groups(impl)
    pl, sl = B.pk_len(impl), B.sig_len(impl)
    for scheme in (0, 1, 2):
        rnd = random.Random(100 * impl + 10 * fmt + scheme)
        msgs = [b"grouped/%d/%d" % (scheme, j) for j in range(len(GROUP_SIZES))] + [b""]
        sizes = GROUP_SIZES + [4]                                  # the empty message signed by 4 items
        idx = [j for j, s in enumerate(sizes) for _ in range(s)]
        n = len(idx)
        keys = _scalars(rnd, n)
        pks, sigs = _sign(eng, B, impl, scheme, keys, [msgs[j] for j in idx])
        # another message of the batch signed by the same keys: "signature over another message"
        _, sigs_other = _sign(eng, B, impl, scheme, keys, [msgs[(j + 1) % len(msgs)] for j in idx])
        big = [i for i in range(n) if idx[i] == len(GROUP_SIZES) - 1]     # the 6L+1 group
        names = {}
        plan = [("undecodable_pk", big[3]), ("undecodable_sig", big[100]), ("header", big[200]), ("identity_pk", big[300]),
                ("identity_sig", big[400]), ("other_message", big[500]), ("other_key", big[501])]
        for name, i in plan:
            names[name] = i
        pks[big[3]] = _off_curve(pkg)
        sigs[big[100]] = _off_curve(sgg)
        pks[big[300]] = _ident(pl)
        sigs[big[400]] = _ident(sl)
        sigs[big[500]] = sigs_other[big[500]]
        sigs[big[501]] = sigs[big[502]]
        i6 = [i for i in range(n) if idx[i] == GROUP_SIZES.index(L)]
        names["other_message_L"] = i6[40]
        sigs[i6[40]] = sigs_other[i6[40]]
        # a valid item whose pk (and signature) appears twice in one group
        pks.append(pks[i6[7]]); sigs.append(sigs[i6[7]]); idx.append(idx[i6[7]])
        names["twice_a"], names["twice_b"] = i6[7], len(idx) - 1
        if fmt == O.LEGACY:
            def conv(group, encs):
                st, outs = eng.recode_points(group, encs, O.MODERN, O.LEGACY)
                return [o if s == 0 else O.modern_to_legacy(e) for e, s, o in zip(encs, st.tolist(), outs)]
            modern = sigs[big[200]]
            pks, sigs = conv(pkg, pks), conv(sgg, sigs)
            sigs[big[200]] = modern if modern[0] & 0x20 else _neg(modern)   # Modern bytes with the y-flag: LegacyFormatError
        else:
            sigs[big[200]] = bytes([sigs[big[200]][0] & 0x7F]) + sigs[big[200]][1:]   # no compression flag
        perm = list(range(len(idx)))
        rnd.shuffle(perm)                                           # items interleaved: msg_idx unsorted
        pks, sigs, idx = [pks[p] for p in perm], [sigs[p] for p in perm], [idx[p] for p in perm]
        where = {name: perm.index(i) for name, i in names.items()}
        st = eng.verify_batch_grouped(impl, scheme, pks, sigs, idx, msgs, fmt)
        want = _expanded(eng, impl, scheme, pks, sigs, idx, msgs, fmt)
        assert st.tolist() == want.tolist(), [(i, a, b) for i, (a, b) in enumerate(zip(st.tolist(), want.tolist())) if a != b]
        got = {name: int(st[i]) for name, i in where.items()}
        assert got["undecodable_pk"] in (O.ERR_DESERIALIZE, O.ERR_LEGACY_FORMAT)
        assert got["undecodable_sig"] in (O.ERR_DESERIALIZE, O.ERR_LEGACY_FORMAT)
        assert got["header"] in (O.ERR_DESERIALIZE, O.ERR_LEGACY_FORMAT)
        assert got["identity_pk"] == O.ERR_PK_IDENTITY and got["identity_sig"] == O.ERR_SIG_IDENTITY
        assert got["other_message"] == got["other_key"] == got["other_message_L"] == 1
        assert got["twice_a"] == got["twice_b"] == 0
        assert sum(1 for s in st.tolist() if s) == 8
        if scheme == 0:   # a sample end to end against the big-int oracle
            for name in ("other_key", "twice_b", "identity_pk"):
                i = where[name]
                assert O.verify(impl, scheme, fmt, pks[i], sigs[i], msgs[idx[i]]) == st[i], name


@pytest.mark.parametrize("impl", [2, 1])
def test_errors_that_cancel_without_weights_are_both_rejected(eng, B, impl):
    """sig_a + D and sig_b - D: their unweighted sum is valid.  Both must be INVALID_SIGNATURE with a and b in one leaf,
    in two leaves of one message, and under two messages.  5,000 items: the bucket route of the signature side."""
    sgg = _groups(impl)[1]
    rnd = random.Random(77 + impl)
    q = 20
    msgs = [b"cancel/%d" % j for j in range(q)]
    idx = [j % q for j in range(4600)] + [0] * 400              # message 0: 630 items, several leaves
    n = len(idx)
    pks, sigs = _sign(eng, B, impl, 0, _scalars(rnd, n), [msgs[j] for j in idx])
    D = _sign(eng, B, impl, 0, _scalars(rnd, 1), [b"D"])[1][0]
    m0 = [i for i in range(n) if idx[i] == 0]
    m3 = [i for i in range(n) if idx[i] == 3]
    for a, b in ((m0[1], m0[2]), (m0[10], m0[-1]), (m3[5], m0[300])):  # one leaf; two leaves of a message; two messages
        bad = list(sigs)
        bad[a] = eng.sum_points(sgg, [sigs[a], D])
        bad[b] = eng.sum_points(sgg, [sigs[b], _neg(D)])
        st = eng.verify_batch_grouped(impl, 0, pks, bad, idx, msgs)
        assert [i for i in range(n) if st[i]] == sorted([a, b]) and st[a] == st[b] == 1


@pytest.fixture(scope="module")
def million(eng, B):
    """2^20 G2Impl items, Basic: signed over 1 message and over 1,000 messages (seeded message per item)"""
    rnd = random.Random(2026)
    n = 1 << 20
    keys = _scalars(rnd, n)
    out = {}
    for q in (1, 1000):
        msgs = [b"million/%d/%d" % (q, j) for j in range(q)]
        idx = np.array([rnd.randrange(q) for _ in range(n)], dtype=np.uint32)
        data_i, off_i = B.pack_messages([msgs[j] for j in idx.tolist()])
        pk, sg = eng.testdata_sign(2, 0, keys, data_i, off_i)
        data, off = B.pack_messages(msgs)
        out[q] = (pk, sg, idx, data, off)
    return out


def _plant(sg, n, bad):
    s = sg.copy().reshape(n, 96)
    for i in bad:       # another item's signature: a valid point that fails its own equation
        s[i] = sg.reshape(n, 96)[(i + 1) % n]
    return s.reshape(-1)


@pytest.mark.parametrize("q", [1, 1000])
def test_failure_search_is_exact_at_scale(eng, B, million, q):
    pk, sg, idx, data, off = million[q]
    n = idx.size
    rnd = random.Random(q)
    for nbad in (0, 1, 1000):
        bad = sorted(rnd.sample(range(n), nbad))
        st = eng.verify_batch_grouped_packed(2, 0, pk, _plant(sg, n, bad), idx, data, off)
        assert np.flatnonzero(st).tolist() == bad and (st[bad] == 1).all()
    e2 = B.Engine([0])
    try:
        bad = sorted(rnd.sample(range(n), 1000))
        planted = _plant(sg, n, bad)
        e2.set_rlc_bits(128)
        st = e2.verify_batch_grouped_packed(2, 0, pk, planted, idx, data, off)
        assert np.flatnonzero(st).tolist() == bad
        e2.set_rlc_bits(64)
        e2.set_rlc_salt(bytes(range(32)))
        pinned = e2.verify_batch_grouped_packed(2, 0, pk, planted, idx, data, off)
        fresh = eng.verify_batch_grouped_packed(2, 0, pk, planted, idx, data, off)
        assert pinned.tolist() == fresh.tolist() == st.tolist()
    finally:
        e2.close()


def test_several_miller_passes(eng, B, million, monkeypatch):
    """More leaves than one pass of the Miller kernels holds (BLSGPU_M6_CHUNK=1200): 130,000 items over 1,000 messages"""
    pk, sg, idx, data, off = million[1000]
    n = 130_000
    pk, sg, idx = pk[:48 * n], sg[:96 * n], idx[:n]
    assert n > 1200 * L
    rnd = random.Random(9)
    bad = sorted(rnd.sample(range(n), 25))
    monkeypatch.setenv("BLSGPU_M6_CHUNK", "1200")
    st = eng.verify_batch_grouped_packed(2, 0, pk, _plant(sg, n, bad), idx, data, off)
    assert np.flatnonzero(st).tolist() == bad


def test_argument_errors_then_the_context_still_verifies(eng, B):
    rnd = random.Random(3)
    msgs = [b"a", b"bb", b"ccc"]
    idx = [2, 0, 1, 0, 2, 2]
    pks, sigs = _sign(eng, B, 2, 0, _scalars(rnd, len(idx)), [msgs[j] for j in idx])
    pk, sg = np.frombuffer(b"".join(pks), dtype=np.uint8), np.frombuffer(b"".join(sigs), dtype=np.uint8)
    data, off = B.pack_messages(msgs)
    ix = np.array(idx, dtype=np.uint32)
    assert eng.verify_batch_grouped_packed(2, 0, pk, sg, ix, data, off).tolist() == [0] * 6
    with pytest.raises(B.EngineError, match=r"\(-1\)"):         # msg_idx >= q
        eng.verify_batch_grouped_packed(2, 0, pk, sg, np.array([2, 0, 1, 0, 3, 2], dtype=np.uint32), data, off)
    bad_off = off.copy()
    bad_off[1], bad_off[2] = bad_off[2], bad_off[1]
    with pytest.raises(B.EngineError, match=r"\(-1\)"):         # decreasing msg_off
        eng.verify_batch_grouped_packed(2, 0, pk, sg, ix, data, bad_off)
    with pytest.raises(B.EngineError, match=r"\(-1\)"):         # a null buffer (no public keys)
        eng.verify_batch_grouped_packed(2, 0, np.zeros(0, dtype=np.uint8), sg, ix, data, off)
    with pytest.raises(B.EngineError, match=r"\(-1\)"):         # a null msgs with non-empty messages
        eng.verify_batch_grouped_packed(2, 0, pk, sg, ix, np.zeros(0, dtype=np.uint8), off)
    sigs[4] = sigs[5]
    st = eng.verify_batch_grouped(2, 0, pks, sigs, idx, msgs)
    assert st.tolist() == [0, 0, 0, 0, 1, 0]
    assert eng.verify_batch_grouped(2, 0, [], [], [], msgs).tolist() == []

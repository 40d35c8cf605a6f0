"""Multi-signatures over signer subsets: every status of blsgpu_verify_multisig_batch[_keyed] must equal blsgpu_sum_points of
the set's keys followed by blsgpu_verify_batch on that sum (and, on a sample, the big-int oracle); keyed equals unkeyed;
blsgpu_sum_points_batch equals per-set blsgpu_sum_points byte for byte; sizes at the chunk and level boundaries; the exact
failure search; no launch per set; argument errors."""
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


def _groups(impl):
    return (1, 2) if impl == 2 else (2, 1)   # (public-key group, signature group)


def _same(got, want):
    assert list(got) == list(want), [(j, x, y) for j, (x, y) in enumerate(zip(list(got), list(want))) if x != y]


def _be32(ks):
    return np.frombuffer(b"".join((k % O.R).to_bytes(32, "big") for k in ks), dtype=np.uint8)


def _secrets(rng, k):
    """k random scalars as 32-byte big-endian rows (192 random bits, odd) and as ints"""
    s = np.zeros((k, 32), dtype=np.uint8)
    s[:, 8:] = rng.integers(0, 256, size=(k, 24), dtype=np.uint8)
    s[:, 31] |= 1
    return s, [int.from_bytes(r.tobytes(), "big") for r in s]


def _multisigs(eng, B, impl, scheme, sums, msgs):
    """[sum_j] H(framed msg_j): the valid multi-signature of a set whose secret keys add up to sum_j (MessageAugmentation
    frames with [sum_j] G, the set's multi key)"""
    return eng.testdata_sign(impl, scheme, _be32(sums), *B.pack_messages(msgs))[1]


def _sum_points_raw(eng, group, fmt, pts):
    """blsgpu_sum_points without the mirror's exception: (status, bad index, sum bytes)"""
    L = 48 if group == 1 else 96
    a = np.frombuffer(b"".join(pts), dtype=np.uint8) if pts else np.zeros(0, dtype=np.uint8)
    out, st, bad = np.zeros(L, dtype=np.uint8), np.zeros(1, dtype=np.uint8), np.full(1, -1, dtype=np.int64)
    rc = eng._lib.blsgpu_sum_points(eng._ctx, group, fmt, len(pts), a.ctypes.data if a.size else None, out.ctypes.data, st.ctypes.data,
                                    bad.ctypes.data)
    assert rc == 0
    return int(st[0]), int(bad[0]), out.tobytes()


def _composed(eng, B, impl, scheme, fmt, keys, sig, msg):
    """the status blsgpu_sum_points + blsgpu_verify_batch give for one multi-signature"""
    st, _, s = _sum_points_raw(eng, _groups(impl)[0], fmt, keys)
    if st != 0:
        return st
    return int(eng.verify_batch(impl, scheme, [s], [sig], [msg], fmt)[0])


N_VALID = 8
DUP, OFF_CURVE, HEADER, IDENT, NEG = 8, 9, 10, 11, 12   # key 2's bytes again, off-curve, bad header, identity, -key 0
# (members, signature: "own" = the set's valid multi-signature on msgs[0] or the one of another row, message to verify)
SETS = [
    ([0, 1, 2, 3, 4], "own", 0),           # 0 valid
    ([4, 3, 2, 1, 0, 5], "own", 0),        # 1 valid, unsorted
    ([1, 2, 3], 0, 0),                     # 2 a wrong signature
    ([0, 1, 2, 3, 4], "own", 1),           # 3 a wrong message
    ([0, 1, 2, 3], 0, 0),                  # 4 a member missing
    ([2, 5, 2, 6], "own", 0),              # 5 the same index twice (counted twice)
    ([2, DUP, 7], "own", 0),               # 6 two set entries with equal bytes
    ([0, OFF_CURVE, 1], 0, 0),             # 7 an off-curve key
    ([0, 1, HEADER], 0, 0),                # 8 a bad-header key
    ([HEADER, OFF_CURVE, 0], 0, 0),        # 9 two bad keys: the first in member order decides
    ([IDENT, 0], "own", 0),                # 10 an identity member adds nothing
    ([0, NEG], 0, 0),                      # 11 P and -P: the sum is the identity
    ([], "ident", 0),                      # 12 empty, identity signature
    ([], 0, 0),                            # 13 empty, non-identity signature
    ([0, 1], "undecodable", 0),            # 14 an undecodable signature
    ([6, 7, 1, 0, 3, 5, 4, 2], "own", 0),  # 15 every valid key
]
WANT = {0: 0, 1: 0, 2: O.ERR_INVALID_SIGNATURE, 3: O.ERR_INVALID_SIGNATURE, 4: O.ERR_INVALID_SIGNATURE, 5: 0, 6: 0, 10: 0,
        11: O.ERR_PK_IDENTITY, 12: O.ERR_SIG_IDENTITY, 13: O.ERR_PK_IDENTITY, 15: 0}


@pytest.mark.parametrize("impl,fmt", [(2, O.MODERN), (2, O.LEGACY), (1, O.MODERN)])
def test_mixed_sets_equal_sum_then_verify_and_the_oracle(eng, B, impl, fmt):
    C = O.IMPLS[impl]
    pkg, sgg = _groups(impl)
    pl, sl = B.pk_len(impl), B.sig_len(impl)
    rnd = random.Random(91 + 10 * impl + fmt)
    sks = [rnd.randrange(1, O.R) for _ in range(N_VALID)]
    kb = [C.pk_ser(O.sk_to_pk(impl, sk), fmt) for sk in sks]
    hdr = C.pk_ser(O.sk_to_pk(impl, sks[0]), O.MODERN)
    neg = C.pk_ser(C.pk_neg(O.sk_to_pk(impl, sks[0])), fmt)
    if fmt == O.LEGACY:
        ident = eng.recode_points(pkg, [_ident(pl)], O.MODERN, O.LEGACY)[1][0]
        kb += [kb[2], O.modern_to_legacy(_off_curve(pkg)), hdr if hdr[0] & 0x20 else bytes([hdr[0] ^ 0x20]) + hdr[1:], ident, neg]
        bad_sig = O.modern_to_legacy(_off_curve(sgg))
        ident_sig = eng.recode_points(sgg, [_ident(sl)], O.MODERN, O.LEGACY)[1][0]
    else:
        kb += [kb[2], _off_curve(pkg), bytes([hdr[0] & 0x7F]) + hdr[1:], _ident(pl), neg]
        bad_sig, ident_sig = _off_curve(sgg), _ident(sl)
    sk_of = sks + [sks[2], 0, 0, 0, -sks[0]]
    ks = eng.key_set(impl, kb, fmt)
    try:
        assert ks.status[OFF_CURVE] in (O.ERR_DESERIALIZE, O.ERR_LEGACY_FORMAT) and ks.status[HEADER] in (O.ERR_DESERIALIZE, O.ERR_LEGACY_FORMAT)
        msgs = [b"multisig %d %d" % (impl, fmt), b"another message"]
        idx_sets = [m for m, _, _ in SETS]
        key_sets = [[kb[k] for k in m] for m in idx_sets]
        qmsgs = [msgs[m] for _, _, m in SETS]
        for scheme in (0, 1, 2):
            own = _multisigs(eng, B, impl, scheme, [sum(sk_of[k] for k in m) or 1 for m in idx_sets], [msgs[0]] * len(SETS))
            own = [own[j * sl:(j + 1) * sl].tobytes() for j in range(len(SETS))]
            if fmt == O.LEGACY:
                own = eng.recode_points(sgg, own, O.MODERN, O.LEGACY)[1]
            sigs = [own[j] if s == "own" else ident_sig if s == "ident" else bad_sig if s == "undecodable" else own[s]
                    for j, (_, s, _) in enumerate(SETS)]
            unkeyed = eng.verify_multisig_batch(impl, scheme, key_sets, sigs, qmsgs, fmt)
            keyed = eng.verify_multisig_batch_keyed(ks, scheme, idx_sets, sigs, qmsgs, fmt)
            _same(keyed, unkeyed)
            _same(unkeyed, [_composed(eng, B, impl, scheme, fmt, key_sets[j], sigs[j], qmsgs[j]) for j in range(len(SETS))])
            w = unkeyed.tolist()
            assert {j: w[j] for j in WANT} == WANT
            for j in (7, 8, 9, 14):
                assert w[j] in (O.ERR_DESERIALIZE, O.ERR_LEGACY_FORMAT), j
            assert w[9] == ks.status[HEADER]
            if scheme == 1:   # a sample end to end against the big-int oracle: O.sum_points, then O.verify on the sum
                for j in (0, 2, 10, 11):
                    st, s, _ = O.sum_points(pkg, fmt, key_sets[j])
                    assert st == 0
                    assert O.verify(impl, scheme, fmt, s, sigs[j], qmsgs[j]) == w[j], j
    finally:
        ks.close()


SIZES = [0, 1, 15, 16, 17, 255, 256, 257, 4097]


@pytest.mark.parametrize("impl", [2, 1])
def test_set_sizes_at_the_chunk_and_level_boundaries(eng, B, impl):
    rng = np.random.default_rng(300 + impl)
    k = 5000
    sec, ints = _secrets(rng, k)
    kb, _ = eng.testdata_sign(impl, 0, sec.reshape(-1), *B.pack_messages([b""] * k))
    pl, sl = B.pk_len(impl), B.sig_len(impl)
    idx_sets = [rng.integers(0, k, size=s, dtype=np.uint32) for s in SIZES]
    q = len(SIZES)
    msgs = [b"sizes %d" % j for j in range(q)]
    ks = eng.key_set(impl, kb)
    try:
        for scheme in (0, 2):
            sigs = _multisigs(eng, B, impl, scheme, [sum(ints[i] for i in m) or 1 for m in idx_sets], msgs).reshape(q, sl)
            sigs[0] = np.frombuffer(_ident(sl), dtype=np.uint8)   # the empty set: identity signature
            koff = np.concatenate([[0], np.cumsum(SIZES)]).astype(np.uint64)
            idx = np.concatenate(idx_sets).astype(np.uint32)
            data, off = B.pack_messages(msgs)
            got = eng.verify_multisig_batch_keyed_packed(ks, scheme, koff, idx, sigs.reshape(-1), data, off)
            assert got.tolist() == [O.ERR_SIG_IDENTITY] + [0] * (q - 1)
            pk = kb.reshape(k, pl)[idx].reshape(-1)
            _same(eng.verify_multisig_batch_packed(impl, scheme, koff, pk, sigs.reshape(-1), data, off), got)
            sigs[0] = sigs[1]   # the empty set: a non-identity signature
            assert eng.verify_multisig_batch_keyed_packed(ks, scheme, koff, idx, sigs.reshape(-1), data, off)[0] == O.ERR_PK_IDENTITY
            # one member less in every set of two or more: each multi-signature fails on its own
            short = [m[1:] for m in idx_sets]
            koff_s = np.concatenate([[0], np.cumsum([len(m) for m in short])]).astype(np.uint64)
            got = eng.verify_multisig_batch_keyed_packed(ks, scheme, koff_s, np.concatenate(short).astype(np.uint32), sigs.reshape(-1), data, off)
            assert got.tolist() == [O.ERR_PK_IDENTITY, O.ERR_PK_IDENTITY] + [O.ERR_INVALID_SIGNATURE] * (q - 2)
    finally:
        ks.close()


def test_one_large_set_beside_many_small_ones(eng, B):
    rng = np.random.default_rng(65539)
    k = (1 << 16) + 3
    sec, ints = _secrets(rng, k)
    kb, _ = eng.testdata_sign(2, 0, sec.reshape(-1), *B.pack_messages([b""] * k))
    idx_sets = [rng.permutation(k).astype(np.uint32)] + [rng.integers(0, k, size=3, dtype=np.uint32) for _ in range(1000)]
    q = len(idx_sets)
    msgs = [b"large beside small %d" % j for j in range(q)]
    sigs = _multisigs(eng, B, 2, 2, [sum(ints[i] for i in m) for m in idx_sets], msgs)
    koff = np.concatenate([[0], np.cumsum([len(m) for m in idx_sets])]).astype(np.uint64)
    idx = np.concatenate(idx_sets)
    data, off = B.pack_messages(msgs)
    ks = eng.key_set(2, kb)
    try:
        got = eng.verify_multisig_batch_keyed_packed(ks, 2, koff, idx, sigs, data, off)
        assert got.tolist() == [0] * q
        _same(eng.verify_multisig_batch_packed(2, 2, koff, kb.reshape(k, 48)[idx].reshape(-1), sigs, data, off), got)
        swapped = sigs.reshape(q, 96).copy()
        swapped[[0, 500]] = swapped[[500, 0]]
        got = eng.verify_multisig_batch_keyed_packed(ks, 2, koff, idx, swapped.reshape(-1), data, off)
        assert np.nonzero(got)[0].tolist() == [0, 500]
    finally:
        ks.close()


@pytest.mark.parametrize("group", [1, 2])
@pytest.mark.parametrize("fmt", [O.MODERN, O.LEGACY])
def test_sum_points_batch_equals_per_set_sum_points(eng, B, group, fmt):
    rng = np.random.default_rng(40 + 2 * group + fmt)
    L = 48 if group == 1 else 96
    impl = 2 if group == 1 else 1   # the impl whose public keys are in `group`
    n = sum(SIZES)
    sec, _ = _secrets(rng, n)
    pts, _ = eng.testdata_sign(impl, 0, sec.reshape(-1), *B.pack_messages([b""] * n))
    if fmt == O.LEGACY:
        pts = eng.recode_points_packed(group, pts, O.MODERN, O.LEGACY)
    sets, o = [], 0
    for s in SIZES:
        sets.append([pts[(o + i) * L:(o + i + 1) * L].tobytes() for i in range(s)])
        o += s
    bad = _off_curve(group) if fmt == O.MODERN else O.modern_to_legacy(_off_curve(group))
    ident = _ident(L) if fmt == O.MODERN else eng.recode_points(group, [_ident(L)], O.MODERN, O.LEGACY)[1][0]
    sets[3][7] = bad                        # a bad point inside a chunk
    sets[5][200], sets[5][16] = bad, bad    # two bad points in different chunks: the first decides
    sets[8][4096] = bad                     # the last point of the largest set
    sets[6][:3] = [ident] * 3               # identity points add nothing
    sets.append([sets[1][0], O.IMPLS[impl].pk_ser(O.IMPLS[impl].pk_neg(O.IMPLS[impl].pk_deser(sets[1][0], fmt)), fmt)])   # P + -P
    st, bad_idx, outs = eng.sum_points_batch(group, sets, fmt)
    for j, s in enumerate(sets):
        want = _sum_points_raw(eng, group, fmt, s)
        assert (int(st[j]), int(bad_idx[j])) == want[:2], j
        assert outs[j] == (want[2] if want[0] == 0 else bytes(L)), j
    assert [int(bad_idx[j]) for j in (3, 5, 8)] == [7, 16, 4096]
    one = eng.sum_points_batch(group, [sets[7]], fmt)
    assert one[2][0] == _sum_points_raw(eng, group, fmt, sets[7])[2]


@pytest.mark.parametrize("bits", [64, 128])
def test_the_failure_search_returns_exactly_the_planted_set(B, bits):
    e = B.Engine([0])
    try:
        e.set_rlc_bits(bits)
        rng = np.random.default_rng(1000 + bits)
        k, q = 2048, 1000
        sec, ints = _secrets(rng, k)
        kb, _ = e.testdata_sign(2, 0, sec.reshape(-1), *B.pack_messages([b""] * k))
        sizes = rng.integers(1, 40, size=q)
        idx_sets = [rng.choice(k, s, replace=False).astype(np.uint32) for s in sizes]
        msgs = [b"failure path %d" % j for j in range(q)]
        sigs = _multisigs(e, B, 2, 2, [sum(ints[i] for i in m) for m in idx_sets], msgs).reshape(q, 96)
        planted = sorted(random.Random(bits).sample(range(q), 13))
        for j in planted:
            sigs[j] = sigs[(j + 1) % q]
        koff = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
        idx = np.concatenate(idx_sets)
        data, off = B.pack_messages(msgs)
        ks = e.key_set(2, kb)
        got = e.verify_multisig_batch_keyed_packed(ks, 2, koff, idx, sigs.reshape(-1), data, off)
        assert np.nonzero(got)[0].tolist() == planted
        assert set(got[planted].tolist()) == {O.ERR_INVALID_SIGNATURE}
        _same(e.verify_multisig_batch_packed(2, 2, koff, kb.reshape(k, 48)[idx].reshape(-1), sigs.reshape(-1), data, off), got)
        ks.close()
    finally:
        e.close()


def test_no_launch_per_set(eng, B):
    """launches of a keyed call minus those of blsgpu_verify_batch on the same q pre-summed keys: the same at q = 10 and
    q = 10,000 (sets of 400)"""
    rng = np.random.default_rng(400)
    k, mem = 4096, 400
    sec, ints = _secrets(rng, k)
    kb, _ = eng.testdata_sign(2, 0, sec.reshape(-1), *B.pack_messages([b""] * k))
    ks = eng.key_set(2, kb)
    try:
        extra = []
        for q in (10, 10_000):
            idx = rng.integers(0, k, size=q * mem, dtype=np.uint32)
            sums = [sum(ints[i] for i in idx[j * mem:(j + 1) * mem].tolist()) for j in range(q)]
            qm = rng.integers(0, 256, size=(q, 32), dtype=np.uint8)
            off = np.arange(q + 1, dtype=np.uint64) * 32
            agg_pk, sigs = eng.testdata_sign(2, 2, _be32(sums), qm.reshape(-1), off)
            koff = np.arange(q + 1, dtype=np.uint64) * mem
            c0 = eng.launch_count()
            st = eng.verify_multisig_batch_keyed_packed(ks, 2, koff, idx, sigs, qm.reshape(-1), off)
            c1 = eng.launch_count()
            st_b = eng.verify_batch_packed(2, 2, agg_pk, sigs, qm.reshape(-1), off)
            c2 = eng.launch_count()
            assert st.tolist() == [0] * q and st_b.tolist() == [0] * q
            extra.append((c1 - c0) - (c2 - c1))
        assert extra[0] == extra[1], extra
    finally:
        ks.close()


def test_argument_errors_then_the_context_still_verifies(B):
    e = B.Engine([0])
    try:
        rnd = random.Random(17)
        secret = _be32([rnd.randrange(1, O.R) for _ in range(4)])
        kb, _ = e.testdata_sign(2, 0, secret, *B.pack_messages([b""] * 4))
        total = sum(int.from_bytes(secret[32 * i:32 * i + 32].tobytes(), "big") for i in range(4))
        sig = _multisigs(e, B, 2, 0, [total], [b"x"]).tobytes()
        ks, gone = e.key_set(2, kb), e.key_set(2, kb)
        gone_id = gone.id
        gone.close()
        for ident in (gone_id, 0, 987654321):
            fake = B.KeySet(e, 2, ident, np.zeros(4, dtype=np.uint8))
            with pytest.raises(B.EngineError, match=r"\(-1\)"):
                e.verify_multisig_batch_keyed(fake, 0, [[0, 1, 2, 3]], [sig], [b"x"])
        with pytest.raises(B.EngineError, match=r"key_idx\[5\]"):
            e.verify_multisig_batch_keyed(ks, 0, [[0, 1], [2, 3, 1, 4]], [sig] * 2, [b"x"] * 2)
        data, off = B.pack_messages([b"x", b"x"])
        sg2 = np.frombuffer(sig * 2, dtype=np.uint8)
        with pytest.raises(B.EngineError, match=r"non-decreasing"):   # key_off decreasing
            e.verify_multisig_batch_keyed_packed(ks, 0, np.array([0, 3, 2], dtype=np.uint64), np.zeros(2, dtype=np.uint32), sg2, data, off)
        with pytest.raises(B.EngineError, match=r"non-decreasing"):
            e.verify_multisig_batch_packed(2, 0, np.array([0, 3, 2], dtype=np.uint64), np.tile(kb[:48], 2), sg2, data, off)
        with pytest.raises(B.EngineError, match=r"non-decreasing"):
            e.sum_points_batch_packed(1, np.array([0, 3, 2], dtype=np.uint64), np.tile(kb[:48], 2))
        bad_moff = np.array([0, 2, 1], dtype=np.uint64)   # msg_off decreasing
        with pytest.raises(B.EngineError, match=r"non-decreasing"):
            e.verify_multisig_batch_keyed_packed(ks, 0, np.array([0, 1, 2], dtype=np.uint64), np.zeros(2, dtype=np.uint32), sg2, data, bad_moff)
        lib, ctx = e._lib, e._ctx
        big = np.array([0, 1 << 32], dtype=np.uint64)   # a set of 2^32 members, a message of 2^32 bytes
        one = np.array([0, 1], dtype=np.uint64)
        idx1, st1, msg1 = np.zeros(1, dtype=np.uint32), np.zeros(1, dtype=np.uint8), np.zeros(1, dtype=np.uint8)
        sg1 = np.frombuffer(sig, dtype=np.uint8)
        P = lambda a: a.ctypes.data
        assert lib.blsgpu_verify_multisig_batch_keyed(ctx, ks.id, 0, 1, 1, P(big), P(idx1), P(sg1), P(msg1), P(one), P(st1)) == -1
        assert lib.blsgpu_verify_multisig_batch(ctx, 2, 0, 1, 1, P(big), P(kb), P(sg1), P(msg1), P(one), P(st1)) == -1
        assert lib.blsgpu_verify_multisig_batch_keyed(ctx, ks.id, 0, 1, 1, P(one), P(idx1), P(sg1), P(msg1), P(big), P(st1)) == -1
        assert lib.blsgpu_verify_multisig_batch(ctx, 2, 0, 1, 1, P(one), P(kb), P(sg1), P(msg1), P(big), P(st1)) == -1
        out, bad = np.zeros(48, dtype=np.uint8), np.zeros(1, dtype=np.int64)
        assert lib.blsgpu_sum_points_batch(ctx, 1, 1, 1, P(big), P(kb), P(out), P(st1), P(bad)) == -1
        # null pointers
        assert lib.blsgpu_verify_multisig_batch_keyed(ctx, ks.id, 0, 1, 1, P(one), None, P(sg1), P(msg1), P(one), P(st1)) == -1
        assert lib.blsgpu_verify_multisig_batch_keyed(ctx, ks.id, 0, 1, 1, P(one), P(idx1), None, P(msg1), P(one), P(st1)) == -1
        assert lib.blsgpu_verify_multisig_batch_keyed(ctx, ks.id, 0, 1, 1, P(one), P(idx1), P(sg1), None, P(one), P(st1)) == -1
        assert lib.blsgpu_verify_multisig_batch_keyed(ctx, ks.id, 0, 1, 1, P(one), P(idx1), P(sg1), P(msg1), None, P(st1)) == -1
        assert lib.blsgpu_verify_multisig_batch_keyed(ctx, ks.id, 0, 1, 1, P(one), P(idx1), P(sg1), P(msg1), P(one), None) == -1
        assert lib.blsgpu_verify_multisig_batch(ctx, 2, 0, 1, 1, P(one), None, P(sg1), P(msg1), P(one), P(st1)) == -1
        assert lib.blsgpu_verify_multisig_batch(ctx, 2, 0, 1, 1, None, P(kb), P(sg1), P(msg1), P(one), P(st1)) == -1
        assert lib.blsgpu_sum_points_batch(ctx, 1, 1, 1, P(one), None, P(out), P(st1), P(bad)) == -1
        assert lib.blsgpu_sum_points_batch(ctx, 1, 1, 1, P(one), P(kb), None, P(st1), P(bad)) == -1
        assert lib.blsgpu_sum_points_batch(ctx, 1, 1, 1, P(one), P(kb), P(out), None, P(bad)) == -1
        assert lib.blsgpu_sum_points_batch(ctx, 3, 1, 1, P(one), P(kb), P(out), P(st1), P(bad)) == -1
        assert lib.blsgpu_verify_multisig_batch(ctx, 2, 3, 1, 1, P(one), P(kb), P(sg1), P(msg1), P(one), P(st1)) == -1
        # q = 0 does nothing, even without buffers
        assert lib.blsgpu_verify_multisig_batch_keyed(ctx, ks.id, 0, 1, 0, None, None, None, None, None, None) == 0
        assert lib.blsgpu_verify_multisig_batch(ctx, 2, 0, 1, 0, None, None, None, None, None, None) == 0
        assert lib.blsgpu_sum_points_batch(ctx, 1, 1, 0, None, None, None, None, None) == 0
        assert lib.blsgpu_sum_points_batch(ctx, 1, 1, 1, P(one), P(kb), P(out), P(st1), None) == 0   # bad_index_out may be NULL
        assert e.verify_multisig_batch_keyed(ks, 0, [[3, 2, 1, 0], [0, 1, 2]], [sig] * 2, [b"x"] * 2).tolist() == [0, 1]
        assert e.verify_multisig_batch_keyed(ks, 0, [], [], []).tolist() == []
        ks.close()
    finally:
        e.close()

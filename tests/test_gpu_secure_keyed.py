"""Keyed secure aggregation: every status and every aggregate byte of blsgpu_verify_secure_batch_keyed /
blsgpu_aggregate_secure_batch_keyed must equal the unkeyed call's on the same quorums with the key bytes written out in the
call's format (and, on a sample, the big-int oracle); both plan paths (device, and host above the cap) agree; the secure view
is built once per format; ids, indices and offsets are checked; the views' device memory dies with the set."""
import json
import os
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import bls_oracle as O

PLAN_CAP = 4096   # SECURE_PLAN_CAP in blsgpu.cu: larger quorums are planned on the host


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


def _groups(impl):
    return (1, 2) if impl == 2 else (2, 1)   # (public-key group, signature group)


def _split(flat, length):
    return [flat[i * length:(i + 1) * length].tobytes() for i in range(flat.size // length)]


def _same(got, want):
    assert list(got) == list(want), [(j, x, y) for j, (x, y) in enumerate(zip(list(got), list(want))) if x != y]


N_VALID = 8
DUP, OFF_CURVE, HEADER, IDENT = 8, 9, 10, 11   # set entries: key 2's bytes again, an off-curve key, a bad header, the identity
# (members, which quorum's aggregate signs it, message): "own" = its own aggregate
QUORUMS = [
    ([0, 1, 2, 3, 4], "own", 0),           # 0 valid
    ([4, 3, 2, 1, 0, 5], "own", 0),        # 1 valid, unsorted
    ([1, 2, 3], 0, 0),                     # 2 a wrong signature
    ([0, 1, 2, 3, 4], "own", 1),           # 3 a wrong message
    ([0, 1, 2, 3], 0, 0),                  # 4 a member missing
    ([2, 5, 2, 6], "own", 0),              # 5 the same index twice
    ([2, DUP, 7], "own", 0),               # 6 two set entries with identical bytes
    ([0, OFF_CURVE, 1], 0, 0),             # 7 an off-curve key
    ([0, 1, HEADER], 0, 0),                # 8 a bad-header key
    ([HEADER, OFF_CURVE, 0], 0, 0),        # 9 two bad keys: the first in member order decides
    ([IDENT, 0], "own", 0),                # 10 the identity key
    ([], "ident", 0),                      # 11 empty, identity signature
    ([], 0, 0),                            # 12 empty, non-identity signature
    ([0, 1], "undecodable", 0),            # 13 an undecodable signature
    ([6, 7, 1, 0, 3, 5, 4, 2], "own", 0),  # 14 every valid key
]


@pytest.mark.parametrize("impl,fmt", [(2, O.MODERN), (2, O.LEGACY), (1, O.MODERN)])
def test_mixed_quorums_equal_the_unkeyed_calls_and_the_oracle(eng, B, impl, fmt):
    C = O.IMPLS[impl]
    pkg, sgg = _groups(impl)
    pl, sl = B.pk_len(impl), B.sig_len(impl)
    rnd = random.Random(77 + 10 * impl + fmt)
    sks = [rnd.randrange(1, O.R) for _ in range(N_VALID)]
    kb = [C.pk_ser(O.sk_to_pk(impl, sk), fmt) for sk in sks]
    hdr = C.pk_ser(O.sk_to_pk(impl, sks[0]), O.MODERN)
    if fmt == O.LEGACY:
        st, ident = eng.recode_points(pkg, [_ident(pl)], O.MODERN, O.LEGACY)
        assert st.tolist() == [0]
        kb += [kb[2], O.modern_to_legacy(_off_curve(pkg)), hdr if hdr[0] & 0x20 else _neg(hdr), ident[0]]
        bad_sig = O.modern_to_legacy(_off_curve(sgg))
        ident_sig = eng.recode_points(sgg, [_ident(sl)], O.MODERN, O.LEGACY)[1][0]
    else:
        kb += [kb[2], _off_curve(pkg), bytes([hdr[0] & 0x7F]) + hdr[1:], _ident(pl)]
        bad_sig, ident_sig = _off_curve(sgg), _ident(sl)
    ks = eng.key_set(impl, kb, fmt)
    try:
        assert ks.status[:N_VALID + 1].tolist() == [0] * (N_VALID + 1) and ks.status[IDENT] == 0
        assert ks.status[OFF_CURVE] in (O.ERR_DESERIALIZE, O.ERR_LEGACY_FORMAT) and ks.status[HEADER] in (O.ERR_DESERIALIZE, O.ERR_LEGACY_FORMAT)
        msgs = [b"keyed secure %d" % impl, b"another message"]
        for scheme in (0, 1, 2):
            # verify_secure hashes the bare message under the scheme's DST (no pk prefix even for MessageAugmentation)
            h = C.hash(msgs[0], O.sig_dst(impl, scheme))
            member = [C.sig_ser(C.sig_mul(h, sk), fmt) for sk in sks]
            member += [member[2], member[0], member[1], ident_sig]   # signatures beside the DUP / bad / identity keys
            idx_sets = [m for m, _, _ in QUORUMS]
            key_sets = [[kb[k] for k in m] for m in idx_sets]
            sig_sets = [[member[k] for k in m] for m in idx_sets]
            sig_sets[5][2] = sig_sets[6][1] = member[0]   # a duplicate key reuses the FIRST match's signature, not its own
            st_u, agg_u = eng.aggregate_secure_batch(impl, key_sets, sig_sets, fmt)
            st_k, agg_k = eng.aggregate_secure_batch_keyed(ks, idx_sets, sig_sets, fmt)
            _same(st_k, st_u)
            assert agg_k == agg_u
            for j in (5, 6, 10, 11):   # duplicates (first match), the identity key, an empty quorum
                assert (int(st_u[j]), agg_u[j]) == O.aggregate_secure(impl, fmt, key_sets[j], sig_sets[j]), j
            sigs = [agg_u[j] if s == "own" else ident_sig if s == "ident" else bad_sig if s == "undecodable" else agg_u[s]
                    for j, (_, s, _) in enumerate(QUORUMS)]
            qmsgs = [msgs[m] for _, _, m in QUORUMS]
            want = eng.verify_secure_batch(impl, scheme, key_sets, sigs, qmsgs, fmt)
            got = eng.verify_secure_batch_keyed(ks, scheme, idx_sets, sigs, qmsgs, fmt)
            _same(got, want)
            w = want.tolist()
            assert [w[j] for j in (0, 1, 5, 6, 11, 14)] == [0] * 6
            assert [w[j] for j in (2, 3, 4, 12)] == [O.ERR_INVALID_SIGNATURE] * 4
            for j in (7, 8, 9, 13):
                assert w[j] in (O.ERR_DESERIALIZE, O.ERR_LEGACY_FORMAT), j
            assert w[9] == ks.status[HEADER]
            if scheme == 0:   # a sample end to end against the big-int oracle
                for j in (0, 4, 6, 9, 10, 12):
                    assert O.verify_secure(impl, scheme, fmt, key_sets[j], sigs[j], qmsgs[j]) == got[j], j
    finally:
        ks.close()


def test_a_set_serves_calls_in_the_other_format(eng, B):
    """A Modern set in Legacy calls and a Legacy set in Modern calls: the keys are hashed in the call's format, as the
    unkeyed call on keys recoded by blsgpu_recode_points"""
    rnd = random.Random(5)
    n = 12
    secret = np.frombuffer(b"".join(rnd.randrange(1, O.R).to_bytes(32, "big") for _ in range(n)), dtype=np.uint8)
    msg = b"cross-format quorum"
    pk_m, sg_m = eng.testdata_sign(2, 0, secret, *B.pack_messages([msg] * n))
    enc = {O.MODERN: (pk_m, sg_m), O.LEGACY: (eng.recode_points_packed(1, pk_m, 1, 0), eng.recode_points_packed(2, sg_m, 1, 0))}
    idx_sets = [list(range(8)), [7, 3, 3, 11, 0], [10, 9], []]
    sets = {f: eng.key_set(2, enc[f][0], f) for f in (O.MODERN, O.LEGACY)}
    try:
        for set_fmt, call_fmt in ((O.MODERN, O.LEGACY), (O.LEGACY, O.MODERN)):
            kb, sb = _split(enc[call_fmt][0], 48), _split(enc[call_fmt][1], 96)
            key_sets = [[kb[k] for k in m] for m in idx_sets]
            sig_sets = [[sb[k] for k in m] for m in idx_sets]
            st_u, agg_u = eng.aggregate_secure_batch(2, key_sets, sig_sets, call_fmt)
            st_k, agg_k = eng.aggregate_secure_batch_keyed(sets[set_fmt], idx_sets, sig_sets, call_fmt)
            _same(st_k, st_u)
            assert agg_k == agg_u and st_u.tolist() == [0] * len(idx_sets)
            sigs = list(agg_u)
            sigs[2] = agg_u[1]   # a wrong signature
            want = eng.verify_secure_batch(2, 0, key_sets, sigs, [msg] * len(idx_sets), call_fmt)
            got = eng.verify_secure_batch_keyed(sets[set_fmt], 0, idx_sets, sigs, [msg] * len(idx_sets), call_fmt)
            _same(got, want)
            assert want.tolist() == [0, 0, 1, 0]
            for j in (0, 1, 2):
                assert O.verify_secure(2, 0, call_fmt, key_sets[j], sigs[j], msg) == got[j], (set_fmt, j)
            # the aggregate of one format does not verify under the other
            other = eng.verify_secure_batch_keyed(sets[set_fmt], 0, idx_sets[:1], sigs[:1], [msg], set_fmt)
            assert other.tolist() == [O.verify_secure(2, 0, set_fmt, [enc[set_fmt][0][48 * k:48 * k + 48].tobytes() for k in idx_sets[0]],
                                                      sigs[0], msg)]
    finally:
        for s in sets.values():
            s.close()


def test_production_57_key_vector_through_a_key_set(eng, B, golden_dir):
    sec = json.load(open(os.path.join(golden_dir, "secure_57.json")))
    pks = [bytes.fromhex(k) for k in sec["keys"]]
    sig, msg = bytes.fromhex(sec["sig"]), bytes.fromhex(sec["message"])
    ks = eng.key_set(2, pks)
    try:
        assert not ks.status.any()
        order = list(range(57))
        perm = order[:]
        random.Random(57).shuffle(perm)
        idx_sets = [order, perm, order[::-1], order[:-1], order[1:]]
        got = eng.verify_secure_batch_keyed(ks, 0, idx_sets, [sig] * 5, [msg] * 5)
        assert got.tolist() == [0, 0, 0, 1, 1]
        _same(got, eng.verify_secure_batch(2, 0, [[pks[k] for k in m] for m in idx_sets], [sig] * 5, [msg] * 5))
    finally:
        ks.close()


def test_quorums_on_both_sides_of_the_plan_cap(eng, B):
    """One call with quorums of PLAN_CAP + 1 members (planned on the host) and PLAN_CAP members (on the device) beside small
    ones; members repeat, so the first-match rule is exercised on both paths"""
    rng = np.random.default_rng(4097)
    k = 5000
    secret = np.zeros((k, 32), dtype=np.uint8)
    secret[:, 8:] = rng.integers(0, 256, size=(k, 24), dtype=np.uint8)
    secret[:, 31] |= 1
    sizes = [3, PLAN_CAP + 1, 17, PLAN_CAP, 1, PLAN_CAP + 1]
    idx_sets = [rng.integers(0, k, size=s, dtype=np.uint32) for s in sizes]
    idx_sets[5] = rng.permutation(k)[:PLAN_CAP + 1].astype(np.uint32)   # distinct members
    koff = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    idx = np.concatenate(idx_sets)
    q = len(sizes)
    qmsgs = [b"cap quorum %d" % j for j in range(q)]
    data_m, off_m = B.pack_messages([qmsgs[j] for j in range(q) for _ in range(sizes[j])])
    _, member = eng.testdata_sign(2, 0, secret[idx].reshape(-1), data_m, off_m)
    kb, _ = eng.testdata_sign(2, 0, secret.reshape(-1), *B.pack_messages([b""] * k))
    ks = eng.key_set(2, kb)
    try:
        pk = kb.reshape(k, 48)[idx].reshape(-1)
        st_u, agg_u = eng.aggregate_secure_batch_packed(2, koff, pk, member)
        st_k, agg_k = eng.aggregate_secure_batch_keyed_packed(ks, koff, idx, member)
        assert st_u.tolist() == [0] * q
        _same(st_k, st_u)
        assert agg_k.tobytes() == agg_u.tobytes()
        data, off = B.pack_messages(qmsgs)
        sigs = agg_u.reshape(q, 96).copy()
        sigs[[1, 2]] = sigs[[2, 1]]
        want = eng.verify_secure_batch_packed(2, 0, koff, pk, sigs.reshape(-1), data, off)
        got = eng.verify_secure_batch_keyed_packed(ks, 0, koff, idx, sigs.reshape(-1), data, off)
        assert want.tolist() == [0, 1, 1, 0, 0, 0]
        _same(got, want)
    finally:
        ks.close()


def test_cfg5_shape_over_a_4096_key_set(eng, B):
    """10,000 quorums x 400 distinct members drawn from one 4,096-key set"""
    rng = np.random.default_rng(5)
    k, q, mem = 4096, 10_000, 400
    secret = np.zeros((k, 32), dtype=np.uint8)
    secret[:, 8:] = rng.integers(0, 256, size=(k, 24), dtype=np.uint8)
    secret[:, 31] |= 1
    idx = np.concatenate([rng.choice(k, mem, replace=False) for _ in range(q)]).astype(np.uint32)
    qm = rng.integers(0, 256, size=(q, 32), dtype=np.uint8)
    tot, chunk = q * mem, 1 << 20
    member = np.empty(tot * 96, dtype=np.uint8)
    for lo in range(0, tot, chunk):
        hi = min(tot, lo + chunk)
        o = np.arange(hi - lo + 1, dtype=np.uint64) * 32
        member[lo * 96:hi * 96] = eng.testdata_sign(2, 0, secret[idx[lo:hi]].reshape(-1), np.ascontiguousarray(qm[np.arange(lo, hi) // mem]).reshape(-1), o)[1]
    kb, _ = eng.testdata_sign(2, 0, secret.reshape(-1), *B.pack_messages([b""] * k))
    koff = np.arange(q + 1, dtype=np.uint64) * mem
    qoff = np.arange(q + 1, dtype=np.uint64) * 32
    ks = eng.key_set(2, kb)
    try:
        st, aggs = eng.aggregate_secure_batch_keyed_packed(ks, koff, idx, member)
        assert int(st.max()) == 0
        assert eng.verify_secure_batch_keyed_packed(ks, 0, koff, idx, aggs, qm.reshape(-1), qoff).tolist() == [0] * q
        swapped = aggs.copy().reshape(q, 96)
        swapped[[3, 4]] = swapped[[4, 3]]
        got = eng.verify_secure_batch_keyed_packed(ks, 0, koff, idx, swapped.reshape(-1), qm.reshape(-1), qoff)
        assert np.nonzero(got)[0].tolist() == [3, 4]
        pk = kb.reshape(k, 48)[idx].reshape(-1)
        _same(got, eng.verify_secure_batch_packed(2, 0, koff, pk, swapped.reshape(-1), qm.reshape(-1), qoff))
    finally:
        ks.close()


@pytest.mark.parametrize("impl", [2, 1])
def test_no_key_decode_and_the_view_is_built_once(eng, B, impl):
    rnd = random.Random(40 + impl)
    n = 16
    secret = np.frombuffer(b"".join(rnd.randrange(1, O.R).to_bytes(32, "big") for _ in range(n)), dtype=np.uint8)
    kb, member = eng.testdata_sign(impl, 0, secret, *B.pack_messages([b"m"] * n))
    pl, sl = B.pk_len(impl), B.sig_len(impl)
    koff = np.array([0, 5, 16], dtype=np.uint64)
    idx = np.arange(n, dtype=np.uint32)[::-1].copy()
    ks = eng.key_set(impl, kb)
    pk = kb.reshape(n, pl)[idx].reshape(-1)
    sg = member.reshape(n, sl)[idx].reshape(-1)
    try:
        def launches(call):
            c0 = eng.launch_count()
            out = call()
            return eng.launch_count() - c0, out
        aggregate = lambda: eng.aggregate_secure_batch_keyed_packed(ks, koff, idx, sg)
        first, (st, aggs) = launches(aggregate)
        second, _ = launches(aggregate)
        third, _ = launches(aggregate)
        assert st.tolist() == [0, 0] and second == third == first - 1   # the first call encodes the view (one k_encode)
        unkeyed, (st_u, aggs_u) = launches(lambda: eng.aggregate_secure_batch_packed(impl, koff, pk, sg))
        assert unkeyed == second + 1 and aggs_u.tobytes() == aggs.tobytes()   # + key decode and subgroup check - the device plan
        data, off = B.pack_messages([b"m", b"m"])
        verify = lambda: eng.verify_secure_batch_keyed_packed(ks, 0, koff, idx, aggs, data, off)
        v1, st = launches(verify)
        v2, _ = launches(verify)
        assert st.tolist() == [0, 0] and v1 == v2   # the view of this format exists already
        vu, st_u = launches(lambda: eng.verify_secure_batch_packed(impl, 0, koff, pk, aggs, data, off))
        assert st_u.tolist() == [0, 0] and vu == v2 + 1
    finally:
        ks.close()


def test_errors_then_the_context_still_verifies(B):
    e, other = B.Engine([0]), B.Engine([0])
    try:
        rnd = random.Random(13)
        secret = np.frombuffer(b"".join(rnd.randrange(1, O.R).to_bytes(32, "big") for _ in range(4)), dtype=np.uint8)
        kb, member = e.testdata_sign(2, 0, secret, *B.pack_messages([b"x"] * 4))
        ks, gone, foreign = e.key_set(2, kb), e.key_set(2, kb), other.key_set(2, kb)
        g1 = e.key_set(1, e.testdata_sign(1, 0, secret, *B.pack_messages([b"x"] * 4))[0])
        sg = _split(member, 96)
        st, aggs = e.aggregate_secure_batch_keyed(ks, [[0, 1, 2, 3]], [sg])
        assert st.tolist() == [0]
        gone_id = gone.id
        gone.close()
        for ident in (gone_id, foreign.id, 0):
            fake = B.KeySet(e, 2, ident, np.zeros(4, dtype=np.uint8))
            with pytest.raises(B.EngineError, match=r"\(-1\)"):
                e.verify_secure_batch_keyed(fake, 0, [[0, 1, 2, 3]], aggs, [b"x"])
            with pytest.raises(B.EngineError, match=r"\(-1\)"):
                e.aggregate_secure_batch_keyed(fake, [[0, 1, 2, 3]], [sg])
        with pytest.raises(B.EngineError, match=r"key_idx\[5\]"):
            e.verify_secure_batch_keyed(ks, 0, [[0, 1], [2, 3, 1, 4]], aggs * 2, [b"x"] * 2)
        with pytest.raises(B.EngineError, match=r"key_idx\[2\]"):
            e.aggregate_secure_batch_keyed(ks, [[0, 1, 9]], [sg[:3]])
        with pytest.raises(B.EngineError, match=r"Legacy"):   # Legacy exists only for Bls12381G2Impl
            e.verify_secure_batch_keyed(g1, 0, [[0]], [bytes(48)], [b"x"], O.LEGACY)
        with pytest.raises(B.EngineError, match=r"Legacy"):
            e.aggregate_secure_batch_keyed(g1, [[0]], [[bytes(48)]], O.LEGACY)
        koff = np.array([0, 3, 2], dtype=np.uint64)   # decreasing
        data, off = B.pack_messages([b"x", b"x"])
        with pytest.raises(B.EngineError, match=r"non-decreasing"):
            e.verify_secure_batch_keyed_packed(ks, 0, koff, np.zeros(2, dtype=np.uint32), np.frombuffer(aggs[0] * 2, dtype=np.uint8), data, off)
        with pytest.raises(B.EngineError, match=r"non-decreasing"):
            e.aggregate_secure_batch_keyed_packed(ks, koff, np.zeros(2, dtype=np.uint32), member[:192])
        assert e.verify_secure_batch_keyed(ks, 0, [[3, 2, 1, 0], [0, 1, 2]], aggs * 2, [b"x"] * 2).tolist() == [0, 1]
        assert e.verify_secure_batch_keyed(ks, 0, [], [], []).tolist() == []
        assert other.verify_secure_batch_keyed(foreign, 0, [[0, 1, 2, 3]], aggs, [b"x"]).tolist() == [0]
        ks.close()
        g1.close()
    finally:
        other.close()
        e.close()


def test_destroying_the_set_frees_its_views(B):
    import torch
    rng = np.random.default_rng(3)
    k = 1 << 18
    secret = np.zeros((4096, 32), dtype=np.uint8)
    secret[:, 8:] = rng.integers(0, 256, size=(4096, 24), dtype=np.uint8)
    secret[:, 31] |= 1
    e = B.Engine([0])
    try:
        kb, member = e.testdata_sign(2, 0, secret.reshape(-1), *B.pack_messages([b"v"] * 4096))
        big = np.tile(kb, k // 4096)
        koff = np.array([0, 3], dtype=np.uint64)
        idx = np.array([0, 1, 2], dtype=np.uint32)
        data, off = B.pack_messages([b"v"])

        def use(ks):
            for fmt in (O.MODERN, O.LEGACY):
                sg = member[:288] if fmt == O.MODERN else e.recode_points_packed(2, member[:288], 1, 0)
                st, agg = e.aggregate_secure_batch_keyed_packed(ks, koff, idx, sg, fmt)
                assert st.tolist() == [0]
                assert e.verify_secure_batch_keyed_packed(ks, 0, koff, idx, agg, data, off, fmt).tolist() == [0]
        warm = e.key_set(2, kb[:48 * 16])
        use(warm)   # loads the kernels and sizes the arena for these calls
        warm.close()
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info(0)[0]
        ks = e.key_set(2, big)
        after_set = torch.cuda.mem_get_info(0)[0]
        use(ks)
        after_views = torch.cuda.mem_get_info(0)[0]
        assert after_set < free0 - 145 * k + 2 * 2 ** 20
        assert after_views <= after_set - 2 * 52 * k + 2 * 2 ** 20   # two views of 52 bytes per key
        ks.close()
        assert abs(torch.cuda.mem_get_info(0)[0] - free0) <= 2 * 2 ** 20
        live = e.key_set(2, big)
        use(live)
    finally:
        e.close()   # frees the live set and its views (and the context's scratch, which free0 still counted)
    live.close()
    assert torch.cuda.mem_get_info(0)[0] >= free0 - 2 * 2 ** 20

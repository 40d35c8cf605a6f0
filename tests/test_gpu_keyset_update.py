"""Key sets changed in place (blsgpu_keyset_update / blsgpu_keyset_append): after any sequence of changes every keyed call
returns byte for byte what it returns on a set created from the final key bytes, and what the unkeyed call returns on those
bytes; live secure views follow the changes without a rebuild; refused calls leave the set as it was; a grown set frees all
of its device memory."""
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


def _groups(impl):
    return (1, 2) if impl == 2 else (2, 1)   # (public-key group, signature group)


def _same(got, want):
    assert list(got) == list(want), [(j, x, y) for j, (x, y) in enumerate(zip(list(got), list(want))) if x != y]


def _secrets(rnd, n):
    return [rnd.randrange(1, O.R).to_bytes(32, "big") for _ in range(n)]


def _sign(eng, B, impl, scheme, secrets, msgs):
    """(pks, sigs) as lists of Modern encodings, item i signed with secrets[i] over msgs[i]"""
    pk, sg = eng.testdata_sign(impl, scheme, np.frombuffer(b"".join(secrets), dtype=np.uint8), *B.pack_messages(msgs))
    pl, sl = B.pk_len(impl), B.sig_len(impl)
    return [pk[i * pl:(i + 1) * pl].tobytes() for i in range(len(msgs))], [sg[i * sl:(i + 1) * sl].tobytes() for i in range(len(msgs))]


class Keys:
    """Public-key encodings of one impl in either format: valid keys of given secrets, and keys that decode to an error or to
    the identity."""

    def __init__(self, eng, B, impl):
        self.eng, self.B, self.impl = eng, B, impl
        self.pkg = _groups(impl)[0]
        self.pl = B.pk_len(impl)

    def recode(self, modern, fmt):
        if fmt == O.MODERN:
            return list(modern)
        st, out = self.eng.recode_points(self.pkg, modern, O.MODERN, fmt)
        assert st.tolist() == [0] * len(modern)
        return list(out)

    def valid(self, secrets, fmt):
        return self.recode(_sign(self.eng, self.B, self.impl, 0, secrets, [b"k"] * len(secrets))[0], fmt)

    def off_curve(self, fmt):
        e = _off_curve(self.pkg)
        return e if fmt == O.MODERN else O.modern_to_legacy(e)

    def bad_header(self, fmt, secret):
        hdr = _sign(self.eng, self.B, self.impl, 0, [secret], [b"k"])[0][0]
        if fmt == O.MODERN:
            return bytes([hdr[0] & 0x7F]) + hdr[1:]   # no compression flag
        return hdr if hdr[0] & 0x20 else _neg(hdr)

    def identity(self, fmt):
        return self.recode([_ident(self.pl)], fmt)[0]


def _statuses(eng, impl, encs, fmt):
    ks = eng.key_set(impl, encs, fmt)
    ks.close()
    return ks.status.tolist()


def _every_keyed_call(eng, B, impl, fmt, sets, final, secret, rnd):
    """Runs every keyed entry point over the key sets in `sets` (all holding the keys `final`, in the set format fmt) and the
    unkeyed calls on the bytes; asserts that all of them agree item for item and byte for byte."""
    n = len(final)
    pkg, sgg = _groups(impl)
    sl = B.sig_len(impl)
    other = rnd.choice([s for s in secret if s is not None])
    signer = [s if s is not None else other for s in secret]
    msgs = [b"update/%d" % j for j in range(3)]
    key_idx = list(range(n)) * 2
    rnd.shuffle(key_idx)
    msg_idx = [rnd.randrange(len(msgs)) for _ in key_idx]
    item_pks = [final[k] for k in key_idx]
    conv = (lambda encs: encs) if fmt == O.MODERN else (lambda encs: list(eng.recode_points(sgg, encs, O.MODERN, fmt)[1]))
    for scheme in (0, 1, 2):
        sigs = conv(_sign(eng, B, impl, scheme, [signer[k] for k in key_idx], [msgs[j] for j in msg_idx])[1])
        sigs[3], sigs[4] = sigs[4], sigs[3]   # two wrong signatures
        item_msgs = [msgs[j] for j in msg_idx]
        want = eng.verify_batch(impl, scheme, item_pks, sigs, item_msgs, fmt)
        if scheme != 1 or fmt == O.MODERN:   # MessageAugmentation signed the Modern key's bytes
            assert (want == 0).sum() > n // 2, want
        for ks in sets:
            _same(eng.verify_batch_keyed(ks, scheme, key_idx, sigs, item_msgs, fmt), want)
        _same(eng.verify_batch_grouped(impl, scheme, item_pks, sigs, msg_idx, msgs, fmt), want)
        for ks in sets:
            _same(eng.verify_batch_grouped_keyed(ks, scheme, key_idx, sigs, msg_idx, msgs, fmt), want)
    # quorums over every key, with repeats; member signatures (Basic) of each member's signer
    quorums = [list(range(n)), [n - 1, 0, n // 2, n - 1], [k for k in range(n) if secret[k] is not None][::-1], [0, 3, 4], [1, 2, 3], []]
    quorums += [rnd.sample(range(n), 5) for _ in range(6)]
    call_fmts = (O.MODERN, O.LEGACY) if impl == 2 else (O.MODERN,)
    for cf in call_fmts:
        # the unkeyed calls take the keys encoded in the call's format: recoded where they decode, as given where they do not
        st = _statuses(eng, impl, final, fmt)
        enc = list(final)
        if cf != fmt:
            ok = [k for k in range(n) if st[k] == 0]
            rec = eng.recode_points(pkg, [final[k] for k in ok], fmt, cf)[1]
            for k, e in zip(ok, rec):
                enc[k] = e
        comparable = [j for j, m in enumerate(quorums) if cf == fmt or all(st[k] == 0 for k in m)]
        key_sets = [[enc[k] for k in m] for m in quorums]
        sig_sets = [conv(_sign(eng, B, impl, 0, [signer[k] for k in m], [msgs[0]] * len(m))[1]) if m else [] for m in quorums]
        if cf != fmt:
            sig_sets = [list(eng.recode_points(sgg, s, fmt, cf)[1]) if s else [] for s in sig_sets]
        st_u, agg_u = eng.aggregate_secure_batch(impl, key_sets, sig_sets, cf)
        got = [eng.aggregate_secure_batch_keyed(ks, quorums, sig_sets, cf) for ks in sets]
        for st_k, agg_k in got:
            _same(st_k, got[0][0])
            assert agg_k == got[0][1]
        for j in comparable:
            assert (int(got[0][0][j]), got[0][1][j]) == (int(st_u[j]), agg_u[j]), j
        assert st_u[2] == 0   # the valid keys
        sigs = list(agg_u)
        sigs[3] = agg_u[2]    # a wrong signature
        for scheme in (0, 1, 2):
            want = eng.verify_secure_batch(impl, scheme, key_sets, sigs, [msgs[0]] * len(quorums), cf)
            got_v = [eng.verify_secure_batch_keyed(ks, scheme, quorums, sigs, [msgs[0]] * len(quorums), cf) for ks in sets]
            for g in got_v:
                _same(g, got_v[0])
            _same([int(got_v[0][j]) for j in comparable], [int(want[j]) for j in comparable])
            if scheme == 0:
                assert got_v[0][2] == 0 and got_v[0][3] == O.ERR_INVALID_SIGNATURE
    # multi-signatures over subsets: the sum of the members' signatures
    for scheme in (0, 2):
        ms = [eng.sum_points(sgg, _sign(eng, B, impl, scheme, [signer[k] for k in m], [msgs[1]] * len(m))[1]) if m else _ident(sl)
              for m in quorums]
        ms = conv(ms)
        ms[1] = ms[0]
        want = eng.verify_multisig_batch(impl, scheme, [[final[k] for k in m] for m in quorums], ms, [msgs[1]] * len(quorums), fmt)
        assert want[2] == 0 and want[1] == O.ERR_INVALID_SIGNATURE   # every valid key; another set's signature
        for ks in sets:
            _same(eng.verify_multisig_batch_keyed(ks, scheme, quorums, ms, [msgs[1]] * len(quorums), fmt), want)


@pytest.mark.parametrize("impl,fmt", [(2, O.MODERN), (2, O.LEGACY), (1, O.MODERN)])
def test_updates_and_appends_equal_a_fresh_set(eng, B, impl, fmt):
    rnd = random.Random(900 + 10 * impl + fmt)
    K = Keys(eng, B, impl)
    n_valid = 10
    secret = _secrets(rnd, n_valid)
    OFF, HDR, IDENT = n_valid, n_valid + 1, n_valid + 2
    final = K.valid(secret, fmt) + [K.off_curve(fmt), K.bad_header(fmt, secret[0]), K.identity(fmt)]
    secret = secret + [None, None, None]
    ks = eng.key_set(impl, final, fmt)
    try:
        # both views live before the changes
        for cf in ((O.MODERN, O.LEGACY) if impl == 2 else (O.MODERN,)):
            eng.verify_secure_batch_keyed(ks, 0, [[0, 1]], [bytes(B.sig_len(impl))], [b"v"], cf)

        def update(idx, encs, f=fmt, final_encs=None):
            st = eng.update_key_set(ks, idx, encs, f)
            assert st.tolist() == _statuses(eng, impl, encs, f)   # what keyset_create gives for the same bytes
            for i, e in zip(idx, final_encs or encs):
                final[i] = e
            return st

        new = _secrets(rnd, 4)
        # valid -> valid, valid -> off-curve, bad -> valid, valid -> identity, in one call with unsorted indices
        update([OFF, 0, 2, 1], K.valid(new[:2], fmt) + [K.identity(fmt), K.off_curve(fmt)])
        secret[OFF], secret[0], secret[2], secret[1] = new[0], new[1], None, None
        update([3], [final[4]])                    # key 3 takes key 4's bytes ...
        secret[3] = secret[4]
        _every_keyed_call(eng, B, impl, fmt, [ks], final, secret, rnd)
        update([3], K.valid([new[2]], fmt))        # ... and stops being equal to it
        secret[3] = new[2]
        other = 1 - fmt
        update([5], K.valid([new[3]], other), other, K.valid([new[3]], fmt))   # the other format
        secret[5] = new[3]
        assert ks.status.tolist() == _statuses(eng, impl, final, fmt)
        app = _secrets(rnd, 3)
        encs = K.valid(app[:2], fmt) + [K.bad_header(fmt, app[2]), K.off_curve(fmt), final[6]]
        st = eng.append_key_set(ks, encs, fmt)
        assert st.tolist() == _statuses(eng, impl, encs, fmt) and st.tolist()[2] != 0 and st.tolist()[3] != 0
        final += encs
        secret += app[:2] + [None, None, secret[6]]
        assert len(ks) == len(final) == 18
        fresh = eng.key_set(impl, final, fmt)
        try:
            _same(ks.status, fresh.status)
            _every_keyed_call(eng, B, impl, fmt, [ks, fresh], final, secret, rnd)
        finally:
            fresh.close()
    finally:
        ks.close()


def test_views_follow_updates(eng, B):
    impl = 2
    rnd = random.Random(31)
    n = 12
    secret = _secrets(rnd, n)
    kb = _sign(eng, B, impl, 0, secret, [b"k"] * n)[0]
    ks = eng.key_set(impl, kb)
    msg = b"views"

    def sigs_of(members, fmt, m=msg):
        s = _sign(eng, B, impl, 0, [secret[k] for k in members], [m] * len(members))[1]
        return s if fmt == O.MODERN else list(eng.recode_points(2, s, O.MODERN, O.LEGACY)[1])

    def keys_in(fmt):
        return kb if fmt == O.MODERN else list(eng.recode_points(1, kb, O.MODERN, O.LEGACY)[1])

    def launches(call):
        c0 = eng.launch_count()
        out = call()
        return eng.launch_count() - c0, out

    def check(quorums, views_exist=True):
        for fmt in (O.MODERN, O.LEGACY):
            kf = keys_in(fmt)
            key_sets = [[kf[k] for k in m] for m in quorums]
            sig_sets = [sigs_of(m, fmt) for m in quorums]
            for j, m in enumerate(quorums):   # a member's own signature beside a repeated key: the first equal key's is used
                for p in range(1, len(m)):
                    if kf[m[p]] in [kf[x] for x in m[:p]]:
                        sig_sets[j][p] = sigs_of([m[p]], fmt, b"not used")[0]
            st_u, agg_u = eng.aggregate_secure_batch(impl, key_sets, sig_sets, fmt)
            call = lambda: eng.aggregate_secure_batch_keyed(ks, quorums, sig_sets, fmt)
            c1, (st_k, agg_k) = launches(call)
            c2, _ = launches(call)
            assert c1 == c2 + (0 if views_exist else 1), (fmt, c1, c2)   # kept current: no rebuild after an update
            _same(st_k, st_u)
            assert agg_k == agg_u
            want = eng.verify_secure_batch(impl, 0, key_sets, agg_u, [msg] * len(quorums), fmt)
            _same(eng.verify_secure_batch_keyed(ks, 0, quorums, agg_u, [msg] * len(quorums), fmt), want)
            assert want.tolist() == [0] * len(quorums)

    try:
        quorums = [list(range(n)), [0, 1, 2], [5, 4, 3, 2, 1, 0], [7, 8]]
        check(quorums, views_exist=False)   # builds both views
        cand_secret, cand = [], []
        while not cand or min(cand) > min(kb) or max(cand) < max(kb):   # smaller / larger than every key of the set (Modern bytes)
            more = _secrets(rnd, 48)
            cand_secret += more
            cand += _sign(eng, B, impl, 0, more, [b"k"] * len(more))[0]
        lo = min(range(len(cand)), key=lambda c: cand[c])
        hi = max(range(len(cand)), key=lambda c: cand[c])
        eng.update_key_set(ks, [4, 9], [cand[lo], cand[hi]])
        kb[4], kb[9], secret[4], secret[9] = cand[lo], cand[hi], cand_secret[lo], cand_secret[hi]
        q2 = quorums + [[9, 4], [4, 0, 9, 1]]
        check(q2)
        eng.update_key_set(ks, [6], [kb[2]])   # keys 2 and 6 become equal
        kb[6], secret[6] = kb[2], secret[2]
        q3 = q2 + [[6, 2, 1], [2, 6], [3, 6, 5, 2, 6]]
        check(q3)
        # the first equal key's signature, against the big-int oracle
        sig_sets = [sigs_of(m, O.MODERN) for m in q3[-3:]]
        sig_sets[0][1] = sigs_of([6], O.MODERN, b"not used")[0]   # key 6 equals key 2, which comes first
        st_k, agg_k = eng.aggregate_secure_batch_keyed(ks, q3[-3:-2], sig_sets[:1], O.MODERN)
        assert (int(st_k[0]), agg_k[0]) == O.aggregate_secure(impl, O.MODERN, [kb[k] for k in q3[-3]], sig_sets[0])
        fresh_secret = _secrets(rnd, 1)
        eng.update_key_set(ks, [6], _sign(eng, B, impl, 0, fresh_secret, [b"k"])[0])   # and stop being equal
        kb[6], secret[6] = _sign(eng, B, impl, 0, fresh_secret, [b"k"])[0][0], fresh_secret[0]
        check(q3)
        fresh = eng.key_set(impl, kb)
        try:
            for fmt in (O.MODERN, O.LEGACY):
                sig_sets = [sigs_of(m, fmt) for m in q3]
                a = eng.aggregate_secure_batch_keyed(ks, q3, sig_sets, fmt)
                b = eng.aggregate_secure_batch_keyed(fresh, q3, sig_sets, fmt)
                _same(a[0], b[0])
                assert a[1] == b[1]
        finally:
            fresh.close()
    finally:
        ks.close()


def test_errors_leave_the_set_unchanged(B):
    e, other = B.Engine([0]), B.Engine([0])
    try:
        rnd = random.Random(17)
        secret = _secrets(rnd, 6)
        kb, sigs = _sign(e, B, 2, 0, secret, [b"e"] * 6)
        ks, gone, foreign = e.key_set(2, kb), e.key_set(2, kb), other.key_set(2, kb)
        quorums = [[0, 1, 2], [3, 4, 5, 0]]
        sig_sets = [[sigs[k] for k in m] for m in quorums]

        def results():
            st, agg = e.aggregate_secure_batch_keyed(ks, quorums, sig_sets)
            v = e.verify_batch_keyed(ks, 0, list(range(6)), sigs, [b"e"] * 6)
            return st.tolist(), agg, v.tolist(), e.verify_secure_batch_keyed(ks, 0, quorums, agg, [b"e"] * 2).tolist()

        before = results()
        assert before[0] == [0, 0] and before[2] == [0] * 6 and before[3] == [0, 0]
        new = _sign(e, B, 2, 0, _secrets(rnd, 2), [b"e"] * 2)[0]
        with pytest.raises(B.EngineError, match=r"\(-1\).*key_idx\[1\] is not below the key set's size 6"):
            e.update_key_set(ks, [0, 6], new)
        with pytest.raises(B.EngineError, match=r"\(-1\).*key_idx\[0\] and key_idx\[2\] both name key 3"):
            e.update_key_set(ks, [3, 1, 3], new + new[:1])
        gone_id = gone.id
        gone.close()
        for ident in (gone_id, foreign.id):
            fake = B.KeySet(e, 2, ident, np.zeros(6, dtype=np.uint8))
            with pytest.raises(B.EngineError, match=r"\(-1\).*is not held by this context"):
                e.update_key_set(fake, [0], new[:1])
            with pytest.raises(B.EngineError, match=r"\(-1\).*is not held by this context"):
                e.append_key_set(fake, new[:1])
        # an append past 2^32 - 16 keys is refused before its bytes are read
        pk = np.zeros(48, dtype=np.uint8)
        assert e._lib.blsgpu_keyset_append(e._ctx, ks.id, 1, 0xfffffff0 - 6 + 1, pk.ctypes.data, None) == -1
        assert b"2^32 - 16" in e._lib.blsgpu_last_error(e._ctx)
        assert e._lib.blsgpu_keyset_update(e._ctx, ks.id, 1, 1, None, pk.ctypes.data, None) == -1   # a NULL key_idx
        assert e._lib.blsgpu_keyset_append(e._ctx, ks.id, 1, 1, None, None) == -1                   # a NULL pks
        assert e._lib.blsgpu_keyset_update(e._ctx, ks.id, 1, 0, None, None, None) == 0             # k = 0
        assert e._lib.blsgpu_keyset_append(e._ctx, ks.id, 1, 0, None, None) == 0
        assert len(ks) == 6 and results() == before
        assert other.verify_batch_keyed(foreign, 0, list(range(6)), sigs, [b"e"] * 6).tolist() == [0] * 6
        assert e.verify_batch(2, 0, kb, sigs, [b"e"] * 6).tolist() == [0] * 6
        ks.close()
    finally:
        other.close()
        e.close()


def test_update_at_scale_equals_a_fresh_set(eng, B):
    """A 2^20-key G2Impl set, 65,536 keys updated (1,000 of them to undecodable bytes), signatures planted bad"""
    rng = np.random.default_rng(20)
    n, base, k, items = 1 << 20, 1 << 16, 1 << 16, 1 << 18
    secret = np.zeros((base + k, 32), dtype=np.uint8)
    secret[:, 8:] = rng.integers(0, 256, size=(base + k, 24), dtype=np.uint8)
    secret[:, 31] |= 1
    kb_all, _ = eng.testdata_sign(2, 0, secret.reshape(-1), *B.pack_messages([b""] * (base + k)))
    kb_all = kb_all.reshape(base + k, 48)
    owner = np.arange(n) % base                  # the secret of every key
    kb = kb_all[owner].copy()
    ks = eng.key_set(2, kb.reshape(-1))
    try:
        upd = rng.permutation(n)[:k].astype(np.uint32)
        new = kb_all[base:].copy()
        undecodable = rng.permutation(k)[:1000]
        new[undecodable] = np.frombuffer(_off_curve(1), dtype=np.uint8)
        st = eng.update_key_set(ks, upd, new.reshape(-1))
        assert np.flatnonzero(st).tolist() == sorted(undecodable.tolist())
        kb[upd] = new
        owner[upd] = base + np.arange(k)
        key_idx = np.concatenate([upd[rng.integers(0, k, size=items // 2)], rng.integers(0, n, size=items // 2)]).astype(np.uint32)
        data, off = B.pack_messages([b"scale %d" % (i % 97) for i in range(items)])
        _, sg = eng.testdata_sign(2, 0, secret[owner[key_idx]].reshape(-1), data, off)
        sg = sg.reshape(items, 96).copy()
        bad = sorted(rng.permutation(items)[:500].tolist())
        sg[bad] = sg[(np.array(bad) + 1) % items]
        got = eng.verify_batch_keyed_packed(ks, 0, key_idx, sg.reshape(-1), data, off)
        fresh = eng.key_set(2, kb.reshape(-1))
        try:
            _same(ks.status, fresh.status)
            want = eng.verify_batch_keyed_packed(fresh, 0, key_idx, sg.reshape(-1), data, off)
        finally:
            fresh.close()
        assert got.tobytes() == want.tobytes()
        hits = set(np.flatnonzero(np.isin(key_idx, upd[undecodable])).tolist())
        assert set(np.flatnonzero(got).tolist()) == hits | set(bad)
        assert len(hits) > 100
    finally:
        ks.close()


def test_appends_free_their_device_memory(B):
    import torch
    rng = np.random.default_rng(18)
    n, k = 1 << 18, 1000
    secret = np.zeros((4096, 32), dtype=np.uint8)
    secret[:, 8:] = rng.integers(0, 256, size=(4096, 24), dtype=np.uint8)
    secret[:, 31] |= 1
    e = B.Engine([0])
    try:
        kb, member = e.testdata_sign(2, 0, secret.reshape(-1), *B.pack_messages([b"a"] * 4096))
        big = np.tile(kb, n // 4096)

        def grow(ks):
            for fmt in (O.MODERN, O.LEGACY):   # both views
                sg = member[:288] if fmt == O.MODERN else e.recode_points_packed(2, member[:288], 1, 0)
                assert e.aggregate_secure_batch_keyed_packed(ks, np.array([0, 3], dtype=np.uint64), np.arange(3, dtype=np.uint32), sg, fmt)[0].tolist() == [0]
            for r in range(4):
                st = e.append_key_set(ks, kb[48 * k * r:48 * k * (r + 1)])
                assert not st.any()
            assert len(ks) == n + 4 * k
            idx = np.array([n + 5, 5, n + 3 * k + 5], dtype=np.uint32)   # keys n + 5 and 5 are equal
            sg = np.concatenate([member[480:576], member[480:576], member[96 * (3 * k + 5):96 * (3 * k + 6)]])
            st, agg = e.aggregate_secure_batch_keyed_packed(ks, np.array([0, 3], dtype=np.uint64), idx, sg)
            assert st.tolist() == [0]

        warm = e.key_set(2, big)
        grow(warm)   # loads the kernels and sizes the arena for these calls
        warm.close()
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info(0)[0]
        ks = e.key_set(2, big)
        grow(ks)
        assert torch.cuda.mem_get_info(0)[0] < free0 - (145 + 2 * 52) * n + 2 * 2 ** 20
        ks.close()
        assert abs(torch.cuda.mem_get_info(0)[0] - free0) <= 2 * 2 ** 20
    finally:
        e.close()

"""blsgpu_aggregate_verify_batch: q x AggregateSignature::verify in one call.  Every status and index must equal what
blsgpu_aggregate_verify returns for that aggregate alone (and, on a sample, the big-int oracle); rejections must be exact
whatever the batch holds, with one pipeline per call."""
import hashlib
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import bls_oracle as O


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


def _scalars(rnd, n):
    return np.frombuffer(b"".join(rnd.randrange(1, O.R).to_bytes(32, "big") for _ in range(n)), dtype=np.uint8)


def _sign(eng, B, impl, scheme, rnd, msgs):
    """(pk list, sig list) for one fresh key per message (Modern encodings)."""
    pks, sigs = eng.testdata_sign(impl, scheme, _scalars(rnd, len(msgs)), *B.pack_messages(msgs))
    pl, sl = B.pk_len(impl), B.sig_len(impl)
    return [pks[i * pl:(i + 1) * pl].tobytes() for i in range(len(msgs))], [sigs[i * sl:(i + 1) * sl].tobytes() for i in range(len(msgs))]


def _groups(impl):
    return (1, 2) if impl == 2 else (2, 1)   # (public-key group, signature group)


def _flat(B, impl, sets, sigs):
    """Packed form of [(pks, msgs)] + signatures for aggregate_verify_batch_packed."""
    soff = np.zeros(len(sets) + 1, dtype=np.uint64)
    soff[1:] = np.cumsum([len(p) for p, _ in sets])
    pk = np.frombuffer(b"".join(b"".join(p) for p, _ in sets), dtype=np.uint8)
    data, off = B.pack_messages([m for _, ms in sets for m in ms])
    return soff, pk, data, off, np.frombuffer(b"".join(sigs), dtype=np.uint8)


def _single(eng, impl, scheme, sets, sigs, fmt):
    out = [eng.aggregate_verify_status(impl, scheme, p, m, s, fmt) for (p, m), s in zip(sets, sigs)]
    return [s for s, _ in out], [list(i) for _, i in out]


SIZES = [1, 5, 6, 7, 12, 13, 40]


@pytest.mark.parametrize("fmt", [O.MODERN, O.LEGACY])
@pytest.mark.parametrize("impl", [2, 1])
def test_mixed_batch_equals_the_single_call_and_the_oracle(eng, B, impl, fmt):
    pkg, sgg = _groups(impl)
    pl, sl = B.pk_len(impl), B.sig_len(impl)
    for scheme in (0, 1, 2):
        rnd = random.Random(1000 * impl + 10 * fmt + scheme)
        sets, sigs, names = [], [], []

        def agg(tag, n, shared=()):
            msgs = [b"%s/%d/%d" % (tag, scheme, i) for i in range(n - len(shared))] + list(shared)
            p, s = _sign(eng, B, impl, scheme, rnd, msgs)
            return p, msgs, eng.sum_points(sgg, s)

        for n in SIZES:                                       # valid aggregates across the group boundaries
            p, m, s = agg(b"ok%d" % n, n)
            sets.append((p, m)); sigs.append(s); names.append("valid%d" % n)
        p, m, s = agg(b"wrong", 13)                           # a signature over different messages
        _, _, s_other = agg(b"other", 13)
        sets.append((p, m)); sigs.append(s_other); names.append("wrong")
        p, m, s = agg(b"wrong1", 1)
        sets.append((p, m)); sigs.append(sigs[0]); names.append("wrong1")
        p, m, s = agg(b"swap", 7)
        m2 = list(m); m2[2], m2[5] = m2[5], m2[2]
        sets.append((p, m2)); sigs.append(s); names.append("swapped")
        p, m, s = agg(b"badpk", 12)
        p2 = list(p); p2[5] = _off_curve(pkg)
        sets.append((p2, m)); sigs.append(s); names.append("undecodable_pk")
        p, m, s = agg(b"idpk", 6)
        p2 = list(p); p2[2] = _ident(pl)
        sets.append((p2, m)); sigs.append(s); names.append("identity_pk")
        p, m, s = agg(b"dup", 12)
        m2 = list(m); m2[9] = m2[3]
        sets.append((p, m2)); sigs.append(s); names.append("duplicate")
        for tag in (b"shareA", b"shareB"):                    # one message in two different aggregates: both valid
            p, m, s = agg(tag, 5, shared=[b"the same message"])
            sets.append((p, m)); sigs.append(s); names.append("shared_" + tag.decode())
        p, m, s = agg(b"idsig", 5)
        sets.append((p, m)); sigs.append(_ident(sl)); names.append("identity_sig")
        p, m, s = agg(b"badsig", 5)
        sets.append((p, m)); sigs.append(_off_curve(sgg)); names.append("undecodable_sig")
        sets.append(([], [])); sigs.append(sigs[1]); names.append("empty")
        p, m, s = agg(b"last", 40)
        sets.append((p, m)); sigs.append(s); names.append("valid40_last")
        if fmt == O.LEGACY:
            def conv(group, encs):
                if not encs:
                    return []
                st, outs = eng.recode_points(group, encs, O.MODERN, O.LEGACY)
                return [o if s == 0 else O.modern_to_legacy(e) for e, s, o in zip(encs, st.tolist(), outs)]
            sets = [(conv(pkg, p), m) for p, m in sets]
            sigs = conv(sgg, sigs)
        st, idx = eng.aggregate_verify_batch_status(impl, scheme, sets, sigs, fmt)
        want_st, want_idx = _single(eng, impl, scheme, sets, sigs, fmt)
        assert st.tolist() == want_st, list(zip(names, st.tolist(), want_st))
        assert idx.tolist() == want_idx, list(zip(names, idx.tolist(), want_idx))
        got = dict(zip(names, zip(st.tolist(), idx.tolist())))
        assert all(got["valid%d" % n] == (0, [-1, -1]) for n in SIZES) and got["valid40_last"][0] == 0
        assert got["shared_shareA"][0] == 0 and got["shared_shareB"][0] == 0
        assert got["wrong"][0] == 1 and got["wrong1"][0] == 1 and got["swapped"][0] == 1 and got["empty"][0] == 1
        assert got["undecodable_pk"][0] in (O.ERR_DESERIALIZE, O.ERR_LEGACY_FORMAT) and got["undecodable_pk"][1] == [5, -1]
        assert got["identity_pk"] == (3, [3, -1])
        assert got["duplicate"] == ((8, [3, 9]) if scheme == 0 else (1, [-1, -1]))
        assert got["identity_sig"][0] == 2 and got["undecodable_sig"][0] in (O.ERR_DESERIALIZE, O.ERR_LEGACY_FORMAT)
        if scheme == 0:   # a sample end to end against the big-int oracle
            for name in ("valid1", "wrong1", "undecodable_pk", "identity_pk", "identity_sig", "empty"):
                j = names.index(name)
                assert O.aggregate_verify(impl, scheme, fmt, sets[j][0], sets[j][1], sigs[j])[0] == st[j], name


def _library(eng, B, rnd, impl=2, scheme=0, variants=2, sizes=range(1, 65)):
    """Valid aggregates of every size, `variants` of each: {size: [(pks, msgs, sig), ...]}."""
    sgg = _groups(impl)[1]
    lib = {}
    for n in sizes:
        lib[n] = []
        for v in range(variants):
            msgs = [hashlib.sha256(b"lib%d/%d/%d" % (n, v, i)).digest()[:8 + i % 24] for i in range(n)]
            p, s = _sign(eng, B, impl, scheme, rnd, msgs)
            lib[n].append((p, msgs, eng.sum_points(sgg, s)))
    return lib


def test_failure_search_is_exact(eng, B):
    """q = 2,000 aggregates of seeded sizes 1-64, with 0, 1, 16 and 300 wrong ones at seeded positions: the rejected set is
    exactly the planted one.  Again with 128-bit scalars, and with a pinned salt against a fresh one."""
    rnd = random.Random(2024)
    lib = _library(eng, B, rnd)
    q = 2000
    sizes = [rnd.randint(1, 64) for _ in range(q)]
    base = [lib[n][j % 2] for j, n in enumerate(sizes)]
    sets = [(p, m) for p, m, _ in base]
    good_sigs = [s for _, _, s in base]
    soff, pk, data, off, _ = _flat(B, 2, sets, good_sigs)

    def planted(nbad):
        bad = sorted(rnd.sample(range(q), nbad))
        sigs = list(good_sigs)
        for j in bad:   # a valid point: the signature of another aggregate
            sigs[j] = lib[sizes[j] % 64 + 1][0][2]
        return bad, np.frombuffer(b"".join(sigs), dtype=np.uint8)

    cases = [planted(n) for n in (0, 1, 16, 300)]
    for bad, sg in cases:
        st, idx = eng.aggregate_verify_batch_packed(2, 0, soff, pk, data, off, sg)
        assert [j for j in range(q) if st[j]] == bad and all(st[j] == 1 for j in bad)
        assert (idx == -1).all()
    bad, sg = cases[2]
    e2 = B.Engine([0])
    try:
        e2.set_rlc_bits(128)
        st, _ = e2.aggregate_verify_batch_packed(2, 0, soff, pk, data, off, sg)
        assert [j for j in range(q) if st[j]] == bad
        e2.set_rlc_bits(64)
        e2.set_rlc_salt(bytes(range(32)))
        pinned, _ = e2.aggregate_verify_batch_packed(2, 0, soff, pk, data, off, sg)
        fresh, _ = eng.aggregate_verify_batch_packed(2, 0, soff, pk, data, off, sg)
        assert pinned.tolist() == fresh.tolist() == st.tolist()
    finally:
        e2.close()


def test_large_aggregate_and_several_miller_passes(eng, B, monkeypatch):
    """One aggregate of 100,000 pairs (cfg 4's shape), valid and wrong, equals blsgpu_aggregate_verify; then a batch whose
    slots go through the Miller kernels in several passes (chunk override) finds its wrong aggregates exactly."""
    rnd = random.Random(5)
    n = 100_000
    msgs = [hashlib.sha256(b"big%d" % i).digest() for i in range(n)]
    pks, sigs = eng.testdata_sign(2, 0, _scalars(rnd, n), *B.pack_messages(msgs))
    agg = eng.sum_points(2, sigs)
    wrong = eng.sum_points(2, sigs[:-96])
    data, off = B.pack_messages(msgs)
    soff = np.array([0, n, 2 * n], dtype=np.uint64)
    off2 = np.concatenate([off, off[1:] + off[-1]])
    st, idx = eng.aggregate_verify_batch_packed(2, 0, soff, np.concatenate([pks, pks]), np.concatenate([data, data]), off2,
                                                np.frombuffer(agg + wrong, dtype=np.uint8))
    pk_list = [pks[i * 48:(i + 1) * 48].tobytes() for i in range(n)]
    assert st.tolist() == [eng.aggregate_verify_status(2, 0, pk_list, msgs, agg)[0], eng.aggregate_verify_status(2, 0, pk_list, msgs, wrong)[0]]
    assert st.tolist() == [0, 1] and (idx == -1).all()

    lib = _library(eng, B, rnd, scheme=1, variants=1, sizes=range(1, 41))
    q = 300
    sizes = [rnd.randint(1, 40) for _ in range(q)]
    sets = [(lib[s][0][0], lib[s][0][1]) for s in sizes]
    sigs = [lib[s][0][2] for s in sizes]
    bad = sorted(rnd.sample(range(q), 7))
    for j in bad:
        sigs[j] = lib[sizes[j] % 40 + 1][0][2]
    monkeypatch.setenv("BLSGPU_M6_CHUNK", "1200")
    soff, pk, data, off, sg = _flat(B, 2, sets, sigs)
    assert sum(sizes) > 3 * 1200
    st, _ = eng.aggregate_verify_batch_packed(2, 1, soff, pk, data, off, sg)
    assert [j for j in range(q) if st[j]] == bad


def _levels(n):
    k = 1
    while n > 1:
        n = (n + 15) // 16
        k += 1
    return k


def test_one_pipeline_per_call(eng, B):
    """Launches of an all-valid call do not grow with the number of aggregates: with equal sizes they differ only by the
    depth of the two 16-ary trees (the digest over pairs and aggregates, the product / sum tree over aggregates)."""
    rnd = random.Random(8)
    msgs = [b"launch%d" % i for i in range(6)]
    p, s = _sign(eng, B, 2, 0, rnd, msgs)
    agg = eng.sum_points(2, s)
    counts = {}
    for q in (100, 1000, 4000):
        soff, pk, data, off, sg = _flat(B, 2, [(p, msgs)] * q, [agg] * q)
        before = eng.launch_count()
        st, _ = eng.aggregate_verify_batch_packed(2, 0, soff, pk, data, off, sg)
        counts[q] = eng.launch_count() - before
        assert st.tolist() == [0] * q
    for a, b in ((100, 1000), (1000, 4000)):
        depth = (_levels(7 * b) - _levels(7 * a)) + 2 * (_levels(b) - _levels(a))
        assert counts[b] - counts[a] == depth, counts
    assert counts[1000] == counts[4000]


def test_context_on_two_devices_cuts_the_aggregates(eng, B):
    """A context on two GPUs verifies contiguous runs of aggregates on each device: statuses and indices equal the
    single-device ones, with wrong, duplicate-message and identity cases in the second device's run."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    rnd = random.Random(31)
    lib = _library(eng, B, rnd, variants=1)
    q = 400
    sizes = [rnd.randint(1, 64) for _ in range(q)]
    sets = [(list(lib[s][0][0]), list(lib[s][0][1])) for s in sizes]
    sigs = [lib[s][0][2] for s in sizes]
    assert sum(sizes) >= 2 * 4096
    big = [j for j in range(q) if sizes[j] >= 12]
    for j in (big[1], big[-1]):                                 # wrong: another size's signature
        sigs[j] = lib[sizes[j] % 64 + 1][0][2]
    j = big[-2]; sets[j][1][9] = sets[j][1][3]                  # duplicate messages (Basic)
    j = big[-3]; sets[j][0][4] = _ident(48)                     # identity public key
    j = big[-4]; sigs[j] = _ident(96)                           # identity signature
    soff, pk, data, off, sg = _flat(B, 2, sets, sigs)
    want_st, want_idx = eng.aggregate_verify_batch_packed(2, 0, soff, pk, data, off, sg)
    assert sorted(set(want_st.tolist())) == [0, 1, 2, 3, 8]
    e2 = B.Engine([0, 1])
    try:
        before = e2.launch_count()
        st, idx = e2.aggregate_verify_batch_packed(2, 0, soff, pk, data, off, sg)
        assert st.tolist() == want_st.tolist() and idx.tolist() == want_idx.tolist()
        assert e2.launch_count() - before > 2 * 20            # both devices launched their own pipeline
    finally:
        e2.close()


def test_decreasing_offsets_are_refused(eng, B):
    rnd = random.Random(4)
    msgs = [b"a", b"b", b"c"]
    p, s = _sign(eng, B, 2, 0, rnd, msgs)
    agg = eng.sum_points(2, s)
    soff, pk, data, off, sg = _flat(B, 2, [(p, msgs), (p, msgs)], [agg, agg])
    assert eng.aggregate_verify_batch_packed(2, 0, soff, pk, data, off, sg)[0].tolist() == [0, 0]
    with pytest.raises(B.EngineError, match=r"\(-1\)"):
        eng.aggregate_verify_batch_packed(2, 0, np.array([0, 4, 3], dtype=np.uint64), pk, data, off, sg)
    bad_off = off.copy()
    bad_off[2], bad_off[3] = bad_off[3], bad_off[2]
    with pytest.raises(B.EngineError, match=r"\(-1\)"):
        eng.aggregate_verify_batch_packed(2, 0, soff, pk, data, bad_off, sg)

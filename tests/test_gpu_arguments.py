"""The argument rules of include/blsgpu.h ("Arguments"), entry point by entry point: every refused call returns BLSGPU_E_ARG,
names its entry point in blsgpu_last_error and leaves the context working; calls over no items accept NULL buffers."""
import ctypes
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import bls_oracle as O

E_ARG = -1
N = 4
MISSING_SET = 0xFFFFFFFFFFFF


@pytest.fixture(scope="module")
def env():
    import blsful_b200 as B
    eng = B.Engine([0])
    rnd = random.Random(5150)
    k = np.frombuffer(b"".join(rnd.randrange(1, O.R).to_bytes(32, "big") for _ in range(N)), dtype=np.uint8)
    data, off = B.pack_messages([b"arguments-%d" % i for i in range(N)])
    pks, sigs = eng.testdata_sign(2, 0, k, data, off)
    ks = eng.key_set(2, pks)
    yield eng, dict(B=B, k=k, data=data, off=off, pks=pks, sigs=sigs, ks=ks)
    eng.close()


def u64(*v):
    return np.array(v, dtype=np.uint64)


def specs(d):
    """entry point -> (arguments after ctx in declaration order, offset array -> the buffer it delimits (None: a set of
    members), pointers that may be NULL with items, pointers a call over no items still needs)"""
    pks, sigs, data, off, k = d["pks"], d["sigs"], d["data"], d["off"], d["k"]
    ks = d["ks"].id
    idx = np.arange(N, dtype=np.uint32)
    midx = np.zeros(N, dtype=np.uint32)
    off1 = u64(0, off[1])
    two = u64(0, 2, 4)  # two sets of two members
    shares = np.frombuffer(b"".join(i.to_bytes(32, "big") + bytes(pks[48 * (i - 1):48 * i]) for i in range(1, N + 1)), dtype=np.uint8)
    id_pk = np.frombuffer(b"".join(bytes(32) + bytes(pks[48 * i:48 * i + 48]) for i in range(N)), dtype=np.uint8)
    id_sig = np.frombuffer(b"".join(bytes(32) + bytes(sigs[96 * i:96 * i + 96]) for i in range(N)), dtype=np.uint8)
    tagged = np.frombuffer(b"".join(b"\x00" + bytes(sigs[96 * i:96 * i + 96]) for i in range(N)), dtype=np.uint8)
    rec = lambda L: np.arange(N + 1, dtype=np.uint64) * np.uint64(L)  # noqa: E731
    st = lambda: np.zeros(64, dtype=np.uint8)  # noqa: E731
    out = lambda: np.zeros(N * 96 + 576, dtype=np.uint8)  # noqa: E731
    i64 = lambda: np.zeros(2 * N, dtype=np.int64)  # noqa: E731
    u64o = lambda: np.zeros(1, dtype=np.uint64)  # noqa: E731
    i32o = lambda: np.zeros(1, dtype=np.int32)  # noqa: E731
    dst = np.frombuffer(b"ARGUMENTS-DST", dtype=np.uint8)
    S = {}
    S["blsgpu_verify_batch"] = (dict(impl=2, scheme=0, format=1, n=N, pks=pks, sigs=sigs, msgs=data, msg_off=off, status_out=st()),
                                {"msg_off": "msgs"}, [], [])
    S["blsgpu_verify_batch_grouped"] = (dict(impl=2, scheme=0, format=1, n=N, pks=pks, sigs=sigs, msg_idx=idx, q=N, msgs=data, msg_off=off,
                                             status_out=st()), {"msg_off": "msgs"}, [], [])
    S["blsgpu_keyset_create"] = (dict(impl=2, format=1, n=N, pks=pks, status_out=st(), keyset_out=u64o()), {}, ["status_out"], ["keyset_out"])
    S["blsgpu_verify_batch_keyed"] = (dict(keyset=ks, scheme=0, format=1, n=N, key_idx=idx, sigs=sigs, msgs=data, msg_off=off, status_out=st()),
                                      {"msg_off": "msgs"}, [], [])
    S["blsgpu_verify_batch_grouped_keyed"] = (dict(keyset=ks, scheme=0, format=1, n=N, key_idx=idx, sigs=sigs, msg_idx=midx, q=1, msgs=data,
                                                   msg_off=off1, status_out=st()), {"msg_off": "msgs"}, [], [])
    S["blsgpu_miller_partial"] = (dict(impl=2, scheme=0, format=1, n=N, pks=pks, sigs=sigs, msgs=data, msg_off=off, gt_out=out(), sum_out=out()),
                                  {"msg_off": "msgs"}, [], ["gt_out", "sum_out"])
    S["blsgpu_pop_verify_batch"] = (dict(impl=2, format=1, n=N, pks=pks, sigs=sigs, status_out=st()), {}, [], [])
    S["blsgpu_aggregate_verify"] = (dict(impl=2, scheme=0, format=1, n=N, pks=pks, msgs=data, msg_off=off, sig=sigs, status_out=st(),
                                         index_out=i64()), {"msg_off": "msgs"}, ["index_out"], ["sig", "status_out", "msg_off"])
    S["blsgpu_aggregate_verify_batch"] = (dict(impl=2, scheme=0, format=1, q=2, set_off=two, pks=pks, msgs=data, msg_off=off, sigs=sigs,
                                               status_out=st(), index_out=i64()), {"msg_off": "msgs", "set_off": None}, ["index_out"], [])
    S["blsgpu_sum_points"] = (dict(group=2, format=1, n=N, points=sigs, out=out(), status_out=st(), bad_index_out=i64()), {}, ["bad_index_out"],
                              ["out", "status_out"])
    S["blsgpu_verify_secure_batch"] = (dict(impl=2, scheme=0, format=1, q=2, key_off=two, pks=pks, sigs=sigs, msgs=data, msg_off=u64(0, 3, 6),
                                            status_out=st()), {"msg_off": "msgs", "key_off": None}, [], [])
    S["blsgpu_aggregate_secure_batch"] = (dict(impl=2, format=1, q=2, key_off=two, pks=pks, member_sigs=sigs, out_sigs=out(), status_out=st()),
                                          {"key_off": None}, [], [])
    S["blsgpu_verify_secure_batch_keyed"] = (dict(keyset=ks, scheme=0, format=1, q=2, key_off=two, key_idx=idx, sigs=sigs, msgs=data,
                                                  msg_off=u64(0, 3, 6), status_out=st()), {"msg_off": "msgs", "key_off": None}, [], [])
    S["blsgpu_aggregate_secure_batch_keyed"] = (dict(keyset=ks, format=1, q=2, key_off=two, key_idx=idx, member_sigs=sigs, out_sigs=out(),
                                                     status_out=st()), {"key_off": None}, [], [])
    S["blsgpu_verify_multisig_batch"] = (dict(impl=2, scheme=0, format=1, q=2, key_off=two, pks=pks, sigs=sigs, msgs=data, msg_off=u64(0, 3, 6),
                                              status_out=st()), {"msg_off": "msgs", "key_off": None}, [], [])
    S["blsgpu_verify_multisig_batch_keyed"] = (dict(keyset=ks, scheme=0, format=1, q=2, key_off=two, key_idx=idx, sigs=sigs, msgs=data,
                                                    msg_off=u64(0, 3, 6), status_out=st()), {"msg_off": "msgs", "key_off": None}, [], [])
    S["blsgpu_sum_points_batch"] = (dict(group=2, format=1, q=2, set_off=two, points=sigs, out=out(), status_out=st(), bad_index_out=i64()),
                                    {"set_off": None}, ["bad_index_out"], [])
    S["blsgpu_hash_to_curve_batch"] = (dict(group=2, n=N, msgs=data, msg_off=off, dst=dst, dst_len=dst.size, out=out()), {"msg_off": "msgs"}, [],
                                       ["msg_off", "dst"])
    S["blsgpu_recode_points"] = (dict(group=1, format_in=1, format_out=0, n=N, inp=pks, out=out(), status_out=st()), {}, [], [])
    S["blsgpu_fp_mul_batch"] = (dict(variant=0, n=1, a=np.zeros(48, dtype=np.uint8), b=np.zeros(48, dtype=np.uint8), out=out()), {}, [], [])
    S["blsgpu_pairing_product_is_one"] = (dict(n=1, g1=pks, g2=sigs, is_one_out=i32o()), {}, [], ["is_one_out"])
    S["blsgpu_testdata_sign"] = (dict(impl=2, scheme=0, n=N, scalars32=k, msgs=data, msg_off=off, out_pks=out(), out_sigs=out()),
                                 {"msg_off": "msgs"}, [], [])
    S["blsgpu_combine_shares_batch"] = (dict(group=1, q=2, share_off=two, shares=shares, out=out(), status_out=st()), {"share_off": None}, [], [])
    S["blsgpu_verify_batch_wire"] = (dict(impl=2, n=N, pks=pks, tagged_sigs=tagged, msgs=data, msg_off=off, status_out=st()), {"msg_off": "msgs"},
                                     [], ["msg_off"])
    S["blsgpu_pairing_check_batch"] = (dict(q=2, pair_off=two, g1_points=pks, g2_points=sigs, ok_out=st(), status_out=st()), {"pair_off": None},
                                       [], [])
    S["blsgpu_signcrypt_valid_batch"] = (dict(impl=2, scheme=0, n=N, u_points=pks, w_points=sigs, v_bytes=data, v_off=off, ok_out=st(),
                                              status_out=st()), {"v_off": "v_bytes"}, [], [])
    S["blsgpu_signcrypt_verify_share_batch"] = (dict(impl=2, scheme=0, n=N, shares=pks, pk_shares=pks, u_points=pks, w_points=sigs, v_bytes=data,
                                                     v_off=off, ok_out=st(), status_out=st()), {"v_off": "v_bytes"}, [], [])
    S["blsgpu_pok_verify_batch"] = (dict(impl=2, scheme=0, n=N, commitments=sigs, proofs=sigs, pks=pks, challenges32=k, msgs=data, msg_off=off,
                                         status_out=st()), {"msg_off": "msgs"}, [], [])
    S["blsgpu_verify_batch_records"] = (dict(impl=2, format=1, scheme_or_tagged=0, n=N, pk_bytes=pks, pk_off=rec(48), sig_bytes=sigs,
                                             sig_off=rec(96), msgs=data, msg_off=off, status_out=st()),
                                        {"pk_off": "pk_bytes", "sig_off": "sig_bytes", "msg_off": "msgs"}, [], [])
    S["blsgpu_verify_share_batch"] = (dict(impl=2, scheme=0, n=N, pk_shares=id_pk, sig_shares=id_sig, msgs=data, msg_off=off, status_out=st()),
                                      {"msg_off": "msgs"}, [], [])
    return S


ENTRIES = ["blsgpu_verify_batch", "blsgpu_verify_batch_grouped", "blsgpu_keyset_create", "blsgpu_verify_batch_keyed",
           "blsgpu_verify_batch_grouped_keyed", "blsgpu_miller_partial", "blsgpu_pop_verify_batch", "blsgpu_aggregate_verify",
           "blsgpu_aggregate_verify_batch", "blsgpu_sum_points", "blsgpu_verify_secure_batch", "blsgpu_aggregate_secure_batch",
           "blsgpu_verify_secure_batch_keyed", "blsgpu_aggregate_secure_batch_keyed", "blsgpu_verify_multisig_batch",
           "blsgpu_verify_multisig_batch_keyed", "blsgpu_sum_points_batch", "blsgpu_hash_to_curve_batch", "blsgpu_recode_points",
           "blsgpu_fp_mul_batch", "blsgpu_pairing_product_is_one", "blsgpu_testdata_sign", "blsgpu_combine_shares_batch",
           "blsgpu_verify_batch_wire", "blsgpu_pairing_check_batch", "blsgpu_signcrypt_valid_batch", "blsgpu_signcrypt_verify_share_batch",
           "blsgpu_pok_verify_batch", "blsgpu_verify_batch_records", "blsgpu_verify_share_batch"]
COUNTS = ("n", "q")
INTS = ("impl", "scheme", "format", "group", "variant", "format_in", "format_out", "scheme_or_tagged", "keyset", "dst_len")
# the null buffers with bytes that the parent of the argument-rules change passed on to the CUDA runtime instead of refusing
NEWLY_REFUSED = {("blsgpu_miller_partial", "msgs"), ("blsgpu_aggregate_verify", "msgs"), ("blsgpu_hash_to_curve_batch", "msgs"),
                 ("blsgpu_testdata_sign", "msgs"), ("blsgpu_verify_secure_batch", "msgs"), ("blsgpu_verify_secure_batch_keyed", "msgs"),
                 ("blsgpu_pok_verify_batch", "msgs"), ("blsgpu_signcrypt_valid_batch", "v_bytes"),
                 ("blsgpu_signcrypt_verify_share_batch", "v_bytes")}
RAGGED = ("msgs", "v_bytes", "pk_bytes", "sig_bytes")


def rows():
    """(id, entry point, how to spoil its arguments, expected rc, substring of the error)"""
    import types
    d = types.SimpleNamespace(pks=np.zeros(N * 48, np.uint8), sigs=np.zeros(N * 96, np.uint8), data=np.zeros(48, np.uint8),
                              off=np.arange(N + 1, dtype=np.uint64) * np.uint64(12), k=np.zeros(N * 32, np.uint8), ks=types.SimpleNamespace(id=1))
    out = []
    for name in ENTRIES:
        args, offs, optional, _ = specs(vars(d))[name]
        for a, v in args.items():
            if isinstance(v, np.ndarray) and a not in optional:
                sub = "is null" if a in RAGGED else None
                tag = "-newly_refused" if (name, a) in NEWLY_REFUSED else ""
                out.append((f"{name}-null-{a}{tag}", name, ("null", a), E_ARG, sub))
        for a in offs:
            out.append((f"{name}-decreasing-{a}", name, ("decreasing", a), E_ARG, "non-decreasing"))
        for a in args:
            if a in INTS and a not in ("keyset", "dst_len"):
                out.append((f"{name}-unknown-{a}", name, ("set", a, 7), E_ARG, None))
        if "keyset" in args:
            out.append((f"{name}-unknown-set", name, ("set", "keyset", MISSING_SET), E_ARG, "is not held"))
            out.append((f"{name}-key-index", name, ("key_idx",), E_ARG, "key_idx["))
        out.append((f"{name}-empty", name, ("empty",), 0, None))
    # Legacy is refused by the secure calls for Bls12381G1Impl
    out.append(("blsgpu_verify_secure_batch-legacy-g1", "blsgpu_verify_secure_batch", ("legacy_g1",), E_ARG, "Legacy"))
    # a NULL buffer whose members span nothing is accepted whatever the first offset
    for name, bufs in [("blsgpu_verify_secure_batch", ["pks"]), ("blsgpu_aggregate_secure_batch", ["pks", "member_sigs"]),
                       ("blsgpu_combine_shares_batch", ["shares"]), ("blsgpu_pairing_check_batch", ["g1_points", "g2_points"])]:
        out.append((f"{name}-null-empty-span", name, ("empty_span", bufs), 0, None))
    out.append(("blsgpu_verify_batch_records-null-msgs-empty-messages", "blsgpu_verify_batch_records", ("null_empty_msgs",), 0, None))
    return out


ROWS = rows()


def call(eng, name, args):
    fn = getattr(eng._lib, name)
    ptrs = []
    for v, t in zip(args.values(), fn.argtypes[1:]):
        ptrs.append(ctypes.cast(ctypes.c_void_p(v.ctypes.data), t) if isinstance(v, np.ndarray) else v)
    return fn(eng._ctx, *ptrs)


def spoiled(d, name, how):
    args, offs, _, keep = specs(d)[name]
    args = dict(args)
    kind = how[0]
    if kind == "null":
        args[how[1]] = None
    elif kind == "decreasing":
        o = args[how[1]].copy()
        o[0] = o[1] + np.uint64(1)
        args[how[1]] = o
    elif kind == "set":
        args[how[1]] = how[2]
    elif kind == "key_idx":
        idx = args["key_idx"].copy()
        idx[-1] = 1000
        args["key_idx"] = idx
    elif kind == "empty":
        for a, v in args.items():
            if a in COUNTS:
                args[a] = 0
            elif isinstance(v, np.ndarray) and a not in keep:
                args[a] = None
        if "msg_off" in keep:
            args["msg_off"] = u64(0)
    elif kind == "legacy_g1":
        args.update(impl=1, format=0)
    elif kind == "empty_span":
        key = "share_off" if "share_off" in args else "pair_off" if "pair_off" in args else "key_off"
        args[key] = u64(2, 2)
        args["q"] = 1
        for b in how[1]:
            args[b] = None
        if "msg_off" in args:
            args["msg_off"] = u64(0, 3)
    elif kind == "null_empty_msgs":
        args["msgs"] = None
        args["msg_off"] = np.zeros(N + 1, dtype=np.uint64)
    return args


@pytest.mark.parametrize("row", ROWS, ids=[r[0] for r in ROWS])
def test_argument_rule(env, row):
    eng, d = env
    _, name, how, want, sub = row
    rc = call(eng, name, spoiled(d, name, how))
    if want == E_ARG:
        msg = eng._lib.blsgpu_last_error(eng._ctx).decode()
        assert rc == E_ARG, (rc, msg)
        assert name in msg, msg
        if sub:
            assert sub in msg, msg
    else:
        assert rc == want, (rc, eng._lib.blsgpu_last_error(eng._ctx))
    # the context keeps working
    st = eng.verify_batch_packed(2, 0, d["pks"], d["sigs"], d["data"], d["off"])
    assert st.tolist() == [0] * N

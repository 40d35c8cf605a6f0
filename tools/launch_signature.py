"""Launch signature of the engine: a fixed matrix of calls with a pinned salt, one line per call holding the sha256 of its
status / index outputs, its number of kernel launches and the per-kernel launch counts of blsgpu_last_kernel_ms.

Two builds of libblsgpu.so that compute the same results with the same launches print the same lines, so a host-side
change can be checked by running this once per build (BLSGPU_LIB selects the library) and comparing the outputs.

    BLSGPU_LIB=/path/to/libblsgpu.so python tools/launch_signature.py [--devices 0,1] > sig.txt
"""
import argparse
import hashlib
import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "agora-blsful_b200")]

import blsful_b200 as B  # noqa: E402
from oracle import bls_oracle as O  # noqa: E402

SALT = bytes(range(32))


def keys(rnd, n):
    return np.frombuffer(b"".join(rnd.randrange(1, O.R).to_bytes(32, "big") for _ in range(n)), dtype=np.uint8)


def spoil(sigs, sl, bad):
    """signature i of `bad` replaced by signature i + 1: a valid point that fails its own equation"""
    s = sigs.copy().reshape(-1, sl)
    n = s.shape[0]
    for i in bad:
        s[i] = sigs.reshape(-1, sl)[(i + 1) % n]
    return s.reshape(-1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--devices", default="0")
    args = ap.parse_args()
    eng = B.Engine([int(d) for d in args.devices.split(",")])
    eng.set_rlc_salt(SALT)

    def line(name, *outs):
        h = hashlib.sha256()
        for o in outs:
            h.update(np.ascontiguousarray(o).tobytes())
        kern = ",".join(f"{k}={c}" for k, (_, c) in eng.last_kernel_ms().items() if c)
        print(f"{name} sha={h.hexdigest()[:16]} launches={eng.launch_count() - line.last} kernels[{kern}]", flush=True)
        line.last = eng.launch_count()

    line.last = eng.launch_count()
    rnd = random.Random(20261020)
    nmax = 10000
    data, off = B.pack_messages([b"sig-%d" % i for i in range(nmax)])
    signed = {impl: eng.testdata_sign(impl, 0, keys(rnd, nmax), data, off) for impl in (2, 1)}
    line.last = eng.launch_count()

    # blsgpu_verify_batch (host buffers): per-item scaling, the bucket route with 64- and 128-bit scalars, several passes
    for impl, n, bits, chunk in [(2, 100, 64, None), (1, 100, 64, None), (2, 5000, 64, None), (2, 5000, 128, None), (1, 5000, 64, None),
                                 (2, 1000, 64, "240"), (2, nmax, 64, None)]:
        pks, sigs = signed[impl]
        pl, sl = B.pk_len(impl), B.sig_len(impl)
        eng.set_rlc_bits(bits)
        if chunk:
            os.environ["BLSGPU_M6_CHUNK"] = chunk
        for tag, bad in [("valid", []), ("bad", sorted(rnd.sample(range(n), 3)))]:
            st = eng.verify_batch_packed(impl, 0, pks[:pl * n], spoil(sigs[:sl * n], sl, bad), data, off[:n + 1])
            line(f"verify_batch impl={impl} n={n} bits={bits} chunk={chunk} {tag}", st)
        os.environ.pop("BLSGPU_M6_CHUNK", None)
    eng.set_rlc_bits(64)

    # blsgpu_verify_batch_dev (device-resident inputs)
    import torch
    for n in (100, 5000):
        pks, sigs = signed[2]
        for tag, bad in [("valid", []), ("bad", sorted(rnd.sample(range(n), 3)))]:
            t = [torch.from_numpy(np.array(a)).cuda() for a in (pks[:48 * n], spoil(sigs[:96 * n], 96, bad), data, off[:n + 1])]
            st = torch.zeros(n, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            eng.verify_batch_dev(2, 0, n, *[x.data_ptr() for x in t], st.data_ptr())
            torch.cuda.synchronize()
            line(f"verify_batch_dev n={n} {tag}", st.cpu().numpy())

    # blsgpu_pop_verify_batch
    none, off0 = B.pack_messages([b""] * 100)
    pks, proofs = eng.testdata_sign(2, 3, keys(rnd, 100), none, off0)
    line.last = eng.launch_count()
    line("pop_verify_batch valid", eng.pop_verify_batch(2, pks, proofs))
    line("pop_verify_batch bad", eng.pop_verify_batch(2, pks, spoil(proofs, 96, [7, 50])))

    # blsgpu_miller_partial -> blsgpu_final_exp_is_one -> blsgpu_partial_finish, and a tampered partial result
    pks, sigs = signed[2]
    for tag, bad in [("valid", []), ("bad", [11])]:
        gt, sm = eng.miller_partial(2, 0, pks[:48 * 200], spoil(sigs[:96 * 200], 96, bad), data, off[:201])
        ok = eng.final_exp_is_one(2, [gt], [sm])
        st = eng.partial_finish(200, ok)
        line(f"miller_partial/final_exp_is_one/partial_finish {tag}", np.frombuffer(gt + sm, dtype=np.uint8), np.array([ok]), st)
    gt, sm = eng.miller_partial(2, 0, pks[:48 * 200], sigs[:96 * 200], data, off[:201])
    tampered = bytearray(gt)
    tampered[100] ^= 1
    line("final_exp_is_one tampered", np.array([eng.final_exp_is_one(2, [bytes(tampered)], [sm])]))

    # blsgpu_aggregate_verify: one aggregate of 300 pairs, then of nmax pairs (cut over the devices of a multi-device context)
    for impl in (2, 1):
        pks, sigs = signed[impl]
        pl, sl = B.pk_len(impl), B.sig_len(impl)
        for n in (300, nmax):
            msgs = [bytes(data[off[i]:off[i + 1]]) for i in range(n)]
            agg = eng.sum_signatures(impl, sigs[:sl * n])
            line.last = eng.launch_count()
            for tag, sig in [("valid", agg), ("wrong", bytes(sigs[:sl]))]:
                st, idx = eng.aggregate_verify_status(impl, 0, pks[:pl * n], msgs, sig)
                line(f"aggregate_verify impl={impl} n={n} {tag}", np.array([st]), np.array(idx))

    # blsgpu_aggregate_verify_batch: aggregates of 1..7 pairs, and 40 of 250 pairs
    pks, sigs = signed[2]
    for sizes in ([1 + (j % 7) for j in range(120)], [250] * 40):
        soff = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
        aggs = [eng.sum_points(2, sigs[96 * int(soff[j]):96 * int(soff[j + 1])]) if sizes[j] > 1 else bytes(sigs[96 * int(soff[j]):96 * int(soff[j] + 1)])
                for j in range(len(sizes))]
        np_ = int(soff[-1])
        line.last = eng.launch_count()
        for tag, wrong in [("valid", []), ("wrong", sorted(rnd.sample(range(len(sizes)), 4)))]:
            sg = np.frombuffer(b"".join(aggs[(j + 1) % len(aggs)] if j in wrong else aggs[j] for j in range(len(aggs))), dtype=np.uint8)
            st, idx = eng.aggregate_verify_batch_packed(2, 0, soff, pks[:48 * np_], data, off[:np_ + 1], sg)
            line(f"aggregate_verify_batch q={len(sizes)} pairs={np_} {tag}", st, idx)

    # blsgpu_verify_secure_batch: key sets of 2..9 members, and 50 of 200 (the signatures are plain ones: the statuses are the rejections)
    for sizes in ([2 + (j % 8) for j in range(60)], [200] * 50):
        koff = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
        q = len(sizes)
        st = eng.verify_secure_batch_packed(2, 0, koff, pks[:48 * int(koff[-1])], sigs[:96 * q], data, off[:q + 1])
        line(f"verify_secure_batch q={q} members={int(koff[-1])}", st)

    # blsgpu_verify_batch_wire (tags 0, 1, 2 and an unknown one) and blsgpu_verify_batch_records (ragged, tagged and raw)
    n = 64
    msgs = [bytes(data[off[i]:off[i + 1]]) for i in range(n)]
    tagged = [bytes([0]) + bytes(sigs[96 * i:96 * i + 96]) for i in range(n)]
    tagged[5] = bytes([1]) + tagged[5][1:]
    tagged[9] = bytes([3]) + tagged[9][1:]
    line("verify_batch_wire", eng.verify_batch_wire(2, pks[:48 * n], tagged, msgs))
    pk_rec = [bytes(pks[48 * i:48 * i + 48]) for i in range(n)]
    pk_rec[3] = pk_rec[3][:47]
    line("verify_batch_records tagged", eng.verify_batch_records(2, 1, -1, pk_rec, tagged, msgs))
    line("verify_batch_records raw", eng.verify_batch_records(2, 1, 0, pk_rec, [t[1:] for t in tagged], msgs))

    # the remaining entry points, appended so that every line above (and the random draws behind it) stays as it was
    # keyed verify: 300 items naming keys of a set of 1000
    ks = eng.key_set(2, pks[:48 * 1000])
    kidx = np.array(rnd.sample(range(1000), 300), dtype=np.uint32)
    kd, ko = B.pack_messages([bytes(data[off[k]:off[k + 1]]) for k in kidx])
    ksg = sigs.reshape(-1, 96)[kidx].reshape(-1)
    line.last = eng.launch_count()
    for tag, bad in [("valid", []), ("bad", sorted(rnd.sample(range(300), 3)))]:
        line(f"verify_batch_keyed n=300 {tag}", eng.verify_batch_keyed_packed(ks, 0, kidx, spoil(ksg, 96, bad), kd, ko))

    # 210 keys, key i signs message i % 7 (Basic and MessageAugmentation): grouped, multisig and secure calls over them
    gq, gn = 7, 210
    gd, go = B.pack_messages([b"grp-%d" % (i % gq) for i in range(gn)])
    gm = [b"grp-%d" % j for j in range(gq)]
    gk = keys(rnd, gn)
    gpk, gsig = eng.testdata_sign(2, 0, gk, gd, go)
    _, gsig_aug = eng.testdata_sign(2, 1, gk, gd, go)
    gks = eng.key_set(2, gpk)
    midx = np.arange(gn, dtype=np.uint32) % gq
    all_idx = np.arange(gn, dtype=np.uint32)
    gmd, gmo = B.pack_messages(gm)
    line.last = eng.launch_count()
    for scheme, sg in [(0, gsig), (1, gsig_aug)]:
        for tag, bad in [("valid", []), ("bad", sorted(rnd.sample(range(gn), 3)))]:
            s = spoil(sg, 96, bad)
            line(f"verify_batch_grouped scheme={scheme} {tag}", eng.verify_batch_grouped_packed(2, scheme, gpk, s, midx, gmd, gmo))
            line(f"verify_batch_grouped_keyed scheme={scheme} {tag}", eng.verify_batch_grouped_keyed_packed(gks, scheme, all_idx, s, midx, gmd, gmo))

    # quorum j = the keys of message j, with its members in key order; multi-signatures are their signatures' sums
    members = np.concatenate([np.arange(j, gn, gq) for j in range(gq)]).astype(np.uint32)
    qoff = np.arange(gq + 1, dtype=np.uint64) * np.uint64(gn // gq)
    mpk = gpk.reshape(-1, 48)[members].reshape(-1)
    msg_sigs = gsig.reshape(-1, 96)[members].reshape(-1)
    st, bad_idx, msums = eng.sum_points_batch_packed(2, qoff, msg_sigs)
    line("sum_points_batch", st, bad_idx, msums)
    broken = msg_sigs.copy()
    broken[96 * 40] ^= 0x01
    line("sum_points_batch bad point", *eng.sum_points_batch_packed(2, qoff, broken))
    for tag, sw in [("valid", []), ("bad", [2, 5])]:
        ms = spoil(msums, 96, sw)
        line(f"verify_multisig_batch {tag}", eng.verify_multisig_batch_packed(2, 0, qoff, mpk, ms, gmd, gmo))
        line(f"verify_multisig_batch_keyed {tag}", eng.verify_multisig_batch_keyed_packed(gks, 0, qoff, members, ms, gmd, gmo))

    # secure aggregation over the same quorums: the aggregates verify; then two of them swapped
    st, secure = eng.aggregate_secure_batch_packed(2, qoff, mpk, msg_sigs)
    line("aggregate_secure_batch", st, secure)
    st, secure_k = eng.aggregate_secure_batch_keyed_packed(gks, qoff, members, msg_sigs)
    line("aggregate_secure_batch_keyed", st, secure_k)
    for tag, sw in [("valid", []), ("bad", [1, 4])]:
        ss = spoil(secure, 96, sw)
        line(f"verify_secure_batch quorums {tag}", eng.verify_secure_batch_packed(2, 0, qoff, mpk, ss, gmd, gmo))
        line(f"verify_secure_batch_keyed {tag}", eng.verify_secure_batch_keyed_packed(gks, 0, qoff, members, ss, gmd, gmo))

    # threshold shares of f(x) = a0 + a1 x: five shares per set, then a set with a repeated identifier
    a0, a1 = rnd.randrange(1, O.R), rnd.randrange(1, O.R)
    xs = list(range(1, 6))
    sh_k = np.frombuffer(b"".join(((a0 + a1 * x) % O.R).to_bytes(32, "big") for x in xs), dtype=np.uint8)
    sd, so = B.pack_messages([b"share"] * len(xs))
    sh_pk, _ = eng.testdata_sign(2, 0, sh_k, sd, so)
    line.last = eng.launch_count()
    recs = [x.to_bytes(32, "big") + bytes(sh_pk[48 * i:48 * i + 48]) for i, x in enumerate(xs)]
    line("combine_shares_batch", *eng.combine_shares_batch(1, [recs, recs[:3], recs[:2] + recs[1:2]]))

    # pairing_check_batch: e(P, Q) e(-P, Q) == 1, and a lone e(P, Q)
    p0, q0 = bytes(pks[:48]), bytes(sigs[:96])
    neg = bytes([p0[0] ^ 0x20]) + p0[1:]
    line("pairing_check_batch", *eng.pairing_check_batch([[(p0, q0), (neg, q0)], [(p0, q0)], []]))

    # the other public checks and building blocks, on the batch's keys and signatures (their statuses are rejections)
    n = 48
    pk_l = [bytes(pks[48 * i:48 * i + 48]) for i in range(n)]
    sig_l = [bytes(sigs[96 * i:96 * i + 96]) for i in range(n)]
    msgs = [bytes(data[off[i]:off[i + 1]]) for i in range(n)]
    ys = [rnd.randrange(1, O.R).to_bytes(32, "big") for _ in range(n)]
    line("pok_verify_batch", eng.pok_verify_batch(2, 0, sig_l, sig_l[1:] + sig_l[:1], pk_l, ys, msgs))
    line("signcrypt_valid_batch", *eng.signcrypt_valid_batch(2, 0, pk_l, sig_l, msgs))
    line("signcrypt_verify_share_batch", *eng.signcrypt_verify_share_batch(2, 0, pk_l, pk_l[1:] + pk_l[:1], pk_l, sig_l, msgs))
    line("hash_to_curve_batch", np.frombuffer(b"".join(eng.hash_to_curve_batch(2, msgs, b"launch-signature-dst")), dtype=np.uint8))
    st, out = eng.recode_points(1, pk_l, 1, 0)
    line("recode_points", st, np.frombuffer(b"".join(out), dtype=np.uint8))
    ids = [rnd.randrange(1, O.R).to_bytes(32, "big") for _ in range(n)]
    pk_sh = [ids[i] + pk_l[i] for i in range(n)]
    for tag, sl_ in [("valid", sig_l), ("bad", sig_l[:5] + [sig_l[6]] + sig_l[6:])]:
        sig_sh = [ids[i] + sl_[i] for i in range(n)]
        line(f"verify_share_batch {tag}", eng.verify_share_batch(2, 0, pk_sh, sig_sh, msgs))
    eng.close()


if __name__ == "__main__":
    main()
